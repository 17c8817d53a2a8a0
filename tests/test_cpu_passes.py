"""CPU tests of the key-range pass scheme (Engine.write_count / write_uniq): the wide-stream part table
against a brute force in string order, and the pass planner on synthetic per-part counts."""
import bisect
import itertools

import numpy as np
import pytest

SYMBOLS16 = "ABCDGHKMNRSTUVWY"


def brute_wide_parts(rna: int, n_parts: int) -> np.ndarray:
    """Part of every 4-symbol prefix: the part of the largest plain 4-mer <= it in Python string order."""
    plain = "ACGU" if rna else "ACGT"
    mers = ["".join(p) for p in itertools.product(plain, repeat=4)]  # ascending: code order == string order
    assert mers == sorted(mers)
    b = n_parts.bit_length() - 1
    out = np.zeros(65536, np.uint8)
    for x in range(65536):
        s = "".join(SYMBOLS16[(x >> (12 - 4 * i)) & 15] for i in range(4))
        code = bisect.bisect_right(mers, s) - 1  # AAAA <= s always
        assert code >= 0
        out[x] = code >> (8 - b)
    return out


@pytest.mark.parametrize("rna", [0, 1])
@pytest.mark.parametrize("n_parts", [2, 4, 16, 256])
def test_wide_part_table_matches_string_order(rna, n_parts):
    from kman_b200.engine import wide_part_table

    got = wide_part_table(rna, n_parts)
    want = brute_wide_parts(rna, n_parts)
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, f"{bad.size} prefixes differ, first {bad[0]:#06x}: got {got[bad[0]]} want {want[bad[0]]}"


def test_wide_part_table_orders_wide_between_narrow_parts():
    """Every wide key of part p sorts after all narrow 4-mers of parts < p and before those of parts > p."""
    from kman_b200.engine import wide_part_table

    t = wide_part_table(0, 16)
    mers = ["".join(p) for p in itertools.product("ACGT", repeat=4)]
    for x in range(0, 65536, 7):
        s = "".join(SYMBOLS16[(x >> (12 - 4 * i)) & 15] for i in range(4))
        p = int(t[x])
        assert all(m <= s for m in mers[: 16 * p]) and all(m >= s for m in mers[16 * (p + 1):]), s


def test_wide_part_table_rejects_bad_n_parts():
    from kman_b200.engine import wide_part_table

    for bad in (0, 3, 512):
        with pytest.raises(AssertionError):
            wide_part_table(0, bad)


def _cost(k=31, mode="count", vb=4, text=64 << 20, n_win=10**9):
    from kman_b200.engine import pass_bytes

    return lambda n, m: pass_bytes(k, mode, n, m, vb, text, n_win)


@pytest.mark.parametrize("mode", ["count", "uniq"])
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_plan_parts_contiguous_cover_and_within_budget(mode, seed):
    from kman_b200.engine import plan_parts

    rng = np.random.default_rng(seed)
    narrow = rng.integers(0, 40_000_000, 256)
    narrow[rng.integers(0, 256, 20)] = 0  # empty parts
    wide = np.where(rng.random(256) < 0.2, rng.integers(1, 2_000_000, 256), 0)
    cost = _cost(mode=mode)
    budget = cost(int(narrow.sum()), int(wide.sum())) // 7
    parts = plan_parts(narrow, wide, cost, budget)
    assert parts[0][0] == 0 and parts[-1][1] == 256
    assert all(lo < hi for lo, hi in parts)
    assert all(a[1] == b[0] for a, b in zip(parts, parts[1:]))
    assert len(parts) >= 7
    for lo, hi in parts:
        assert cost(int(narrow[lo:hi].sum()), int(wide[lo:hi].sum())) <= budget
        if hi < 256:  # greedy: the next part would not have fit
            assert cost(int(narrow[lo:hi + 1].sum()), int(wide[lo:hi + 1].sum())) > budget


def test_pass_bytes_grows_with_keys():
    cost = _cost()
    assert cost(10**6, 0) < cost(2 * 10**6, 0) <= cost(2 * 10**6, 10**5) < cost(2 * 10**6, 10**6)
    assert _cost(k=40, mode="uniq", vb=8)(10**6, 10**3) > _cost(k=40, mode="uniq", vb=4)(10**6, 10**3)


def test_make_plan_one_pass_when_everything_fits():
    from kman_b200.engine import make_plan

    def no_counts():
        raise AssertionError("a one-pass plan needs no per-part counts")

    plan = make_plan(31, 10**12, 10**11, (10**9, 0), no_counts, _cost())
    assert plan.n_parts == 1 and plan.parts == [(0, 1)] and plan.n_passes == 1
    # k < 12 is fine as long as it fits
    assert make_plan(8, 10**12, 10**11, (10**9, 5), no_counts, _cost(k=8)).n_passes == 1
    # nothing to do: one (empty) pass whatever the budget
    assert make_plan(31, 0, 10**6, (0, 0), no_counts, _cost()).n_passes == 1


def test_make_plan_multi_pass():
    from kman_b200.engine import make_plan

    narrow = np.full(256, 10_000_000, np.int64)
    wide = np.zeros(256, np.int64)
    wide[100] = 1000
    cost = _cost()
    budget = cost(int(narrow.sum()), 1000) // 4
    plan = make_plan(31, budget, 10**13, (int(narrow.sum()), 1000), lambda: (narrow, wide), cost)
    assert plan.n_parts == 256 and plan.n_passes >= 4
    assert sum(hi - lo for lo, hi in plan.parts) == 256
    assert max(plan.pass_bytes) <= budget and len(plan.pass_bytes) == plan.n_passes


def test_make_plan_oversized_part_raises():
    from kman_b200.engine import make_plan

    narrow = np.zeros(256, np.int64)
    narrow[37] = 10**9
    cost = _cost()
    with pytest.raises(ValueError, match="part 37 of 256 needs"):
        make_plan(31, cost(10**9, 0) - 1, 10**13, (10**9, 0), lambda: (narrow, np.zeros(256, np.int64)), cost)


def test_make_plan_small_k_that_does_not_fit_raises():
    from kman_b200.engine import make_plan

    with pytest.raises(ValueError, match="k >= 12"):
        make_plan(11, 10**9, 10**10, (10**8, 0), lambda: (np.zeros(256), np.zeros(256)), _cost(k=11))


def test_device_budget_env_override(monkeypatch):
    """KMG_DEVICE_BUDGET (bytes) is the job's budget minus the resident input."""
    import torch

    from kman_b200.engine import Engine

    class D:
        bases = torch.empty(1000, dtype=torch.uint8)
        rec_starts = torch.empty(3, dtype=torch.int64)
        names_buf = None
        name_offs = None

    monkeypatch.setenv("KMG_DEVICE_BUDGET", "50000")
    assert Engine.device_budget(object.__new__(Engine), D()) == 50000 - 1000 - 24
    assert Engine.device_budget(object.__new__(Engine), D(), 9000) == 9000 - 1024
