"""CPU tests of the pass model of the abundance vectors (plan_passes(mode="vec")): the cost grows with the keys
of both streams, a pass costs its larger stage, and the resident vector pair comes out of the budget."""
import numpy as np
import torch


def _vec(k=31, vb=8, text=1 << 20, n_win=10**9):
    from kman_b200.engine import pass_bytes

    return lambda n, m: pass_bytes(k, "vec", n, m, vb, text, n_win)


def test_vec_pass_bytes_grows_with_keys():
    for k in (12, 31, 40, 63):
        c = _vec(k=k)
        assert c(10**6, 0) < c(2 * 10**6, 0) < c(4 * 10**6, 0), k
        assert c(0, 10**6) < c(0, 2 * 10**6) < c(0, 4 * 10**6), k
        assert c(10**6, 10**6) <= c(10**6, 2 * 10**6), k
    assert _vec(vb=8)(10**6, 10**3) > _vec(vb=4)(10**6, 10**3)


def test_vec_pass_bytes_takes_the_larger_stage():
    """The narrow buffers are freed before the wide stream is extracted: no sum of the stages, no merge term."""
    from kman_b200 import _lib

    lib = _lib.load()
    for k in (31, 40, 63):
        c = _vec(k=k)
        n, m = 10**8, 10**8
        both = c(n, m)
        assert max(c(n, 0), c(0, m)) <= both
        # what both stages share is the extraction workspace and, beside the wide stage, the narrow sort's workspace
        assert both <= max(c(n, 0), c(0, m)) + lib.kmg_radix_sort_workspace_bytes(n, 16 if k > 32 else 8, 8, 0, 2 * k)
        assert both < c(n, 0) + c(0, m) - lib.kmg_extract_workspace_bytes(10**9)
    # a few wide keys beside many narrow ones cost nothing extra (the count / uniq model adds merge ranks)
    c = _vec(k=31)
    assert c(10**8, 1000) == c(10**8, 0)


def _fake_input(n: int):
    from kman_b200 import alphabet as ab
    from kman_b200.engine import DeviceInput
    from kman_b200.fasta import FlatInput

    flat = FlatInput(np.zeros(n, np.uint8), np.array([0, n // 2, n], np.uint64), ["a", "b"], ["a", "b"])
    return DeviceInput(torch.empty(n + 16, dtype=torch.uint8), n, flat, "ACGT", ab.NATYPES.DNA, None, None,
                       rec_starts=torch.zeros(3, dtype=torch.int64))


def test_vec_plan_takes_the_resident_vectors_from_the_budget(monkeypatch):
    from kman_b200 import _lib
    from kman_b200.engine import PASS_PARTS, Engine

    n, k = 10**6, 31
    d = _fake_input(n)
    n_keys = n - 2 * k
    narrow = np.full(PASS_PARTS, n_keys // PASS_PARTS, np.int64)
    narrow[0] += n_keys - int(narrow.sum())
    monkeypatch.setattr(Engine, "count_windows", lambda self, d, k, rc: (n_keys, 0))
    monkeypatch.setattr(Engine, "part_counts", lambda self, d, k, rc, n_parts: (narrow, np.zeros(n_parts, np.int64)))
    eng = object.__new__(Engine)
    eng.lib = _lib.load()
    plan_passes = Engine.plan_passes.__wrapped__  # (without the device switch)
    _, text_bytes = eng._text_plan(d, k, "vec", 1000)
    one = eng._one_pass_bytes(d, k, False, "vec", 0, d.payload_bytes, text_bytes)
    vectors, resident = 8 * (n + 1), eng._resident_bytes(d)

    plan = plan_passes(eng, d, k, False, "vec", budget_bytes=resident + vectors + one, chunk_rows=1000)
    assert plan.n_passes == 1 and plan.pass_bytes == [one]
    # the same budget without room for the vectors: key-range passes that leave it free
    plan = plan_passes(eng, d, k, False, "vec", budget_bytes=resident + one, chunk_rows=1000)
    assert plan.n_parts == PASS_PARTS and plan.n_passes >= 2
    assert max(plan.pass_bytes) <= one - vectors
    assert sum(hi - lo for lo, hi in plan.parts) == PASS_PARTS
