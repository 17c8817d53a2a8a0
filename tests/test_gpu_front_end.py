"""The byte-2 region partition of the fused pipeline (pb = 16) on a skewed input.  Its CTAs take their region and
first key from the tile list prefix16_starts_kernel writes (one entry per tile, then empty entries up to the grid
the host sizes from the key count) and pull the tile of a CTA one wave later into L2.  An A-rich input makes the
top-byte regions very uneven: one region of many tiles, many regions of one partial tile or none.  Tables and
singletons are checked bit for bit against the oracle for 8- and 16-byte keys, forward, `-r` and canonical, and
payloads of 4 and 8 bytes."""
import functools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import kmer_oracle as ko  # noqa: E402

import canonical_oracle as co  # noqa: E402
from gpu_util import first_diff, limbs_to_rows  # noqa: E402

MODES = ["fwd", "rc", "canonical"]


@pytest.fixture(scope="module")
def eng():
    from kman_b200.engine import get_engine

    return get_engine()


@pytest.fixture(autouse=True)
def _pb16(eng):
    eng.lib.kmg_set_option(b"hybrid", 1)
    eng.lib.kmg_set_option(b"hybrid_pb", 16)
    yield
    eng.lib.kmg_set_option(b"hybrid_pb", 0)


@functools.lru_cache(maxsize=None)
def _records():
    """Two records of A-rich sequence with N runs: the top byte AAAA (with -r also TTTT) holds about a fifth of
    the keys."""
    n, p_a = 1_300_000, 0.68
    rng = np.random.default_rng(4242)
    q = (1 - p_a) / 3
    b = np.frombuffer(b"ACGT", np.uint8)[rng.choice(4, size=n, p=[p_a, q, q, q])].copy()
    for _ in range(6):
        s, ln = int(rng.integers(0, n - 3000)), int(rng.integers(1, 2500))
        b[s : s + ln] = ord("N")
    cut = n // 3
    return (("chrA skewed", b[:cut].tobytes().decode()), ("chrB", b[cut:].tobytes().decode()))


@functools.lru_cache(maxsize=None)
def _oracle(k, mode):
    """(keys as Engine host rows, position << 1 | strand) of every narrow window in position order"""
    recs = list(_records())
    ex = co.extract_np(recs, k) if mode == "canonical" else ko.extract_np(recs, k, mode == "rc")
    rows = limbs_to_rows(ex["narrow"]["keys"])
    vals = (ex["narrow"]["pos"].astype(np.uint64) << np.uint64(1)) | ex["narrow"]["strand"].astype(np.uint64)
    return rows, vals


def _sorted(rows, vals):
    order = np.argsort(rows, kind="stable") if rows.ndim == 1 else np.lexsort((rows[:, 0], rows[:, 1]))
    sk, sv = rows[order], vals[order]
    ne = (sk[1:] != sk[:-1]) if rows.ndim == 1 else (sk[1:] != sk[:-1]).any(axis=1)
    head = np.ones(len(sk), bool)
    head[1:] = ne
    return sk, sv, head


def _rc_arg(mode):
    from kman_b200.engine import CANONICAL

    return {"fwd": 0, "rc": 1, "canonical": CANONICAL}[mode]


def _device(eng):
    from kman_b200 import fasta

    return eng.upload(fasta.from_records(list(_records())))


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("k", [31, 45])
def test_count_on_uneven_regions(eng, k, mode):
    tab, _ = eng.count_narrow(_device(eng), k, _rc_arg(mode))
    sk, _, head = _sorted(*_oracle(k, mode))
    idx = np.flatnonzero(head)
    wk, wc = sk[idx], np.diff(np.append(idx, len(sk))).astype(np.uint64)
    assert tab.n == len(wk), (tab.n, len(wk))
    assert first_diff(tab.keys_host(), wk) == "equal"
    assert first_diff(tab.counts_host().astype(np.uint64), wc) == "equal"


@pytest.mark.parametrize("vb", [4, 8])
@pytest.mark.parametrize("k", [31, 45])
def test_uniq_on_uneven_regions(eng, k, vb):
    s, _ = eng.uniq_narrow(_device(eng), k, False, val_bytes=vb)
    sk, sv, head = _sorted(*_oracle(k, "fwd"))
    tail = np.ones(len(sk), bool)
    tail[:-1] = head[1:]
    one = head & tail
    assert s.n == int(one.sum()), (s.n, int(one.sum()))
    assert first_diff(s.keys_host(), sk[one]) == "equal"
    assert first_diff(s.vals_host().astype(np.uint64), sv[one]) == "equal"
