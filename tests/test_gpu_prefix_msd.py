"""GPU parity tests of the fused device path with the 16-bit prefix built top byte first: the extraction
scatters by the top key byte, region_partition_kernel splits every top-byte region by byte 2 with the
bucket starts of the prefix-16 pre-pass, and the local sort takes its tile bounds from those starts.
Everything is compared bit-exactly with the CPU oracle's numpy tier (oracle/kmer_oracle.py)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import kmer_oracle as ko  # noqa: E402
from gpu_util import first_diff, limbs_to_rows  # noqa: E402


@pytest.fixture(scope="module")
def eng():
    from kman_b200.engine import get_engine

    return get_engine()


@pytest.fixture(autouse=True)
def _default_options(eng):
    eng.lib.kmg_set_option(b"hybrid", 1)
    eng.lib.kmg_set_option(b"hybrid_pb", 0)
    yield
    eng.lib.kmg_set_option(b"hybrid_pb", 0)


def _flat(recs):
    from kman_b200 import fasta

    return fasta.from_records(recs)


def _rows(keys):
    return limbs_to_rows(keys)


def _table(rows):
    """distinct keys ascending + multiplicities"""
    if rows.ndim == 1:
        return np.unique(rows, return_counts=True)
    order = np.lexsort((rows[:, 0], rows[:, 1]))
    srt = rows[order]
    head = np.ones(len(srt), bool)
    head[1:] = (srt[1:] != srt[:-1]).any(axis=1)
    idx = np.flatnonzero(head)
    return srt[idx], np.diff(np.append(idx, len(srt)))


def _singletons(rows, vals):
    order = np.argsort(rows, kind="stable") if rows.ndim == 1 else np.lexsort((rows[:, 0], rows[:, 1]))
    sk, sv = rows[order], vals[order]
    ne = (sk[1:] != sk[:-1]) if rows.ndim == 1 else (sk[1:] != sk[:-1]).any(axis=1)
    head = np.ones(len(sk), bool)
    tail = np.ones(len(sk), bool)
    head[1:] = ne
    tail[:-1] = ne
    one = head & tail
    return sk[one], sv[one]


def _narrow(ex, sel=None):
    rows = _rows(ex["narrow"]["keys"])
    vals = (ex["narrow"]["pos"].astype(np.uint64) << np.uint64(1)) | ex["narrow"]["strand"].astype(np.uint64)
    if sel is not None:
        rows, vals = rows[sel], vals[sel]
    return rows, vals


def _genome(seed, n, p_n=0.0002, lower=True, dup=True):
    """one record of n random ACGT bases with N runs, isolated IUPAC symbols, a soft-masked stretch and
    a duplicated stretch (counts > 1)"""
    rng = np.random.default_rng(seed)
    b = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, size=n, dtype=np.uint8)].copy()
    if dup:
        b[n // 2 : n // 2 + n // 5] = b[: n // 5]
    if p_n:
        for _ in range(12):
            s, ln = int(rng.integers(0, n - 5000)), int(rng.integers(1, 4000))
            b[s : s + ln] = ord("N")
        iso = rng.integers(0, n, size=max(1, int(n * p_n)))
        b[iso] = np.frombuffer(b"RYKMSWN", np.uint8)[rng.integers(0, 7, size=iso.size)]
    if lower:
        s = n // 3
        b[s : s + n // 7] |= 0x20
    return [("chrM test", b.tobytes().decode())]


def _check_count(eng, d, recs, k, rc, lo=None, hi=None):
    ex = ko.extract_np(recs, k, rc)
    sel = None
    kw = {}
    if lo is not None:
        pos = ex["narrow"]["pos"]
        sel = (pos >= lo) & (pos < hi)
        kw = {"win_begin": lo, "win_end": hi}
    tab, _ = eng.count_narrow(d, k, rc, **kw)
    wk, wc = _table(_narrow(ex, sel)[0])
    assert tab.n == len(wk), (tab.n, len(wk))
    assert first_diff(tab.keys_host(), wk) == "equal"
    assert first_diff(tab.counts_host().astype(np.uint64), wc.astype(np.uint64)) == "equal"
    return ex


def _check_uniq(eng, d, ex, k, rc, vb, lo=None, hi=None):
    sel = None
    kw = {}
    if lo is not None:
        pos = ex["narrow"]["pos"]
        sel = (pos >= lo) & (pos < hi)
        kw = {"win_begin": lo, "win_end": hi}
    s, _ = eng.uniq_narrow(d, k, rc, val_bytes=vb, **kw)
    wk, wv = _singletons(*_narrow(ex, sel))
    assert s.n == len(wk), (s.n, len(wk))
    assert first_diff(s.keys_host(), wk) == "equal"
    assert first_diff(s.vals_host().astype(np.uint64), wv) == "equal"


@pytest.mark.parametrize("rc", [False, True])
@pytest.mark.parametrize("k", [16, 31, 45, 63])
def test_count_and_uniq_match_oracle(eng, k, rc):
    """N runs, IUPAC symbols, soft-masked bases; count and uniq (4- and 8-byte payload) at pb = 16 and 24"""
    recs = _genome(4000 + k + rc, 1_200_000)
    d = eng.upload(_flat(recs))
    for pb in (16, 24):
        eng.lib.kmg_set_option(b"hybrid_pb", pb)
        ex = _check_count(eng, d, recs, k, rc)
        assert eng.lib.kmg_get_stat(b"sort_passes") == pb // 8 - 1
        for vb in (4, 8):
            _check_uniq(eng, d, ex, k, rc, vb)
            assert eng.lib.kmg_get_stat(b"sort_passes") == pb // 8 - 1


@pytest.mark.parametrize("k,rc", [(31, False), (31, True), (45, True)])
def test_window_subrange(eng, k, rc):
    recs = _genome(77 + k, 1_500_000)
    d = eng.upload(_flat(recs))
    lo, hi = 98_765, 1_432_101
    ex = _check_count(eng, d, recs, k, rc, lo, hi)
    _check_uniq(eng, d, ex, k, rc, 8, lo, hi)


@pytest.mark.parametrize("rc", [False, True])
def test_poly_a_spills_the_shared_counters(eng, rc):
    """Poly-A over most of an input that spans several rounds of the pre-pass' persistent grid: one
    8-mer passes 2^15 inside a single CTA's share, so its counter spills to the global row.  With the
    16-bit prefix forced the huge bucket makes the fused count stand down (oversize tiles)."""
    rng = np.random.default_rng(11)
    n = 8_000_000
    b = np.full(n, ord("A"), np.uint8)
    b[:1_000_000] = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, size=1_000_000, dtype=np.uint8)]
    b[4_000_000:4_200_000] = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, size=200_000, dtype=np.uint8)]
    recs = [("chrA", b.tobytes().decode())]
    d = eng.upload(_flat(recs), alphabet="ACGT")
    eng.lib.kmg_set_option(b"hybrid_pb", 16)
    _check_count(eng, d, recs, 31, rc)
    assert eng.lib.kmg_get_stat(b"hybrid_path") in (2, 3)


@pytest.mark.parametrize("k", [31, 45])
def test_empty_regions_and_a_region_of_whole_tiles(eng, k):
    """Keys of only 82 top-byte regions: a G-free record fills 81 regions, 12288 records of exactly one
    window each (GGGG...) fill one more with a multiple of every region_partition tile size."""
    rng = np.random.default_rng(k)
    bulk = np.frombuffer(b"ACT", np.uint8)[rng.integers(0, 3, size=1_300_000, dtype=np.uint8)].tobytes().decode()
    tails = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, size=(12288, k - 4), dtype=np.uint8)]
    recs = [("bulk", bulk)] + [("g%d" % i, "GGGG" + tails[i].tobytes().decode()) for i in range(12288)]
    d = eng.upload(_flat(recs), alphabet="ACGT")
    ex = ko.extract_np(recs, k, False)
    rows = _rows(ex["narrow"]["keys"])
    top = (rows >> np.uint64(2 * k - 8)) if rows.ndim == 1 else (rows[:, 1] >> np.uint64(2 * k - 8 - 64))
    assert int((top == 0xAA).sum()) == 12288 and len(np.unique(top)) == 82
    eng.lib.kmg_set_option(b"hybrid_pb", 16)
    _check_count(eng, d, recs, k, False)
    assert eng.lib.kmg_get_stat(b"sort_passes") == 1 and eng.lib.kmg_get_stat(b"hybrid_path") == 1
    for vb in (4, 8):
        _check_uniq(eng, d, ex, k, False, vb)
