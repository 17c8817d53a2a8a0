"""GPU parity tests of the fused device path (kmg_extract_sort_count / kmg_extract_sort_uniq, pipeline.cu):
the extraction kernel doubles as the hybrid sort's first prefix pass.  Everything is compared
bit-exactly with the CPU oracle's numpy tier (oracle/kmer_oracle.py: extract_np restates
kmermaid/seq.py:284-328, rc :245-282; the table is what kmermaid/join.py:95-130 groups)."""
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


def _rows(keys_2d_or_1d):
    return keys_2d_or_1d


def _want_table(ex):
    """distinct narrow keys ascending + multiplicities (what join.py:95-130 groups)"""
    rows = limbs_to_rows(ex["narrow"]["keys"])
    if rows.ndim == 1:
        return np.unique(rows, return_counts=True)
    order = np.lexsort((rows[:, 0], rows[:, 1]))
    srt = rows[order]
    head = np.ones(len(srt), bool)
    head[1:] = (srt[1:] != srt[:-1]).any(axis=1)
    idx = np.flatnonzero(head)
    return srt[idx], np.diff(np.append(idx, len(srt)))


def _want_singletons(ex, pos_offset=0):
    rows = limbs_to_rows(ex["narrow"]["keys"])
    vals = ((ex["narrow"]["pos"].astype(np.uint64) + np.uint64(pos_offset)) << np.uint64(1)) | \
        ex["narrow"]["strand"].astype(np.uint64)
    if rows.ndim == 1:
        order = np.argsort(rows, kind="stable")
    else:
        order = np.lexsort((rows[:, 0], rows[:, 1]))
    sk, sv = rows[order], vals[order]
    ne = (sk[1:] != sk[:-1]) if rows.ndim == 1 else (sk[1:] != sk[:-1]).any(axis=1)
    head = np.ones(len(sk), bool)
    tail = np.ones(len(sk), bool)
    head[1:] = ne
    tail[:-1] = ne
    one = head & tail
    return sk[one], sv[one]


def _genome(seed, n, n_rec=3, p_n=0.0, dup=False, lower=False):
    """n random ACGT bases over n_rec records; optional N runs / isolated IUPAC symbols, a duplicated
    stretch (counts > 1) and soft-masked lower case."""
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
    cuts = sorted(int(x) for x in rng.integers(1, n - 1, size=n_rec - 1)) if n_rec > 1 else []
    recs, prev = [], 0
    for i, c in enumerate(cuts + [n]):
        recs.append(("chr%d test" % (i + 1), b[prev:c].tobytes().decode()))
        prev = c
    return recs


CASES = [
    # k, rc, n, kwargs
    (31, False, 1_400_000, {}),
    (31, True, 1_300_000, {"dup": True}),
    (21, False, 1_500_000, {"p_n": 0.0002, "lower": True, "dup": True}),
    (16, False, 1_300_000, {"dup": True}),
    (25, True, 1_200_000, {"p_n": 0.0003, "lower": True}),
    (45, False, 1_300_000, {"dup": True, "p_n": 0.0001}),
    (63, True, 1_100_000, {"dup": True}),
    (31, False, 300_000, {"dup": True}),   # below 2^20 keys: the stage path inside the same call
    (11, False, 1_300_000, {}),            # k < 16: stage path
]


@pytest.mark.parametrize("k,rc,n,kw", CASES)
def test_count_narrow_matches_oracle(eng, k, rc, n, kw):
    recs = _genome(1000 + k, n, **kw)
    ex = ko.extract_np(recs, k, rc)
    d = eng.upload(_flat(recs))
    tab, n_other = eng.count_narrow(d, k, rc)
    wk, wc = _want_table(ex)
    assert tab.n == len(wk), (tab.n, len(wk))
    assert first_diff(tab.keys_host(), wk) == "equal"
    assert first_diff(tab.counts_host().astype(np.uint64), wc.astype(np.uint64)) == "equal"
    assert n_other == ex["wide"]["pos"].shape[0] // (2 if rc else 1)
    big = len(limbs_to_rows(ex["narrow"]["keys"])) >= (1 << 20) and k >= 16
    if big and not kw.get("p_n"):
        assert eng.lib.kmg_get_stat(b"hybrid_path") == 1  # fused extraction + count, no fallback


@pytest.mark.parametrize("k,rc,n,kw", CASES)
def test_uniq_narrow_matches_oracle(eng, k, rc, n, kw):
    recs = _genome(2000 + k, n, **kw)
    ex = ko.extract_np(recs, k, rc)
    d = eng.upload(_flat(recs))
    # global position of bases[0]: 0, payloads straddling 2^32, and past it (8-byte payloads only)
    for off, vb in ((0, 4), (0, 8), ((1 << 31) - n // 2, 8), (2**32 + 3, 8), (2**47 + 5, 8)):
        d.pos_offset = off
        s, n_other = eng.uniq_narrow(d, k, rc, val_bytes=vb)
        wk, wv = _want_singletons(ex, off)
        assert s.n == len(wk), (s.n, len(wk))
        assert first_diff(s.keys_host(), wk) == "equal"
        assert first_diff(s.vals_host().astype(np.uint64), wv) == "equal", (off, vb)
        assert n_other == ex["wide"]["pos"].shape[0] // (2 if rc else 1)
    d.pos_offset = 2**32 + 3
    with pytest.raises(ValueError, match="val_bytes=4"):
        eng.uniq_narrow(d, k, rc, val_bytes=4)


@pytest.mark.parametrize("pb", [16, 24])
def test_forced_prefix_width(eng, pb):
    """Both prefix widths (two / three prefix passes, the first one inside the extraction kernel)."""
    recs = _genome(77, 1_400_000, dup=True)
    ex = ko.extract_np(recs, 31, False)
    d = eng.upload(_flat(recs))
    eng.lib.kmg_set_option(b"hybrid_pb", pb)
    tab, _ = eng.count_narrow(d, 31, False)
    wk, wc = _want_table(ex)
    assert first_diff(tab.keys_host(), wk) == "equal"
    assert first_diff(tab.counts_host().astype(np.uint64), wc.astype(np.uint64)) == "equal"
    assert eng.lib.kmg_get_stat(b"sort_passes") == pb // 8 - 1  # one pass fewer than prefix bytes


def test_window_subrange_and_skewed_genome(eng):
    """win_begin / win_end (multi-GPU chunks) and a low-complexity input: poly-A + microsatellite make
    huge prefix buckets, so the fused launch stands down and the sort + run-length path finishes."""
    rng = np.random.default_rng(5)
    n = 1_600_000
    b = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, size=n, dtype=np.uint8)].copy()
    b[100_000:160_000] = ord("A")
    b[700_000:760_000] = np.frombuffer(b"CA" * 30_000, np.uint8)
    recs = [("chrS", b.tobytes().decode())]
    d = eng.upload(_flat(recs))
    k = 31
    lo, hi = 123_457, 1_500_001
    tab, _ = eng.count_narrow(d, k, False, win_begin=lo, win_end=hi)
    ex = ko.extract_np(recs, k, False)
    keys = ex["narrow"]["keys"][0]
    pos = ex["narrow"]["pos"]
    sel = (pos >= lo) & (pos < hi)
    wk, wc = np.unique(keys[sel], return_counts=True)
    assert first_diff(tab.keys_host(), wk) == "equal"
    assert first_diff(tab.counts_host().astype(np.uint64), wc.astype(np.uint64)) == "equal"
    assert eng.lib.kmg_get_stat(b"hybrid_path") in (2, 3)


def test_text_paths_use_the_pipeline_and_match_the_oracle(eng):
    """count_text / uniq_text (what `kmer count` / `kmer uniq` write) on > 2^20 k-mers with both
    streams present (default IUPAC alphabet: N windows go to the wide stream)."""
    recs = _genome(31337, 1_250_000, n_rec=4, p_n=0.0002, dup=True, lower=True)
    d = eng.upload(_flat(recs))
    assert eng.count_text(d, 25, False) == ko.count_text_np(recs, 25, False)
    assert eng.uniq_text(d, 25, True) == ko.uniq_text_np(recs, 25, True)


def test_rle_count_overflow_reaches_the_caller(eng):
    """ADVICE r1: the run-length stage of kmg_sort_count keeps its status word in its own workspace
    header; it must reach the header callers check.  The limit is lowered through a test option so
    that no 2^32-fold k-mer is needed."""
    import torch

    from kman_b200.engine import KeyArray

    raw = np.repeat(np.arange(50, dtype=np.uint64), 2000)  # runs of 2000
    n = len(raw)
    t = torch.from_numpy(raw.view(np.uint8).copy()).to(eng.device)
    a = KeyArray(t, torch.zeros(n * 8, dtype=torch.uint8, device=eng.device), None, None, n, 8, 0, 31, False)
    eng.lib.kmg_set_option(b"count_limit", 1500)
    try:
        with pytest.raises(ValueError, match="count does not fit"):
            eng.sort_count(a, 62)
    finally:
        eng.lib.kmg_set_option(b"count_limit", 0)
    a = KeyArray(t, torch.zeros(n * 8, dtype=torch.uint8, device=eng.device), None, None, n, 8, 0, 31, False)
    tab = eng.sort_count(a, 62)
    assert tab.n == 50 and int(tab.counts_host()[0]) == 2000
