"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle and the golden
vectors produced by the unmodified reference.  Bit-exact everywhere (integer/byte work)."""
import ctypes as C
import hashlib
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import kmer_oracle as ko  # noqa: E402
from gpu_util import first_diff, limbs_to_rows, widen  # noqa: E402


@pytest.fixture(scope="module")
def eng():
    from kman_b200.engine import get_engine

    return get_engine()


@pytest.fixture(autouse=True)
def _fresh_sort_heuristics(eng):
    """The hybrid sort adapts to what the calling thread saw before (tile width search, back-off
    after crowded data); every test starts from the default state."""
    eng.lib.kmg_set_option(b"hybrid", 1)
    yield


def _flat(recs):
    from kman_b200 import fasta

    return fasta.from_records(recs)


def _rand_records(rng, n_rec, max_len, alphabet="ACGT", p_other=0.0):
    recs = []
    for r in range(n_rec):
        n = int(rng.integers(0, max_len))
        s = rng.choice(list("ACGT"), size=n)
        if p_other:
            m = rng.random(n) < p_other
            s[m] = rng.choice(list("NRYacgtnX-"), size=int(m.sum()))
        recs.append(("rec%d desc" % r, "".join(s)))
    return recs


# Global position of bases[0] (DeviceInput.pos_offset): 0, one that makes the payloads straddle 2^32,
# and two past it.  Payloads are (global position << 1) | strand in 8 bytes; 4-byte payloads are refused.
POS_OFFSETS = [0, "straddle", 2**32 + 3, 2**47 + 5]


def _pos_offset(p, n_bases: int) -> int:
    return (1 << 31) - n_bases // 2 if p == "straddle" else p


def _want_vals(st, offset: int) -> np.ndarray:
    """Payloads the device stores for the oracle stream `st` of an input whose bases[0] is at `offset`."""
    return ((st["pos"].astype(np.uint64) + np.uint64(offset)) << np.uint64(1)) | st["strand"].astype(np.uint64)


def _payload64(rng, lo: np.ndarray) -> np.ndarray:
    """8-byte payloads whose upper word is non-zero (bit 63 set) and unrelated to the lower word `lo`: a
    kernel that moves only the low 32 bits of a payload fails on them."""
    hi = rng.permutation(len(lo)).astype(np.uint64) + np.uint64(0x8000_0001)
    return (hi << np.uint64(32)) | lo.astype(np.uint64)


# ---- K1+K2 ---------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [2, 3, 15, 16, 17, 21, 31, 32, 33, 47, 63, 64])
@pytest.mark.parametrize("rc", [False, True])
def test_extract_narrow_matches_oracle(eng, k, rc):
    rng = np.random.default_rng(100 + k)
    recs = _rand_records(rng, 4, 9000, p_other=0.01)
    ex = ko.extract_np(recs, k, rc)
    d = eng.upload(_flat(recs))
    want = limbs_to_rows(ex["narrow"]["keys"])
    for p in POS_OFFSETS:
        d.pos_offset = _pos_offset(p, d.n_bases)
        for vb in (0, 4, 8):
            if vb == 4 and d.payload_bytes == 8:
                with pytest.raises(ValueError, match="val_bytes=4"):
                    eng.extract(d, k, rc, wide=False, val_bytes=vb)
                continue
            a = eng.extract(d, k, rc, wide=False, val_bytes=vb)
            assert a.n == want.shape[0], (a.n, want.shape[0])
            assert first_diff(a.keys_host(), want) == "equal"
            assert a.n_other == ex["wide"]["pos"].shape[0] // (2 if rc else 1)
            if vb:
                assert first_diff(a.vals_host().astype(np.uint64), _want_vals(ex["narrow"], d.pos_offset)) == "equal", (p, vb)


@pytest.mark.parametrize("k", [2, 5, 16, 17, 25, 32, 33, 45, 48, 49, 63, 64])
@pytest.mark.parametrize("rc", [False, True])
def test_extract_wide_matches_oracle(eng, k, rc):
    rng = np.random.default_rng(200 + k)
    recs = _rand_records(rng, 3, 6000, p_other=0.03)
    ex = ko.extract_np(recs, k, rc)
    d = eng.upload(_flat(recs))
    want = limbs_to_rows(widen(ex["wide"]["keys"]))
    for p in POS_OFFSETS:
        d.pos_offset = _pos_offset(p, d.n_bases)
        a = eng.extract(d, k, rc, wide=True, val_bytes=8)
        assert a.n == want.shape[0]
        assert first_diff(a.keys_host(), want) == "equal"
        assert first_diff(a.vals_host(), _want_vals(ex["wide"], d.pos_offset)) == "equal", p


@pytest.mark.parametrize("k", [33, 40, 47, 48, 57, 64])
@pytest.mark.parametrize("rc", [False, True])
def test_wide_stream_beyond_k32_count_and_uniq_text(eng, k, rc):
    """Windows holding N / IUPAC symbols at k > 32 (256-bit 4-bit-code keys, kmermaid/seq.py:317-318 has no
    bound on k): kmg_sort256 + run-length / singleton stage + text + the narrow/wide interleave, byte for
    byte against the oracle (duplicated stretches so that counts > 1 and non-singletons exist)."""
    rng = np.random.default_rng(3300 + k)
    recs = _rand_records(rng, 3, 7000, p_other=0.004)
    t, s0 = recs[0]
    recs[0] = (t, s0 + s0[: len(s0) // 2] + "N" * 150 + s0[-300:])
    d = eng.upload(_flat(recs))
    assert eng.count_text(d, k, rc) == ko.count_text_np(recs, k, rc), (k, rc)
    assert eng.uniq_text(d, k, rc) == ko.uniq_text_np(recs, k, rc), (k, rc)


def test_extract_window_ranges_partition_the_input(eng):
    """k-1 overlap chunking (seq.py:361-383): windows of disjoint start ranges concatenate."""
    rng = np.random.default_rng(7)
    recs = _rand_records(rng, 3, 20000, p_other=0.005)
    k = 31
    d = eng.upload(_flat(recs))
    full = eng.extract(d, k, False, val_bytes=8)
    n_win = d.n_bases - k + 1
    cuts = [0, 1, 4095, 4096, 4097, 12345, n_win // 2, n_win - 1, n_win]
    keys, vals = [], []
    for b, e in zip(cuts[:-1], cuts[1:]):
        a = eng.extract(d, k, False, val_bytes=8, win_begin=b, win_end=e)
        keys.append(a.keys_host().copy())
        vals.append(a.vals_host().copy())
    assert first_diff(np.concatenate(keys), full.keys_host()) == "equal"
    assert first_diff(np.concatenate(vals), full.vals_host()) == "equal"


# ---- K3 ---------------------------------------------------------------------------------------
def _sort_case(eng, n, kb, vb, bits, seed, dup=False):
    import torch

    from kman_b200.engine import KeyArray

    rng = np.random.default_rng(seed)
    limbs = kb // 8
    raw = rng.integers(0, 2**63, size=(n, limbs), dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, size=(n, limbs), dtype=np.uint64)
    if dup:
        raw = raw[rng.integers(0, max(1, n // 50), size=n)]
    # keep only `bits` low bits
    if limbs == 1:
        raw[:, 0] &= np.uint64((1 << bits) - 1) if bits < 64 else np.uint64(2**64 - 1)
    else:
        hb = bits - 64
        raw[:, 1] &= np.uint64((1 << hb) - 1) if hb < 64 else np.uint64(2**64 - 1)
    vals = np.arange(n, dtype=np.uint32) if vb == 4 else _payload64(rng, np.arange(n))
    dev = eng.device
    t = lambda x: torch.from_numpy(x.view(np.uint8).reshape(-1).copy()).to(dev)  # noqa: E731
    a = KeyArray(t(raw), t(np.zeros_like(raw)), t(vals) if vb else None, t(np.zeros_like(vals)) if vb else None,
                 n, kb, vb, bits // 2, False)
    a = eng.sort(a, 0, bits)
    eng._status(eng._last_sort_ws) if n > 1 else None
    if limbs == 1:
        order = np.argsort(raw[:, 0], kind="stable")
        want = raw[order, 0]
    else:
        order = np.lexsort((raw[:, 0], raw[:, 1]))
        want = raw[order]
    assert first_diff(a.keys_host(), want) == "equal", (n, kb, vb, bits)
    if vb:
        assert first_diff(a.vals_host().astype(np.uint64), vals[order].astype(np.uint64)) == "equal", "payload/stability"


# (8-byte keys sort in tiles of 6144 keys; the range partition and 16-byte keys in tiles of 4096)
@pytest.mark.parametrize("n", [0, 1, 2, 31, 4095, 4096, 4097, 6143, 6144, 6145, 12_289, 70001, 1_000_003])
def test_radix_sort_u64_sizes(eng, n):
    _sort_case(eng, n, 8, 0, 62, seed=n)
    _sort_case(eng, n, 8, 8, 62, seed=n + 1, dup=True)


@pytest.mark.parametrize("bits", [4, 8, 9, 16, 42, 50, 62, 64])
def test_radix_sort_u64_bit_ranges(eng, bits):
    _sort_case(eng, 300_000, 8, 4, bits, seed=bits, dup=True)


@pytest.mark.parametrize("vb", [0, 4, 8])
def test_radix_sort_u64_payload_widths(eng, vb):
    _sort_case(eng, 500_009, 8, vb, 62, seed=30 + vb, dup=True)


@pytest.mark.parametrize("bits", [66, 100, 126, 128])
@pytest.mark.parametrize("vb", [0, 8])
def test_radix_sort_u128(eng, bits, vb):
    _sort_case(eng, 200_003, 16, vb, bits, seed=bits + vb, dup=True)


# ---- K4 ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("kb", [8, 16])
@pytest.mark.parametrize("n", [1, 2, 33, 4096, 4097, 300_001])
def test_rle_and_singletons(eng, kb, n):
    import torch

    from kman_b200.engine import KeyArray

    rng = np.random.default_rng(n + kb)
    limbs = kb // 8
    # long runs, short runs and singletons mixed; a run longer than a tile when n allows
    base = np.sort(rng.integers(0, max(2, n // 3), size=n).astype(np.uint64))
    if n > 10000:
        base[1000:9000] = base[1000]
        base = np.sort(base)
    raw = np.zeros((n, limbs), np.uint64)
    raw[:, 0] = base
    if limbs == 2:
        raw[:, 1] = base // np.uint64(7)
        raw = raw[np.lexsort((raw[:, 0], raw[:, 1]))]
    vals = _payload64(rng, rng.permutation(n))
    dev = eng.device
    t = lambda x: torch.from_numpy(x.view(np.uint8).reshape(-1).copy()).to(dev)  # noqa: E731
    a = KeyArray(t(raw), t(np.zeros_like(raw)), t(vals), t(np.zeros_like(vals)), n, kb, 8, 31, False, is_sorted=True)
    rows = raw[:, 0] if limbs == 1 else raw
    diff = (raw[1:] != raw[:-1]).any(axis=1)
    heads = np.concatenate(([0], np.flatnonzero(diff) + 1))
    lens = np.diff(np.concatenate((heads, [n])))
    tab = eng.rle_count(a)
    assert tab.n == heads.size
    assert first_diff(tab.keys_host(), rows[heads]) == "equal"
    assert first_diff(tab.counts_host().astype(np.int64), lens) == "equal"
    a = KeyArray(t(raw), t(np.zeros_like(raw)), t(vals), t(np.zeros_like(vals)), n, kb, 8, 31, False, is_sorted=True)
    s = eng.singletons(a)
    sel = heads[lens == 1]
    assert s.n == sel.size
    assert first_diff(s.keys_host(), rows[sel]) == "equal"
    assert first_diff(s.vals_host(), vals[sel]) == "equal"


# ---- K5 ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_parts", [1, 2, 3, 4, 8])
def test_range_partition(eng, n_parts):
    import torch

    from kman_b200.engine import KeyArray

    rng = np.random.default_rng(n_parts)
    n, k = 400_007, 31
    raw = rng.integers(0, 1 << 62, size=n, dtype=np.uint64)
    vals = np.arange(n, dtype=np.uint64)
    dev = eng.device
    t = lambda x: torch.from_numpy(x.view(np.uint8).reshape(-1).copy()).to(dev)  # noqa: E731
    a = KeyArray(t(raw), t(np.zeros_like(raw)), t(vals), t(np.zeros_like(vals)), n, 8, 8, k, False)
    a, pc = eng.range_partition(a, n_parts)
    part = ((raw >> np.uint64(62 - 16)) * np.uint64(n_parts)) >> np.uint64(16)
    order = np.argsort(part, kind="stable")
    assert list(pc) == list(np.bincount(part.astype(np.int64), minlength=n_parts))
    assert first_diff(a.keys_host(), raw[order]) == "equal"
    assert first_diff(a.vals_host(), vals[order]) == "equal"
    # parts are ordered ranges of the key space
    bounds = np.concatenate(([0], np.cumsum(pc)))
    ks = a.keys_host()
    for p in range(1, n_parts):
        if pc[p - 1] and pc[p]:
            assert ks[bounds[p - 1] : bounds[p]].max() < ks[bounds[p] : bounds[p + 1]].min()


# ---- whole path vs goldens -----------------------------------------------------------------------
def test_golden_edge_cases(eng, golden):
    from kman_b200 import fasta

    bad = []
    for c in golden["cases"]:
        d = eng.upload(fasta.parse_bytes(c["fasta_text"].encode("latin-1")), alphabet=c["alphabet"])
        for cmd, fn in (("count", eng.count_text), ("uniq", eng.uniq_text)):
            got = fn(d, c["k"], c["rc"])
            if got != c[cmd].encode("latin-1"):
                bad.append((c["name"], c["k"], c["alphabet"], c["rc"], cmd, got[:80], c[cmd][:80]))
    assert not bad, (len(bad), bad[:5])


@pytest.mark.parametrize("name", ["syn_100k", "syn_1m"])
def test_golden_synthetic_hashes(eng, golden, name):
    from kman_b200 import fasta

    ent = [e for e in golden["synthetic"] if e["name"] == name][0]
    data = ko.synth_fasta_bytes([("chr1 synthetic seed=%d" % ent["seed"], ko.synth_bases(ent["n"], ent["seed"]))])
    assert hashlib.sha256(data).hexdigest() == ent["fasta_sha256"]
    d = eng.upload(fasta.parse_bytes(data))
    out = eng.count_text(d, ent["k"])
    assert (out.count(b"\n"), hashlib.sha256(out).hexdigest()) == (ent["count_lines"], ent["count_sha256"])
    out = eng.uniq_text(d, ent["k"])
    assert (out.count(b"\n"), hashlib.sha256(out).hexdigest()) == (ent["uniq_lines"], ent["uniq_sha256"])


def test_golden_syn_dup(eng, golden):
    from kman_b200 import fasta

    for ent in [e for e in golden["synthetic"] if e["name"] == "syn_dup"]:
        d = eng.upload(fasta.parse_bytes(ent["fasta_text"].encode()))
        for cmd, fn in (("count", eng.count_text), ("uniq", eng.uniq_text)):
            out = fn(d, ent["k"], ent["rc"])
            assert (out.count(b"\n"), hashlib.sha256(out).hexdigest()) == (ent[cmd + "_lines"], ent[cmd + "_sha256"]), (ent["k"], ent["rc"], cmd)


@pytest.mark.parametrize("k,rc", [(25, False), (25, True), (31, False), (12, True)])
def test_cfg4_like_n_runs_and_softmask_vs_oracle(eng, k, rc):
    """config 4: N-runs, soft-masked lower case, isolated IUPAC symbols, runs touching record ends."""
    from kman_b200 import fasta

    rng = np.random.default_rng(4321)
    recs = []
    for r, n in enumerate((300_000, 150_000, 50_000)):
        s = np.frombuffer(ko.synth_bases(n, 4321 + r), np.uint8).copy()
        for _ in range(12):
            L = int(np.exp(rng.uniform(0, np.log(20000))))
            p = int(rng.integers(0, n))
            s[p : p + L] = ord("N")
        for _ in range(30):
            L = int(rng.integers(100, 5000))
            p = int(rng.integers(0, n))
            s[p : p + L] |= 0x20  # lower-case
        for c in b"RYKMSW":
            s[int(rng.integers(0, n))] = c
        if r == 0:
            s[:37] = ord("N")
        if r == 1:
            s[-41:] = ord("n")
        recs.append(("chr%d cfg4" % (r + 1), s.tobytes().decode()))
    # second half of record 3 repeats its first half -> counts > 1
    a = recs[2][1]
    recs[2] = (recs[2][0], a[: len(a) // 2] + a[: len(a) // 2])
    d = eng.upload(fasta.from_records(recs))
    for ab in ("IUPAC", "ACGT"):
        d = eng.upload(fasta.from_records(recs), alphabet=ab)
        assert eng.count_text(d, k, rc) == ko.count_text_np(recs, k, rc, ab), ("count", ab)
        assert eng.uniq_text(d, k, rc) == ko.uniq_text_np(recs, k, rc, ab), ("uniq", ab)


# ---- host-buffer C-ABI calls ----------------------------------------------------------------------
@pytest.mark.parametrize("k,rc", [(21, False), (31, True), (40, False)])
def test_host_api_count_and_uniq(eng, k, rc):
    from kman_b200 import _lib, alphabet as ab, fasta

    lib = _lib.load()
    seq = ko.synth_bases(200_000, 99).decode()
    recs = [("a", seq[:120_000] + seq[:30_000]), ("b", seq[100_000:])]
    flat = fasta.from_records(recs)
    lut, _ = ab.lut_tables("ACGT", ab.NATYPES.DNA)
    ctx = C.c_void_p()
    _lib.check(lib.kmg_ctx_create(0, C.byref(ctx)))
    try:
        kb = 8 if k <= 32 else 16
        cap = flat.bases.size * (2 if rc else 1)
        keys = np.zeros(cap * kb // 8, np.uint64)
        counts = np.zeros(cap, np.uint32)
        n_out = C.c_uint64(0)
        _lib.check(lib.kmg_count_host(ctx, flat.bases.ctypes.data, flat.bases.size, k, int(rc), lut.ctypes.data,
                                      keys.ctypes.data, counts.ctypes.data, cap, C.byref(n_out)))
        _, cw, det = ko.count_np(recs, k, rc, "ACGT")
        want = limbs_to_rows(det["narrow"]["keys"])
        got = keys[: n_out.value] if kb == 8 else keys[: 2 * n_out.value].reshape(-1, 2)
        assert first_diff(got, want) == "equal"
        assert first_diff(counts[: n_out.value].astype(np.int64), det["narrow"]["counts"]) == "equal"
        vals = np.zeros(cap, np.uint64)
        _lib.check(lib.kmg_uniq_host(ctx, flat.bases.ctypes.data, flat.bases.size, k, int(rc), lut.ctypes.data,
                                     keys.ctypes.data, vals.ctypes.data, cap, C.byref(n_out)))
        *_, det = ko.uniq_np(recs, k, rc, "ACGT")
        want = limbs_to_rows(det["narrow"]["keys"])
        got = keys[: n_out.value] if kb == 8 else keys[: 2 * n_out.value].reshape(-1, 2)
        assert first_diff(got, want) == "equal"
        wv = (det["narrow"]["pos"].astype(np.uint64) << np.uint64(1)) | det["narrow"]["strand"].astype(np.uint64)
        assert first_diff(vals[: n_out.value], wv) == "equal"
    finally:
        lib.kmg_ctx_destroy(ctx)


def test_errors_follow_reference_conventions(eng):
    from kman_b200 import fasta

    d = eng.upload(fasta.from_records([("a", "ACGTACGT")]))
    with pytest.raises(AssertionError):  # batcher.py:477-478
        eng.count_text(d, 1)
    with pytest.raises(ValueError):
        eng.count_text(d, 65)
    assert eng.count_text(d, 9) == b""  # k > len -> empty output (join.py:107-111)


# ---- full-size properties (config 2: 100 Mbp, k=31) ------------------------------------------------
def test_cfg2_properties_100mbp(eng):
    """Size-independent invariants at BASELINE.json's config-2 size: counts sum to the number
    of windows, distinct keys strictly ascending, and the duplicated-half variant doubles counts."""
    import torch

    from kman_b200 import fasta

    n, k = 100_000_000, 31
    half = np.frombuffer(ko.synth_bases(n // 2, 1234), np.uint8)
    bases = np.concatenate([half, half, np.array([10], np.uint8)])
    flat = fasta.FlatInput(bases, np.array([0, n + 1], np.uint64), ["chr1"], ["chr1"])
    d = eng.upload(flat, alphabet="ACGT", with_names=False)
    (tab,) = eng.count(d, k)
    keys = tab.keys[: tab.n * 8].view(torch.int64)
    counts = tab.counts[: tab.n * 4].view(torch.int32)
    assert int(counts.sum(dtype=torch.int64)) == n - k + 1
    assert bool((keys[1:] > keys[:-1]).all())  # 62-bit keys: signed compare is fine
    # windows fully inside either half occur twice; the k-1 windows spanning the seam are extra
    assert int((counts == 2).sum()) >= n // 2 - k + 1 - 64
    assert int(counts.max()) <= 4
    # checksum of checksums: sum(key*count) equals the sum over all extracted keys
    a = eng.extract(d, k)
    all_keys = a.keys[: a.n * 8].view(torch.int64)
    assert int((keys * counts.to(torch.int64)).sum()) == int(all_keys.sum())


# ---- fused digit histograms (extract -> sort hand-off) ------------------------------------------------
@pytest.mark.parametrize("k", [4, 5, 7, 8, 11, 12, 13, 16, 21, 31, 32, 33, 45, 64])
@pytest.mark.parametrize("rc", [False, True])
def test_extract_fused_histograms_match_key_digits(eng, k, rc):
    """kmg_extract derives every radix pass' digit histogram from one 4-mer histogram of the bases
    (+ edge / skipped-window corrections); it must equal the histogram of the emitted keys."""
    rng = np.random.default_rng(900 + k)
    recs = _rand_records(rng, 4, 12000, p_other=0.01) + [("tiny", "ACG"), ("short", "ACGTAC")]
    d = eng.upload(_flat(recs))
    n_win = d.n_bases - k + 1
    for (wb, we) in ((0, None), (3, n_win - 5), (4096, 4096 + 5000)):
        a = eng.extract(d, k, rc, val_bytes=0, win_begin=wb, win_end=we, want_hist=True)
        assert a.hist is not None
        hist = a.hist.cpu().numpy().view(np.uint64).reshape(16, 256)
        keys = a.keys_host()
        P = (2 * k + 7) // 8
        for p in range(P):
            bits = 8 if p + 1 < P else 2 * k - 8 * (P - 1)
            sh = 8 * p
            if keys.ndim == 1:
                dig = (keys >> np.uint64(sh)) & np.uint64((1 << bits) - 1)
            else:
                lo, hi = keys[:, 0], keys[:, 1]
                if sh >= 64:
                    v = hi >> np.uint64(sh - 64)
                elif sh == 0:
                    v = lo
                else:
                    v = (lo >> np.uint64(sh)) | (hi << np.uint64(64 - sh))
                dig = v & np.uint64((1 << bits) - 1)
            want = np.bincount(dig.astype(np.int64), minlength=256).astype(np.uint64)
            assert first_diff(hist[p], want) == "equal", (k, rc, wb, we, p)
        if keys.ndim == 1 and k >= 12:
            # rows 13..15: the three top key bytes (prefix passes of the hybrid sort)
            for j in range(3):
                dig = (keys >> np.uint64(2 * k - 8 * (j + 1))) & np.uint64(0xFF)
                want = np.bincount(dig.astype(np.int64), minlength=256).astype(np.uint64)
                assert first_diff(hist[15 - j], want) == "equal", (k, rc, wb, we, "top", j)
            assert not hist[P:13].any()
        else:
            assert not hist[P:].any()


@pytest.mark.parametrize("pattern", ["all_equal", "two_values", "sorted", "reversed", "low_bits_only", "poly_a_genome"])
def test_radix_sort_adversarial_distributions(eng, pattern):
    """Skewed digit distributions: every lane of a warp in the same bin, presorted input, ..."""
    import torch

    from kman_b200.engine import KeyArray

    n = 700_001
    rng = np.random.default_rng(11)
    if pattern == "all_equal":
        raw = np.full(n, 0x2AAAAAAAAAAAAAAA, np.uint64)
    elif pattern == "two_values":
        raw = np.where(rng.random(n) < 0.5, np.uint64(3), np.uint64(0x3FFFFFFFFFFFFFFF)).astype(np.uint64)
    elif pattern == "sorted":
        raw = np.sort(rng.integers(0, 1 << 62, size=n, dtype=np.uint64))
    elif pattern == "reversed":
        raw = np.sort(rng.integers(0, 1 << 62, size=n, dtype=np.uint64))[::-1].copy()
    elif pattern == "low_bits_only":
        raw = rng.integers(0, 7, size=n, dtype=np.uint64)
    else:
        raw = None
    if raw is not None:
        vals = np.arange(n, dtype=np.uint64)
        t = lambda x: torch.from_numpy(x.view(np.uint8).reshape(-1).copy()).to(eng.device)  # noqa: E731
        a = KeyArray(t(raw), t(np.zeros_like(raw)), t(vals), t(np.zeros_like(vals)), n, 8, 8, 31, False)
        a = eng.sort(a, 0, 62)
        order = np.argsort(raw, kind="stable")
        assert first_diff(a.keys_host(), raw[order]) == "equal"
        assert first_diff(a.vals_host(), vals[order]) == "equal"  # stable
        return
    # low-complexity genome: long homopolymer and dinucleotide runs through the whole path
    from kman_b200 import fasta

    s = "A" * 200_000 + "ACGT" * 10 + "T" * 150_000 + "AC" * 100_000 + ko.synth_bases(50_000, 5).decode() + "A" * 5000
    recs = [("low complexity", s), ("again", s[100_000:400_000])]
    d = eng.upload(fasta.from_records(recs), alphabet="ACGT")
    for k, rc in ((31, False), (31, True), (12, False)):
        assert eng.count_text(d, k, rc) == ko.count_text_np(recs, k, rc, "ACGT"), (k, rc)
        assert eng.uniq_text(d, k, rc) == ko.uniq_text_np(recs, k, rc, "ACGT"), (k, rc)


# ---- fused extract + range partition + (peer) stores, emulated on one GPU -----------------------------
@pytest.mark.parametrize("k,rc,n_parts", [(31, False, 8), (21, True, 4), (45, False, 3), (12, True, 2), (8, False, 5)])
def test_extract_scatter_partitions_like_extract_plus_range_partition(eng, k, rc, n_parts):
    """kmg_extract_scatter with all destination buffers on this GPU: every destination must receive
    exactly the keys (and payloads) of its key range -- as a multiset, the order inside a
    destination is not defined -- and the count-only launch must size the regions exactly."""
    import torch

    from kman_b200 import _lib

    rng = np.random.default_rng(500 + k)
    recs = _rand_records(rng, 3, 40000, p_other=0.002)
    ex = ko.extract_np(recs, k, rc, "ACGT")
    d = eng.upload(_flat(recs), alphabet="ACGT")
    lib = eng.lib
    kb = 8 if k <= 32 else 16
    n_win = d.n_bases - k + 1
    counts = torch.zeros(n_parts + 1, dtype=torch.int64, device=eng.device)
    _lib.check(lib.kmg_extract_scatter(d.bases.data_ptr(), d.n_bases, 0, n_win, k, int(rc), d.lut.data_ptr(), n_parts, None,
                                       None, kb, 0, 0, None, counts.data_ptr(), 1, eng._stream()))
    cnt = counts.cpu().numpy()
    limbs = ex["narrow"]["keys"]
    top16 = (limbs[0] >> np.uint64(2 * k - 16 - (64 if len(limbs) == 2 else 0))) if (len(limbs) == 1 or 2 * k - 16 >= 64) else None
    if top16 is None:  # 128-bit key whose top 16 bits straddle the limbs
        sh = 2 * k - 16
        top16 = ((limbs[1] >> np.uint64(sh)) | (limbs[0] << np.uint64(64 - sh))) & np.uint64(0xFFFF)
    top16 = top16 & np.uint64(0xFFFF)
    part = ((top16 * np.uint64(n_parts)) >> np.uint64(16)).astype(np.int64)
    want_counts = np.bincount(part, minlength=n_parts)
    assert list(cnt[:n_parts]) == list(want_counts)
    assert cnt[n_parts] == 0
    rows = limbs_to_rows(limbs)
    for po in POS_OFFSETS:
        off = _pos_offset(po, d.n_bases)
        bufs = [torch.zeros(max(int(c), 1) * kb, dtype=torch.uint8, device=eng.device) for c in want_counts]
        vbufs = [torch.zeros(max(int(c), 1) * 8, dtype=torch.uint8, device=eng.device) for c in want_counts]
        ptrs = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device=eng.device)
        vptrs = torch.tensor([b.data_ptr() for b in vbufs], dtype=torch.int64, device=eng.device)
        cursors = torch.zeros(n_parts, dtype=torch.int64, device=eng.device)
        _lib.check(lib.kmg_extract_scatter(d.bases.data_ptr(), d.n_bases, 0, n_win, k, int(rc), d.lut.data_ptr(), n_parts,
                                           ptrs.data_ptr(), vptrs.data_ptr(), kb, 8, off, cursors.data_ptr(), None, 0,
                                           eng._stream()))
        torch.cuda.synchronize()
        assert list(cursors.cpu().numpy()) == list(want_counts)
        wv = _want_vals(ex["narrow"], off)
        for p in range(n_parts):
            c = int(want_counts[p])
            got_k = bufs[p][: c * kb].cpu().numpy().view(np.uint64)
            got_k = got_k if kb == 8 else got_k.reshape(-1, 2)
            got_v = vbufs[p][: c * 8].cpu().numpy().view(np.uint64)
            sel = part == p
            o_got, o_want = np.argsort(got_v), np.argsort(wv[sel])  # payloads are unique: align by them
            assert first_diff(got_v[o_got], wv[sel][o_want]) == "equal", (po, p)
            assert first_diff(got_k[o_got], rows[sel][o_want]) == "equal", (po, p)


# ---- hybrid finish of key-only sorts (top-prefix passes + one shared-memory local sort) ---------------
def _keyonly_sort(eng, raw, bits):
    import torch

    from kman_b200.engine import KeyArray

    n = len(raw)
    t = lambda x: torch.from_numpy(x.view(np.uint8).reshape(-1)).to(eng.device)  # noqa: E731
    a = KeyArray(t(raw), torch.zeros(n * 8, dtype=torch.uint8, device=eng.device), None, None, n, 8, 0, bits // 2, False)
    a = eng.sort(a, 0, bits)
    eng._status(eng._last_sort_ws)
    return a


@pytest.mark.parametrize("n", [1 << 20, 1_300_007, 5_000_011])
@pytest.mark.parametrize("bits", [32, 40, 62, 64])
@pytest.mark.parametrize("pb", [0, 24])
def test_hybrid_sort_random(eng, n, bits, pb):
    rng = np.random.default_rng(n + bits)
    raw = rng.integers(0, 2**63, size=n, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, size=n, dtype=np.uint64)
    if bits < 64:
        raw &= np.uint64((1 << bits) - 1)
    eng.lib.kmg_set_option(b"hybrid_pb", pb)
    try:
        a = _keyonly_sort(eng, raw, bits)
    finally:
        eng.lib.kmg_set_option(b"hybrid_pb", 0)
    assert eng.lib.kmg_get_stat(b"hybrid_path") == 1  # the local sort handled every tile
    assert eng.lib.kmg_get_stat(b"hybrid_irregular") == 0
    assert eng.lib.kmg_get_stat(b"sort_passes") == (3 if pb == 24 else 2)
    assert first_diff(a.keys_host(), np.sort(raw)) == "equal"


_SKEWED = {"dup50": None, "dup3": 1, "all_equal": 3, "clustered": 3, "one_big_bucket": 2, "few_big_buckets": 2, "sorted": 1,
           "ramp": 3, "crowded_cells": 2}


@pytest.mark.parametrize("pattern", sorted(_SKEWED))
def test_hybrid_sort_skewed_inputs_fall_back_or_finish(eng, pattern):
    """hybrid_path: 1 = local sort finished everything, 2 = a few huge prefix buckets were gathered
    and re-sorted, 3 = most keys sat in such buckets and the plain passes sorted everything."""
    n = 2_000_003
    rng = np.random.default_rng(5)
    rnd = rng.integers(0, 1 << 62, size=n, dtype=np.uint64)
    if pattern == "dup50":
        raw = rnd[rng.integers(0, n // 50, size=n)]
    elif pattern == "dup3":
        raw = rnd[rng.integers(0, n // 3, size=n)]
    elif pattern == "all_equal":
        raw = np.full(n, 0x1234567890ABCDE, np.uint64)
    elif pattern == "clustered":  # two far-apart dense clusters plus a sparse background
        raw = np.concatenate([rnd[: n // 3] >> np.uint64(30), (rnd[n // 3: 2 * n // 3] >> np.uint64(30)) | np.uint64(1 << 61),
                              rnd[2 * n // 3:]])
    elif pattern == "one_big_bucket":  # 5% of the keys share one 16-bit prefix
        raw = rnd.copy()
        raw[: n // 20] = (raw[: n // 20] & np.uint64((1 << 46) - 1)) | np.uint64(0x1F3 << 46)
    elif pattern == "few_big_buckets":
        raw = rnd.copy()
        for j, pref in enumerate((0x0000, 0x7A31, 0xFFFF)):
            seg = slice(j * 30_000, (j + 1) * 30_000)
            raw[seg] = (raw[seg] & np.uint64((1 << 46) - 1)) | np.uint64(pref << 46)
    elif pattern == "sorted":
        raw = np.sort(rnd)
    elif pattern == "crowded_cells":  # thousands of DISTINCT keys that agree in the 16 + 13 bits the cells see
        raw = rnd.copy()
        raw[:6000] = (raw[:6000] & np.uint64((1 << 30) - 1)) | np.uint64(0x2222_0000_0000_000)
    else:
        raw = np.arange(n, dtype=np.uint64) * np.uint64(977)
    a = _keyonly_sort(eng, raw, 62)
    if _SKEWED[pattern] is not None:
        assert eng.lib.kmg_get_stat(b"hybrid_path") == _SKEWED[pattern], pattern
    assert first_diff(a.keys_host(), np.sort(raw)) == "equal", pattern


def test_hybrid_sort_can_be_switched_off(eng):
    rng = np.random.default_rng(9)
    raw = rng.integers(0, 1 << 62, size=1_500_000, dtype=np.uint64)
    eng.lib.kmg_set_option(b"hybrid", 0)
    try:
        a = _keyonly_sort(eng, raw, 62)
        assert eng.lib.kmg_get_stat(b"sort_passes") == 8
        assert eng.lib.kmg_get_stat(b"hybrid_path") == 0
    finally:
        eng.lib.kmg_set_option(b"hybrid", 1)
    assert first_diff(a.keys_host(), np.sort(raw)) == "equal"


@pytest.mark.parametrize("skew", [False, True])
def test_hybrid_sort_prefix_width_follows_the_skew_large(eng, skew):
    """125 M keys: uniform keys take the 16-bit prefix (two passes); keys whose top byte is skewed
    like a real genome's take 24 bits (three passes).  torch.sort is the checker."""
    import torch

    from kman_b200.engine import KeyArray

    n = 125_000_000
    g = torch.Generator(device=eng.device).manual_seed(3)
    keys = torch.randint(0, 1 << 62, (n,), dtype=torch.int64, device=eng.device, generator=g)
    if skew:  # a third of the keys move into one eighth of the key space
        keys[: n // 3] >>= 3
    want = torch.sort(keys).values
    a = KeyArray(keys.view(torch.uint8), torch.zeros(n * 8, dtype=torch.uint8, device=eng.device), None, None, n, 8, 0, 31, False)
    a = eng.sort(a, 0, 62)
    eng._status(eng._last_sort_ws)
    assert eng.lib.kmg_get_stat(b"hybrid_path") == 1
    assert eng.lib.kmg_get_stat(b"sort_passes") == (3 if skew else 2)
    got = a.keys.view(torch.int64)[:n]
    assert torch.equal(got, want)


# ---- kmg_sort_count: sort + run-length count in one call (fused into the hybrid finish) ---------------
def _sort_count(eng, raw, bits):
    import torch

    from kman_b200.engine import KeyArray

    n = len(raw)
    kb = 8 if raw.ndim == 1 else 16
    t = lambda x: torch.from_numpy(x.view(np.uint8).reshape(-1)).to(eng.device)  # noqa: E731
    a = KeyArray(t(raw), torch.zeros(max(n * kb, 16), dtype=torch.uint8, device=eng.device), None, None, n, kb, 0,
                 bits // 2, False)
    tab = eng.sort_count(a, bits)
    keys = tab.keys[: tab.n * kb].cpu().numpy().view(np.uint64)
    counts = tab.counts[: tab.n * 4].cpu().numpy().view(np.uint32)
    return (keys if kb == 8 else keys.reshape(-1, 2)), counts


@pytest.mark.parametrize("n", [1, 2, 77, 4097, 300_001, 1 << 20, 2_500_003])
@pytest.mark.parametrize("dup", [1, 3, 40])
def test_sort_count_u64_matches_numpy_unique(eng, n, dup):
    rng = np.random.default_rng(n * 7 + dup)
    pool = rng.integers(0, 1 << 62, size=max(1, n // dup), dtype=np.uint64)
    raw = pool[rng.integers(0, len(pool), size=n)]
    keys, counts = _sort_count(eng, raw, 62)
    wk, wc = np.unique(raw, return_counts=True)
    assert first_diff(keys, wk) == "equal", (n, dup)
    assert first_diff(counts.astype(np.uint64), wc.astype(np.uint64)) == "equal", (n, dup)
    if n >= 1 << 20 and dup < 40:
        assert eng.lib.kmg_get_stat(b"hybrid_path") == 1  # fused: the local sort wrote the table


@pytest.mark.parametrize("pattern", ["one_big_bucket", "all_equal", "crowded_cells", "high_bits_constant"])
def test_sort_count_skewed_inputs(eng, pattern):
    n = 2_000_003
    rng = np.random.default_rng(77)
    rnd = rng.integers(0, 1 << 62, size=n, dtype=np.uint64)
    bits = 62
    if pattern == "one_big_bucket":
        raw = rnd.copy()
        raw[: n // 20] = (raw[: n // 20] & np.uint64((1 << 40) - 1)) | np.uint64(0x1F3 << 46)
    elif pattern == "all_equal":
        raw = np.full(n, 12345678901234567, np.uint64)
    elif pattern == "crowded_cells":
        raw = rnd.copy()
        raw[:6000] = (raw[:6000] & np.uint64((1 << 30) - 1)) | np.uint64(0x2222_0000_0000_000)
    else:  # what a rank sorts after the range partition: the top bits are equal in all keys, not zero
        bits = 59
        raw = (rnd & np.uint64((1 << 59) - 1)) | np.uint64(0b101 << 59)
    keys, counts = _sort_count(eng, raw, bits)
    wk, wc = np.unique(raw, return_counts=True)
    assert first_diff(keys, wk) == "equal", pattern
    assert first_diff(counts.astype(np.uint64), wc.astype(np.uint64)) == "equal", pattern
    assert eng.lib.kmg_get_stat(b"hybrid_path") == {"one_big_bucket": 2, "all_equal": 3, "crowded_cells": 2,
                                                    "high_bits_constant": 1}[pattern]


def test_sort_count_u128(eng):
    rng = np.random.default_rng(4)
    n = 400_003
    pool = rng.integers(0, 1 << 62, size=(n // 3, 2), dtype=np.uint64)
    raw = pool[rng.integers(0, len(pool), size=n)]
    keys, counts = _sort_count(eng, raw, 126)
    order = np.lexsort((raw[:, 0], raw[:, 1]))
    srt = raw[order]
    head = np.ones(n, bool)
    head[1:] = (srt[1:] != srt[:-1]).any(axis=1)
    idx = np.flatnonzero(head)
    assert first_diff(keys, srt[idx]) == "equal"
    assert first_diff(counts.astype(np.uint64), np.diff(np.append(idx, n)).astype(np.uint64)) == "equal"


@pytest.mark.parametrize("k,rc", [(31, True), (16, False), (33, False)])
def test_low_complexity_genome_through_the_hybrid_sort(eng, k, rc):
    """> 2^20 keys with homopolymer / microsatellite runs (huge prefix buckets -> irregular tiles are
    gathered and re-sorted), soft-masked lower case, N runs and several records: count and uniq text
    must equal the oracle's byte for byte."""
    from kman_b200 import fasta

    rnd = ko.synth_bases(1_200_000, 21).decode()
    s1 = rnd[:400_000] + "A" * 60_000 + rnd[400_000:800_000].lower() + "AC" * 40_000 + "N" * 5_000 + rnd[800_000:] + "T" * 30_000
    s2 = rnd[100_000:700_000] + "GATTACA" * 9_000 + rnd[:50_000]
    recs = [("chr1 low complexity", s1), ("chr2", s2), ("tiny", "ACGTACGT")]
    d = eng.upload(fasta.from_records(recs), alphabet="ACGT")
    got = eng.count_text(d, k, rc)
    if k <= 32:
        assert eng.lib.kmg_get_stat(b"hybrid_path") in (1, 2, 3)
    assert got == ko.count_text_np(recs, k, rc, "ACGT"), (k, rc)
    assert eng.uniq_text(d, k, rc) == ko.uniq_text_np(recs, k, rc, "ACGT"), (k, rc)


@pytest.mark.parametrize("k,rc,n_parts", [(31, True, 4), (45, False, 3)])
def test_extract_scatter_shared_cursors(eng, k, rc, n_parts):
    """kmg_extract_scatter_shared on one GPU: one cursor per destination, advanced by every tile;
    each destination receives exactly its key range (as a multiset); a capacity that is too small
    is reported through the status word and nothing is stored past it."""
    import torch

    from kman_b200 import _lib

    rng = np.random.default_rng(900 + k)
    recs = _rand_records(rng, 3, 30000, p_other=0.0)
    ex = ko.extract_np(recs, k, rc, "ACGT")
    d = eng.upload(_flat(recs), alphabet="ACGT")
    lib = eng.lib
    kb = 8 if k <= 32 else 16
    n_win = d.n_bases - k + 1
    limbs = ex["narrow"]["keys"]
    sh = 2 * k - 16
    if len(limbs) == 1:
        top16 = limbs[0] >> np.uint64(sh)
    elif sh >= 64:
        top16 = limbs[0] >> np.uint64(sh - 64)
    else:
        top16 = (limbs[1] >> np.uint64(sh)) | (limbs[0] << np.uint64(64 - sh))
    part = (((top16 & np.uint64(0xFFFF)) * np.uint64(n_parts)) >> np.uint64(16)).astype(np.int64)
    want_counts = np.bincount(part, minlength=n_parts)
    cap = int(want_counts.max())
    rows = limbs_to_rows(limbs)
    runs = [(po, cap, False) for po in POS_OFFSETS] + [(POS_OFFSETS[-1], cap - 1, True)]
    for po, capacity, expect_overflow in runs:
        off = _pos_offset(po, d.n_bases)
        wv = _want_vals(ex["narrow"], off)
        bufs = [torch.zeros(cap * kb, dtype=torch.uint8, device=eng.device) for _ in range(n_parts)]
        vbufs = [torch.zeros(cap * 8, dtype=torch.uint8, device=eng.device) for _ in range(n_parts)]
        cursors = torch.zeros(n_parts * 32, dtype=torch.int64, device=eng.device)  # one cursor per 256-byte line
        ptrs = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device=eng.device)
        vptrs = torch.tensor([b.data_ptr() for b in vbufs], dtype=torch.int64, device=eng.device)
        cptrs = torch.tensor([cursors.data_ptr() + 256 * i for i in range(n_parts)], dtype=torch.int64, device=eng.device)
        status = torch.zeros(2, dtype=torch.int32, device=eng.device)
        _lib.check(lib.kmg_extract_scatter_shared(d.bases.data_ptr(), d.n_bases, 0, n_win, k, int(rc), d.lut.data_ptr(),
                                                  n_parts, ptrs.data_ptr(), vptrs.data_ptr(), kb, 8, off, cptrs.data_ptr(),
                                                  capacity, status.data_ptr(), eng._stream()))
        torch.cuda.synchronize()
        st = status.cpu().numpy()
        assert bool(st[0]) == expect_overflow and st[1] == 0
        if expect_overflow:
            continue
        assert list(cursors.cpu().numpy()[::32]) == list(want_counts)
        for p in range(n_parts):
            c = int(want_counts[p])
            got_k = bufs[p][: c * kb].cpu().numpy().view(np.uint64)
            got_k = got_k if kb == 8 else got_k.reshape(-1, 2)
            got_v = vbufs[p][: c * 8].cpu().numpy().view(np.uint64)
            sel = part == p
            o_got, o_want = np.argsort(got_v), np.argsort(wv[sel])
            assert first_diff(got_v[o_got], wv[sel][o_want]) == "equal", p
            assert first_diff(got_k[o_got], rows[sel][o_want]) == "equal", p


# ---- the hybrid finish on 16-byte keys (k > 32) ---------------------------------------------------------
def _u128_sorted(raw):
    order = np.lexsort((raw[:, 0], raw[:, 1]))
    return raw[order]


def _u128_keys(rng, n, bits, dup=1):
    pool = rng.integers(0, 2**63, size=(max(1, n // dup), 2), dtype=np.uint64) * np.uint64(2) + \
        rng.integers(0, 2, size=(max(1, n // dup), 2), dtype=np.uint64)
    hb = bits - 64
    if hb < 64:
        pool[:, 1] &= np.uint64((1 << hb) - 1)
    return pool if dup == 1 else pool[rng.integers(0, len(pool), size=n)]


def _keyonly_sort_u128(eng, raw, bits):
    import torch

    from kman_b200.engine import KeyArray

    n = len(raw)
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x).view(np.uint8).reshape(-1)).to(eng.device)  # noqa: E731
    a = KeyArray(t(raw), torch.zeros(n * 16, dtype=torch.uint8, device=eng.device), None, None, n, 16, 0, bits // 2, False)
    a = eng.sort(a, 0, bits)
    eng._status(eng._last_sort_ws)
    return a


@pytest.mark.parametrize("bits", [66, 90, 126, 128])
@pytest.mark.parametrize("pb", [0, 24])
def test_hybrid_sort_u128_random(eng, bits, pb):
    rng = np.random.default_rng(bits * 3 + pb)
    raw = _u128_keys(rng, 1_400_003, bits)
    eng.lib.kmg_set_option(b"hybrid_pb", pb)
    try:
        a = _keyonly_sort_u128(eng, raw, bits)
    finally:
        eng.lib.kmg_set_option(b"hybrid_pb", 0)
    assert eng.lib.kmg_get_stat(b"hybrid_path") == 1
    assert eng.lib.kmg_get_stat(b"sort_passes") == (3 if pb == 24 else 2)
    assert first_diff(a.keys_host(), _u128_sorted(raw)) == "equal"


@pytest.mark.parametrize("pattern", ["dup7", "one_big_bucket", "all_equal", "low_limb_only"])
def test_hybrid_sort_count_u128_skewed(eng, pattern):
    rng = np.random.default_rng(31)
    n, bits = 1_600_001, 126
    raw = _u128_keys(rng, n, bits, dup=7 if pattern == "dup7" else 1)
    if pattern == "one_big_bucket":  # 6 % of the keys share their top 16 bits (and differ below)
        raw[: n // 16, 1] = (raw[: n // 16, 1] & np.uint64((1 << 46) - 1)) | np.uint64(0x2A5B << 46)
    elif pattern == "all_equal":
        raw[:] = raw[0]
    elif pattern == "low_limb_only":  # everything above bit 64 equal: one huge prefix bucket
        raw[:, 1] = np.uint64(0x1234567)
    keys, counts = _sort_count(eng, raw, bits)
    srt = _u128_sorted(raw)
    head = np.ones(n, bool)
    head[1:] = (srt[1:] != srt[:-1]).any(axis=1)
    idx = np.flatnonzero(head)
    assert first_diff(keys, srt[idx]) == "equal", pattern
    assert first_diff(counts.astype(np.uint64), np.diff(np.append(idx, n)).astype(np.uint64)) == "equal", pattern
    assert eng.lib.kmg_get_stat(b"hybrid_path") == {"dup7": 1, "one_big_bucket": 2, "all_equal": 3, "low_limb_only": 3}[pattern]


# ---- kmg_sort_uniq: sort (hybrid finish with payload) + singletons in one call --------------------------
def _sort_uniq(eng, raw, vals, bits):
    import torch

    from kman_b200.engine import KeyArray

    n = len(raw)
    kb = 8 if raw.ndim == 1 else 16
    vb = vals.dtype.itemsize
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x).view(np.uint8).reshape(-1)).to(eng.device)  # noqa: E731
    z = lambda b: torch.zeros(max(b, 16), dtype=torch.uint8, device=eng.device)  # noqa: E731
    a = KeyArray(t(raw), z(n * kb), t(vals), z(n * vb), n, kb, vb, bits // 2, False)
    r = eng.sort_uniq(a, bits)
    keys = r.keys[: r.n * kb].cpu().numpy().view(np.uint64)
    got_v = r.vals[: r.n * vb].cpu().numpy().view(vals.dtype)
    return (keys if kb == 8 else keys.reshape(-1, 2)), got_v


def _want_singletons(raw, vals):
    order = np.argsort(raw, kind="stable")
    sk, sv = raw[order], vals[order]
    head = np.ones(len(raw), bool)
    head[1:] = sk[1:] != sk[:-1]
    tail = np.ones(len(raw), bool)
    tail[:-1] = sk[1:] != sk[:-1]
    one = head & tail
    return sk[one], sv[one]


@pytest.mark.parametrize("n", [1, 2, 4097, 300_001, 1 << 20, 3_000_017])
@pytest.mark.parametrize("vdt", [np.uint32, np.uint64])
@pytest.mark.parametrize("dup", [1, 2, 30])
def test_sort_uniq_u64_matches_numpy(eng, n, vdt, dup):
    rng = np.random.default_rng(n + dup)
    pool = rng.integers(0, 1 << 62, size=max(1, n // dup), dtype=np.uint64)
    raw = pool[rng.integers(0, len(pool), size=n)] if dup > 1 else pool[:n]
    vals = np.arange(n, dtype=vdt) * vdt(3) + vdt(1)
    if vdt == np.uint64:
        vals = _payload64(rng, vals)
    keys, got_v = _sort_uniq(eng, raw, vals, 62)
    wk, wv = _want_singletons(raw, vals)
    assert first_diff(keys, wk) == "equal", (n, dup)
    assert first_diff(got_v.astype(np.uint64), wv.astype(np.uint64)) == "equal", (n, dup)
    if n >= 1 << 20 and dup < 30:
        assert eng.lib.kmg_get_stat(b"hybrid_path") == 1 and eng.lib.kmg_get_stat(b"sort_passes") == 2


@pytest.mark.parametrize("pattern", ["one_big_bucket", "all_equal", "crowded_cells", "high_bits_constant"])
def test_sort_uniq_skewed_inputs(eng, pattern):
    n = 2_000_003
    rng = np.random.default_rng(78)
    rnd = rng.integers(0, 1 << 62, size=n, dtype=np.uint64)
    bits = 62
    if pattern == "one_big_bucket":
        raw = rnd.copy()
        raw[: n // 20] = (raw[: n // 20] & np.uint64((1 << 40) - 1)) | np.uint64(0x1F3 << 46)
    elif pattern == "all_equal":
        raw = np.full(n, 12345678901234567, np.uint64)
    elif pattern == "crowded_cells":
        raw = rnd.copy()
        raw[:6000] = (raw[:6000] & np.uint64((1 << 30) - 1)) | np.uint64(0x2222_0000_0000_000)
    else:
        bits = 59
        raw = (rnd & np.uint64((1 << 59) - 1)) | np.uint64(0b101 << 59)
    vals = _payload64(rng, np.arange(n))
    keys, got_v = _sort_uniq(eng, raw, vals, bits)
    wk, wv = _want_singletons(raw, vals)
    assert first_diff(keys, wk) == "equal", pattern
    assert first_diff(got_v, wv) == "equal", pattern
    assert eng.lib.kmg_get_stat(b"hybrid_path") == {"one_big_bucket": 2, "all_equal": 3, "crowded_cells": 2,
                                                    "high_bits_constant": 1}[pattern]


@pytest.mark.parametrize("mode", ["sort", "count", "uniq"])
def test_hybrid_crowded_runs_are_sorted_by_the_block(eng, mode):
    """Hundreds of DISTINCT keys that agree in every bit the cells look at (diverged copies of a
    repeat family): the thread that owns them hands the run to the whole block (rank sort) instead
    of giving the tile up -- the local sort still finishes everything (hybrid_path 1)."""
    n = 1_500_007
    rng = np.random.default_rng(2024)
    raw = rng.integers(0, 1 << 62, size=n, dtype=np.uint64)
    for j in range(300):  # 300 groups of 500 keys sharing their top 40 bits; a few exact duplicates inside
        seg = slice(j * 500, (j + 1) * 500)
        top = rng.integers(0, 1 << 40, dtype=np.uint64) << np.uint64(22)
        raw[seg] = top | (raw[seg] & np.uint64((1 << 22) - 1))
        raw[j * 500 + 7] = raw[j * 500 + 3]
    if mode == "sort":
        a = _keyonly_sort(eng, raw, 62)
        assert first_diff(a.keys_host(), np.sort(raw)) == "equal"
    elif mode == "count":
        keys, counts = _sort_count(eng, raw, 62)
        wk, wc = np.unique(raw, return_counts=True)
        assert first_diff(keys, wk) == "equal"
        assert first_diff(counts.astype(np.uint64), wc.astype(np.uint64)) == "equal"
    else:
        vals = np.arange(n, dtype=np.uint32)
        keys, got_v = _sort_uniq(eng, raw, vals, 62)
        wk, wv = _want_singletons(raw, vals)
        assert first_diff(keys, wk) == "equal"
        assert first_diff(got_v.astype(np.uint64), wv.astype(np.uint64)) == "equal"
    # (a 500-key bucket that straddles the end of a full-width tile can still overflow it: path 2)
    assert eng.lib.kmg_get_stat(b"hybrid_path") in (1, 2)
    assert eng.lib.kmg_get_stat(b"hybrid_irregular") <= 40


def test_hybrid_crowded_data_is_exact_and_history_free(eng):
    """Thousands of crowded cells (runs the whole block has to sort): the sort is exact, and a second
    call takes the very same path -- the sort keeps no per-thread history (no back-off, no remembered
    tile width): timing depends on the input alone."""
    n = 1_200_011
    rng = np.random.default_rng(5150)
    raw = rng.integers(0, 1 << 62, size=n, dtype=np.uint64)
    g = 3000  # 3000 groups of 300 distinct keys sharing their top 40 bits: most of the input
    tops = rng.integers(0, 1 << 40, size=g, dtype=np.uint64) << np.uint64(22)
    raw[: g * 300] = np.repeat(tops, 300) | (raw[: g * 300] & np.uint64((1 << 22) - 1))
    seen = []
    for _ in range(2):
        a = _keyonly_sort(eng, raw, 62)
        assert first_diff(a.keys_host(), np.sort(raw)) == "equal"
        seen.append(tuple(int(eng.lib.kmg_get_stat(s)) for s in (b"hybrid_path", b"sort_passes", b"hybrid_big_runs",
                                                                 b"hybrid_irregular")))
    assert seen[0] == seen[1], seen
    assert seen[0][0] in (1, 2) and seen[0][2] >= 1500


@pytest.mark.parametrize("seed", [7, 8])
def test_hybrid_sort_family_fuzz(eng, seed, monkeypatch, capsys):
    """A dozen randomised trials of tools/fuzz_sort.py (sort / count / uniq, 8- and 16-byte keys,
    clustered + duplicated + skewed keys, forced prefix and tile widths) against numpy."""
    import runpy

    monkeypatch.setattr(sys, "argv", ["fuzz_sort.py", "--trials", "12", "--seconds", "120", "--seed", str(seed)])
    runpy.run_path(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "fuzz_sort.py"),
                   run_name="__main__")
    assert "FUZZ_OK 12 trials" in capsys.readouterr().out


# ---- tiles without output (no prefix bucket starts in them) in the persistent local sort -----------------
def _sparse_prefix_keys(rng, n, n_prefixes, bits, dup):
    """n keys of `bits` bits whose top 24 bits take only `n_prefixes` values: prefix buckets of
    n / n_prefixes keys, several narrow tiles wide."""
    pref = rng.choice(1 << 24, size=n_prefixes, replace=False).astype(np.uint64)
    pool_n = max(1, n // dup)
    pool = (pref[rng.integers(0, n_prefixes, size=pool_n)] << np.uint64(bits - 24)) | \
        rng.integers(0, 1 << (bits - 24), size=pool_n, dtype=np.uint64)
    return pool if dup == 1 else pool[rng.integers(0, pool_n, size=n)]


@pytest.mark.parametrize("mode", ["count", "count_dup3", "uniq", "uniq_dup2", "sort"])
def test_hybrid_tiles_without_output_keep_the_tile_prefix_moving(eng, mode):
    """Buckets of ~5000 keys under 2048-wide tiles: three tiles in five own no bucket start and emit nothing.
    Such a tile's resolve also publishes its group's sum, so a CTA of the persistent kernel has to resolve
    it AFTER the tile it still holds (config 3 on 8 GPUs -- one 16-bit bucket per tile, 8 % of the tiles
    empty -- ran into the look-back spin limit when it did not)."""
    n, bits = 4_000_037, 62
    rng = np.random.default_rng(len(mode))
    dup = 3 if mode == "count_dup3" else 2 if mode == "uniq_dup2" else 1
    raw = _sparse_prefix_keys(rng, n, 800, bits, dup)
    eng.lib.kmg_set_option(b"hybrid_pb", 24)
    eng.lib.kmg_set_option(b"local_tile", 2048)
    try:
        if mode.startswith("count"):
            keys, counts = _sort_count(eng, raw, bits)
            wk, wc = np.unique(raw, return_counts=True)
            assert first_diff(keys, wk) == "equal"
            assert first_diff(counts.astype(np.uint64), wc.astype(np.uint64)) == "equal"
        elif mode.startswith("uniq"):
            vals = np.arange(n, dtype=np.uint32)
            keys, got_v = _sort_uniq(eng, raw, vals, bits)
            wk, wv = _want_singletons(raw, vals)
            assert first_diff(keys, wk) == "equal"
            assert first_diff(got_v.astype(np.uint64), wv.astype(np.uint64)) == "equal"
        else:
            a = _keyonly_sort(eng, raw, bits)
            assert first_diff(a.keys_host(), np.sort(raw)) == "equal"
    finally:
        eng.lib.kmg_set_option(b"hybrid_pb", 0)
        eng.lib.kmg_set_option(b"local_tile", 7936)
    assert eng.lib.kmg_get_stat(b"hybrid_path") == 1
    assert eng.lib.kmg_get_stat(b"hybrid_irregular") == 0


@pytest.mark.parametrize("mode", ["sort", "count", "uniq"])
def test_hybrid_one_bucket_tiles_take_the_first_local_sort_kernel(eng, mode):
    """Tiles narrower than two average prefix buckets are finished by local_sort_kernel: the persistent
    fine-cell kernel's tile prefix jams there.  72 M random 62-bit keys under a 16-bit prefix make buckets
    of n / 2^16 = 1099 keys on average.  With local_tile 2048 the target width min(2048, cap - 1.35 * 1099)
    is 2048 < 2 * 1099 for both the key-only tile (cap 8192: sort, count) and the tile with a u32 payload
    (cap 6144: uniq), so few_bucket_tiles holds and sort_impl picks the first kernel.  A third of the keys
    repeat another one: counts of 2 and dropped pairs."""
    n, bits = 72_000_000, 62
    rng = np.random.default_rng(1099)
    raw = rng.integers(0, 1 << 62, size=n, dtype=np.uint64)
    raw[1::3] = raw[::3]
    eng.lib.kmg_set_option(b"hybrid_pb", 16)
    eng.lib.kmg_set_option(b"local_tile", 2048)
    try:
        if mode == "sort":
            a = _keyonly_sort(eng, raw, bits)
            assert first_diff(a.keys_host(), np.sort(raw)) == "equal"
        elif mode == "count":
            keys, counts = _sort_count(eng, raw, bits)
            wk, wc = np.unique(raw, return_counts=True)
            assert first_diff(keys, wk) == "equal"
            assert first_diff(counts.astype(np.uint64), wc.astype(np.uint64)) == "equal"
        else:
            vals = np.arange(n, dtype=np.uint32)
            keys, got_v = _sort_uniq(eng, raw, vals, bits)
            wk, wv = _want_singletons(raw, vals)
            assert first_diff(keys, wk) == "equal"
            assert first_diff(got_v.astype(np.uint64), wv.astype(np.uint64)) == "equal"
    finally:
        eng.lib.kmg_set_option(b"hybrid_pb", 0)
        eng.lib.kmg_set_option(b"local_tile", 7936)
    assert eng.lib.kmg_get_stat(b"hybrid_path") == 1
    assert eng.lib.kmg_get_stat(b"sort_passes") == 2


def test_hybrid_tiles_without_output_u128(eng):
    n, bits = 3_000_017, 126
    rng = np.random.default_rng(77)
    raw = _u128_keys(rng, n, bits)
    pref = rng.choice(1 << 24, size=1500, replace=False).astype(np.uint64)
    raw[:, 1] = (raw[:, 1] & np.uint64((1 << 38) - 1)) | (pref[rng.integers(0, 1500, size=n)] << np.uint64(38))
    eng.lib.kmg_set_option(b"hybrid_pb", 24)
    eng.lib.kmg_set_option(b"local_tile", 2048)
    try:
        keys, counts = _sort_count(eng, raw, bits)
    finally:
        eng.lib.kmg_set_option(b"hybrid_pb", 0)
        eng.lib.kmg_set_option(b"local_tile", 7936)
    assert first_diff(keys, _u128_sorted(raw)) == "equal"
    assert int(counts.astype(np.uint64).sum()) == n
    assert eng.lib.kmg_get_stat(b"hybrid_path") in (1, 2)  # (two bucket starts in one window can overflow a tile)
