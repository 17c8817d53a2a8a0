"""Canonical k-mers (`--canonical`, rc = KMG_CANONICAL) on the device: count, uniq, histo and the count range,
bit for bit against the canonical oracle (tests/canonical_oracle.py, itself pinned to the reference's `-r` outputs
by tests/test_cpu_canonical.py), on every path of the pipeline."""
import ctypes as C
import io
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import kmer_oracle as ko  # noqa: E402
import synth_configs as sc  # noqa: E402  (oracle/ is on sys.path, see conftest.py)

import canonical_oracle as co  # noqa: E402
from gpu_util import first_diff, limbs_to_rows  # noqa: E402

K_GOLDEN = (2, 7, 12, 16, 25, 31, 32, 33, 45, 63, 64)
M = 2**32 - 1


@pytest.fixture(scope="module")
def eng():
    from kman_b200.engine import get_engine

    return get_engine()


@pytest.fixture(scope="module")
def CAN():
    from kman_b200.engine import CANONICAL

    return CANONICAL


@pytest.fixture(autouse=True)
def _default_options(eng):
    yield
    eng.lib.kmg_set_option(b"hybrid", 1)
    eng.lib.kmg_set_option(b"hybrid_pb", 0)
    eng.lib.kmg_set_option(b"local_tile", 7936)


def _upload(eng, recs, alphabet="IUPAC", with_names=True):
    from kman_b200 import fasta

    return eng.upload(fasta.from_records(recs), alphabet=alphabet, with_names=with_names)


def _synth(n, seed):
    return ko.synth_bases(n, seed).decode()


def _rc(s, alphabet="IUPAC"):
    return ko.mkrc_py(s, ko.ALPHABETS[alphabet]["DNA"])


def _keep(text, lo, hi):
    hi = M if hi is None else hi
    return b"".join(ln for ln in text.splitlines(keepends=True) if lo <= int(ln.rsplit(b"\t", 1)[1]) <= hi)


def _spectrum(counts):
    m, n = np.unique(np.asarray(counts, np.int64), return_counts=True)
    return m.astype(np.uint64), n.astype(np.uint64)


def _mixed_records(n, seed):
    """N runs, IUPAC symbols, soft masking, a copied stretch, and a stretch pasted back as its reverse complement."""
    rng = np.random.default_rng(seed)
    s = np.frombuffer(_synth(n, seed).encode(), np.uint8).copy()
    for _ in range(40):
        a = int(rng.integers(0, n - 3000))
        s[a:a + int(rng.integers(1, 3000))] = ord("N")
    for a in rng.integers(0, n, size=300):
        s[a] = ord("RYKMSWBDHV"[int(rng.integers(0, 10))])
    for _ in range(30):
        a = int(rng.integers(0, n - 20000))
        seg = s[a:a + int(rng.integers(100, 20000))]
        seg[:] = np.where(seg < 97, seg + 32, seg)
    t = s.tobytes().decode()
    back = _rc(t[n // 5: n // 5 + n // 10])
    t = t[: n // 2] + t[n // 10: n // 10 + n // 15] + t[n // 2:] + back
    cuts = [0, n // 3, n // 3 + 17, 2 * n // 3, len(t)]
    return [(f"chr{i}", t[cuts[i]:cuts[i + 1]]) for i in range(len(cuts) - 1)]


def _check(eng, CAN, recs, k, alphabet="IUPAC", d=None, ranges=((2, None), (1, 1)), uniq=True):
    """count, count range, histo and uniq of the canonical rule against the oracle; returns the failures."""
    d = _upload(eng, recs, alphabet) if d is None else d
    bad = []
    txt, counts, _ = co.count_np(recs, k, alphabet)
    want = ko.count_text_from(txt, counts, k)
    got = eng.count_text(d, k, CAN)
    if got != want:
        bad.append(("count", k, alphabet))
    for lo, hi in ranges:
        if eng.count_text(d, k, CAN, lo, hi) != _keep(want, lo, hi):
            bad.append(("range", k, alphabet, lo, hi))
    m, n = eng.histogram(d, k, CAN)
    wm, wn = _spectrum(counts)
    if not (np.array_equal(m, wm) and np.array_equal(n, wn)):
        bad.append(("histo", k, alphabet))
    elif counts.size and int((m * n).sum()) != int(counts.sum()):
        bad.append(("histo sum", k, alphabet))
    if uniq and eng.uniq_text(d, k, CAN) != co.uniq_text_np(recs, k, alphabet):
        bad.append(("uniq", k, alphabet))
    return bad


# ---- 1. golden texts ---------------------------------------------------------------------------------------
def test_golden_texts_every_k(eng, CAN, golden):
    texts = {}
    for c in golden["cases"]:
        texts.setdefault(c["name"], c["fasta_text"])
    bad = []
    for name, text in sorted(texts.items()):
        recs = ko.parse_fasta_text(text)
        for alphabet in ("IUPAC", "ACGT"):
            d = _upload(eng, recs, alphabet)
            for k in K_GOLDEN:
                bad += [(name,) + b for b in _check(eng, CAN, recs, k, alphabet, d=d)]
    assert not bad, (len(bad), bad[:5])


# ---- 2. palindromes -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_rep", [50, 400_000])
def test_palindromes_count_once(eng, CAN, n_rep):
    """(ACGT)^n and embedded EcoRI sites: at even k a palindrome counts once per occurrence, with strand '+'.
    The long input (1.6 Mbp) takes the fused pipeline at k >= 16."""
    s = _synth(max(4 * n_rep, 20_000), 7)
    recs = [("pal", "ACGT" * n_rep), ("eco", "".join(s[i:i + 97] + "GAATTC" for i in range(0, len(s) - 97, 97))),
            ("at", "AATT" * 300 + "TTAA" * 300)]
    for k in (4, 6, 16, 32, 40, 64):
        assert not _check(eng, CAN, recs, k, "ACGT", ranges=((2, None),)), k
    d = _upload(eng, recs, "ACGT")
    for k in (4, 6, 32):
        lines = eng.uniq_text(d, k, CAN).decode().splitlines()
        assert all(h.endswith(":+") for h, s_ in zip(lines[::2], lines[1::2]) if s_ == _rc(s_, "ACGT"))


# ---- 3. 3 Mbp mixed inputs, fused pipeline at both prefix widths ----------------------------------------------
@pytest.mark.parametrize("pb", [16, 24])
@pytest.mark.parametrize("k", [21, 31, 45])
def test_fused_mixed_input(eng, CAN, pb, k):
    eng.lib.kmg_set_option(b"hybrid_pb", pb)
    recs = _mixed_records(3_000_000, 11 + k)
    d = _upload(eng, recs)
    assert not _check(eng, CAN, recs, k, d=d)
    eng.count_narrow(d, k, CAN)  # (the last sort of count_text is the wide stream's)
    assert eng.lib.kmg_get_stat(b"hybrid_path") in (1, 2)


# ---- 4. every path ------------------------------------------------------------------------------------------
def test_plain_passes(eng, CAN):
    """Fewer than 2^20 keys, k < 16 and the hybrid finish switched off: kmg_extract + the plain sort."""
    recs = _mixed_records(400_000, 6)
    d = _upload(eng, recs)
    for k in (31, 12):
        assert not _check(eng, CAN, recs, k, d=d)
        eng.count_text(d, k, CAN)
        assert eng.lib.kmg_get_stat(b"hybrid_path") == 0
    eng.lib.kmg_set_option(b"hybrid", 0)
    recs = _mixed_records(3_000_000, 8)
    d = _upload(eng, recs)
    assert not _check(eng, CAN, recs, 31, d=d)
    eng.count_text(d, 31, CAN)
    assert eng.lib.kmg_get_stat(b"hybrid_path") == 0


def test_oversize_tiles(eng, CAN):
    """Poly-A and copied stretches (hybrid_path 2); a poly-A run beyond the gather buffer (hybrid_path 3)."""
    s = _synth(3_000_000, 21)
    recs = [("chrR", s[:1_500_000] + "A" * 30_000 + s[200_000:700_000] + s[1_500_000:] + "T" * 12_000 + _rc(s[:100_000]))]
    assert not _check(eng, CAN, recs, 31, "ACGT", uniq=False)
    eng.count_text(_upload(eng, recs, "ACGT"), 31, CAN)
    assert eng.lib.kmg_get_stat(b"hybrid_path") == 2
    s = _synth(1_300_000, 22)
    recs = [("chrA", s[:600_000] + "A" * 400_000 + s[600_000:] + "G" * 200_000)]
    assert not _check(eng, CAN, recs, 31, "ACGT", uniq=False)
    eng.count_text(_upload(eng, recs, "ACGT"), 31, CAN)
    assert eng.lib.kmg_get_stat(b"hybrid_path") == 3


def test_one_bucket_tiles(eng, CAN):
    """A 16-bit prefix and tiles of 2048 positions: the first local-sort kernel takes the one-bucket tiles."""
    eng.lib.kmg_set_option(b"hybrid_pb", 16)
    eng.lib.kmg_set_option(b"local_tile", 2048)
    s = _synth(4_000_000, 23)
    recs = [("r", s + _rc(s[:1_000_000]))]
    d = _upload(eng, recs, "ACGT")
    assert not _check(eng, CAN, recs, 31, "ACGT", d=d)
    eng.count_text(d, 31, CAN)
    assert eng.lib.kmg_get_stat(b"hybrid_path") == 1


def test_wide_32_byte_keys(eng, CAN):
    recs = _mixed_records(400_000, 5)
    for k in (33, 40, 63, 64):
        assert not _check(eng, CAN, recs, k), k


def test_forced_passes_equal_one_pass(eng, CAN):
    """Key-range passes under a small budget: the canonical part counts size them exactly (extract_parts checks
    the count of every pass), and the texts equal the one-pass texts and the oracle."""
    from kman_b200.engine import pass_bytes

    recs = _mixed_records(3_000_000, 31)
    d = _upload(eng, recs)
    k = 31
    narrow, wide = eng.part_counts(d, k, CAN, 256)
    ex = co.extract_np(recs, k)
    top = ex["narrow"]["keys"][0] >> np.uint64(2 * k - 8)
    assert np.array_equal(narrow, np.bincount(top.astype(np.int64), minlength=256))
    assert int(wide.sum()) == ex["wide"]["pos"].size
    assert eng.count_windows(d, k, CAN) == (ex["narrow"]["pos"].size, ex["wide"]["pos"].size)
    n_win = d.n_bases - k + 1
    for mode, write in (("count", eng.write_count), ("uniq", eng.write_uniq)):
        _, text_bytes = eng._text_plan(d, k, mode, 5000)
        cost = lambda a, b: pass_bytes(k, mode, a, b, d.payload_bytes, text_bytes, n_win)  # noqa: E731
        budget = max(cost(-(-int(narrow.sum()) // 4), -(-int(wide.sum()) // 4)),
                     max(cost(int(a), int(b)) for a, b in zip(narrow, wide))) + eng._resident_bytes(d)
        one, multi = io.BytesIO(), io.BytesIO()
        write(d, k, CAN, one)
        p = write(d, k, CAN, multi, budget_bytes=budget, chunk_rows=5000)
        assert p.n_passes > 1
        want = (co.count_text_np if mode == "count" else co.uniq_text_np)(recs, k)
        assert multi.getvalue() == one.getvalue() == want, mode
    fh = io.BytesIO()
    budget = max(pass_bytes(k, "histo", int(a), int(b), 0, 0, n_win) for a, b in zip(narrow, wide)) * 3
    p = eng.write_histogram(d, k, CAN, fh, budget_bytes=budget + eng._resident_bytes(d))
    assert p.n_passes > 1
    m, n = _spectrum(co.count_np(recs, k)[1])
    assert fh.getvalue() == "".join("%d\t%d\n" % mn for mn in zip(m.tolist(), n.tolist())).encode()


# ---- 5. 8-byte payloads past 2^32 ---------------------------------------------------------------------------
@pytest.mark.parametrize("offset", [(1 << 31) - 200_000, 2**32 + 3, 2**47 + 5])
def test_uniq_payloads_past_2_32(eng, CAN, offset):
    recs = _mixed_records(3_000_000, 41)
    d = _upload(eng, recs)
    d.pos_offset = offset
    *_, det = co.uniq_np(recs, 31)
    st = det["narrow"]
    want = ((st["pos"].astype(np.uint64) + np.uint64(offset)) << np.uint64(1)) | st["strand"].astype(np.uint64)
    assert st["strand"].any() and not st["strand"].all()
    s, _ = eng.uniq_narrow(d, 31, CAN)
    assert s.val_bytes == 8
    assert first_diff(s.keys_host(), limbs_to_rows(st["keys"])) == "equal"
    assert first_diff(s.vals_host().astype(np.uint64), want) == "equal"
    w = eng.sort_uniq(eng.extract(d, 31, CAN, wide=True, val_bytes=8))
    sw = det["wide"]
    want = ((sw["pos"].astype(np.uint64) + np.uint64(offset)) << np.uint64(1)) | sw["strand"].astype(np.uint64)
    assert first_diff(w.vals_host().astype(np.uint64), want) == "equal"


# ---- 6. host-buffer calls and argument errors ------------------------------------------------------------------
@pytest.mark.parametrize("k", [21, 31, 45])
def test_host_buffer_calls(eng, CAN, k):
    from kman_b200 import _lib, alphabet as ab, fasta

    lib = _lib.load()
    seq = _synth(1_500_000, 99)
    recs = [("a", seq[:1_200_000] + _rc(seq[:300_000])), ("b", seq[1_000_000:])]
    flat = fasta.from_records(recs)
    lut, _ = ab.lut_tables("ACGT", ab.NATYPES.DNA)
    ctx = C.c_void_p()
    _lib.check(lib.kmg_ctx_create(0, C.byref(ctx)))
    try:
        kb = 8 if k <= 32 else 16
        cap = flat.bases.size
        keys = np.zeros(cap * kb // 8, np.uint64)
        counts = np.zeros(cap, np.uint32)
        n_out = C.c_uint64(0)
        _lib.check(lib.kmg_count_host(ctx, flat.bases.ctypes.data, flat.bases.size, k, CAN, lut.ctypes.data,
                                      keys.ctypes.data, counts.ctypes.data, cap, C.byref(n_out)))
        _, _, det = co.count_np(recs, k, "ACGT")
        got = keys[: n_out.value] if kb == 8 else keys[: 2 * n_out.value].reshape(-1, 2)
        assert first_diff(got, limbs_to_rows(det["narrow"]["keys"])) == "equal"
        assert first_diff(counts[: n_out.value].astype(np.int64), det["narrow"]["counts"]) == "equal"
        vals = np.zeros(cap, np.uint64)
        _lib.check(lib.kmg_uniq_host(ctx, flat.bases.ctypes.data, flat.bases.size, k, CAN, lut.ctypes.data,
                                     keys.ctypes.data, vals.ctypes.data, cap, C.byref(n_out)))
        *_, det = co.uniq_np(recs, k, "ACGT")
        got = keys[: n_out.value] if kb == 8 else keys[: 2 * n_out.value].reshape(-1, 2)
        assert first_diff(got, limbs_to_rows(det["narrow"]["keys"])) == "equal"
        wv = (det["narrow"]["pos"].astype(np.uint64) << np.uint64(1)) | det["narrow"]["strand"].astype(np.uint64)
        assert first_diff(vals[: n_out.value], wv) == "equal"
    finally:
        lib.kmg_ctx_destroy(ctx)


def test_argument_errors(eng, CAN):
    import torch

    from kman_b200 import _lib

    lib = _lib.load()
    d = _upload(eng, [("a", _synth(100_000, 3))], "ACGT")
    k, n_win = 31, d.n_bases - 31 + 1
    keys = torch.empty(n_win * 8, dtype=torch.uint8, device=eng.device)
    hist = torch.empty(16 * 256 * 8, dtype=torch.uint8, device=eng.device)
    ws_bytes = lib.kmg_extract_workspace_bytes(n_win)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=eng.device)
    small = torch.zeros(4, dtype=torch.int64, device=eng.device)
    st = eng._stream()
    args = (d.bases.data_ptr(), d.n_bases, 0, n_win, k, CAN, 0, d.lut.data_ptr(), d.comp16.data_ptr(), keys.data_ptr(),
            8, None, 0, 0, small.data_ptr())
    assert lib.kmg_extract(*args, hist.data_ptr(), ws.data_ptr(), ws_bytes, st) == _lib.KMG_ERR_ARG
    assert lib.kmg_extract(*args, None, ws.data_ptr(), ws_bytes, st) == _lib.KMG_OK
    cnt = torch.zeros(3, dtype=torch.int64, device=eng.device)
    assert lib.kmg_extract_scatter(d.bases.data_ptr(), d.n_bases, 0, n_win, k, CAN, d.lut.data_ptr(), 2, None, None, 8, 0,
                                   0, None, cnt.data_ptr(), 1, st) == _lib.KMG_ERR_ARG
    status = torch.zeros(2, dtype=torch.int32, device=eng.device)
    cur = torch.zeros(2, dtype=torch.int64, device=eng.device)
    ptrs = torch.zeros(2, dtype=torch.int64, device=eng.device)
    assert lib.kmg_extract_scatter_checked(d.bases.data_ptr(), d.n_bases, 0, n_win, k, CAN, d.lut.data_ptr(), 2,
                                           ptrs.data_ptr(), None, 8, 0, 0, cur.data_ptr(), 1 << 20, status.data_ptr(),
                                           st) == _lib.KMG_ERR_ARG
    assert lib.kmg_extract_scatter_shared(d.bases.data_ptr(), d.n_bases, 0, n_win, k, CAN, d.lut.data_ptr(), 2,
                                          ptrs.data_ptr(), None, 8, 0, 0, ptrs.data_ptr(), 1 << 20, status.data_ptr(),
                                          st) == _lib.KMG_ERR_ARG
    torch.cuda.synchronize()
    with pytest.raises(AssertionError):
        eng.abundance(d, k, CAN)


# ---- 7. the commands ----------------------------------------------------------------------------------------
def _cli(*argv):
    from click.testing import CliRunner

    from kman_b200.scripts import kmer

    return CliRunner().invoke(kmer.main, list(argv))


def test_cli_count_uniq_histo(eng, tmp_path, monkeypatch):
    monkeypatch.setenv("KMG_ALPHABET", "IUPAC")
    recs = _mixed_records(500_000, 43)
    inp = tmp_path / "in.fa"
    inp.write_bytes(ko.synth_fasta_bytes([(n, s.encode()) for n, s in recs]))
    recs = ko.read_fasta(str(inp))
    for k in (21, 40):
        txt, counts, _ = co.count_np(recs, k, "IUPAC")
        want = ko.count_text_from(txt, counts, k)
        out = tmp_path / "count.tsv"
        r = _cli("count", "--canonical", str(inp), str(out), str(k))
        assert r.exit_code == 0, (r.output, r.exception)
        assert out.read_bytes() == want
        r = _cli("count", "--canonical", "--min-count", "2", str(inp), str(out), str(k))
        assert r.exit_code == 0, (r.output, r.exception)
        assert out.read_bytes() == _keep(want, 2, None) != b""
        r = _cli("uniq", "--canonical", str(inp), str(out), str(k))
        assert r.exit_code == 0, (r.output, r.exception)
        assert out.read_bytes() == co.uniq_text_np(recs, k, "IUPAC")
        r = _cli("histo", "--canonical", str(inp), str(out), str(k))
        assert r.exit_code == 0, (r.output, r.exception)
        m, n = _spectrum(counts)
        assert out.read_bytes() == "".join("%d\t%d\n" % mn for mn in zip(m.tolist(), n.tolist())).encode()
        r = _cli("count", str(inp), str(out), str(k))  # without the option: the forward table, as before
        assert r.exit_code == 0 and out.read_bytes() == ko.count_text_np(recs, k, False, "IUPAC")


# ---- 8. full size, without the oracle ----------------------------------------------------------------------
def _rc_keys(x, k):
    y = ~x
    r = np.zeros_like(x)
    for i in range(k):
        r = (r << np.uint64(2)) | ((y >> np.uint64(2 * i)) & np.uint64(3))
    return r


def test_config2_with_a_reverse_complemented_half(eng, CAN):
    """Config 2 (100 Mbp, one record) with its second half replaced by the reverse complement of the first: the
    canonical table equals the GPU `-r` table restricted to keys <= their rc, palindrome counts halved, and the
    spectrum is that table's."""
    b = sc.random_acgt(100_000_000, 1234)
    h = b.size // 2
    comp = np.zeros(256, np.uint8)
    for x, y in zip(b"ACGT", b"TGCA"):
        comp[x] = y
    b[h:2 * h] = comp[b[:h][::-1]]
    recs = [("chr1 synthetic seed=1234", b.tobytes().decode("latin-1"))]
    d = _upload(eng, recs, "ACGT", with_names=False)
    k = 31
    r = eng.count_narrow(d, k, True)[0]
    rk, rcnt = r.keys_host().copy(), r.counts_host().astype(np.int64)
    del r
    c = eng.count_narrow(d, k, CAN)[0]
    assert eng.lib.kmg_get_stat(b"hybrid_path") in (1, 2)
    ck, ccnt = c.keys_host().copy(), c.counts_host().astype(np.int64)
    del c
    rr = _rc_keys(rk, k)
    keep = rk <= rr
    want_c = np.where(rk[keep] == rr[keep], rcnt[keep] // 2, rcnt[keep])
    assert first_diff(ck, rk[keep]) == "equal"
    assert first_diff(ccnt, want_c) == "equal"
    assert int(ccnt.sum()) == b.size - k + 1
    m, n = eng.histogram(d, k, CAN)
    wm, wn = _spectrum(want_c)
    assert np.array_equal(m, wm) and np.array_equal(n, wn)
