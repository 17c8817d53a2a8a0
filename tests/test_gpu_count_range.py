"""`kmer count --min-count / --max-count` and the calls behind it (kmg_sort_count_range,
kmg_extract_sort_count_range, kmg_filter_counts): the count table restricted to
min_count <= count <= max_count must be `kmer count`'s output with the other lines removed, bit for bit."""
import importlib.util
import io
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import kmer_oracle as ko  # noqa: E402
import synth_configs as sc  # noqa: E402  (oracle/ is on sys.path, see conftest.py)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
M = 2**32 - 1
K_GOLDEN = (2, 7, 12, 16, 25, 31, 32, 33, 45, 63, 64)
RANGES = ((1, 1), (2, None), (2, 3), (3, 3))


@pytest.fixture(scope="module")
def eng():
    from kman_b200.engine import get_engine

    return get_engine()


@pytest.fixture(autouse=True)
def _default_options(eng):
    yield
    eng.lib.kmg_set_option(b"hybrid", 1)
    eng.lib.kmg_set_option(b"hybrid_pb", 0)
    eng.lib.kmg_set_option(b"local_tile", 7936)
    eng.lib.kmg_set_option(b"count_limit", 0)


def _keep(text, lo, hi):
    """The lines of a `kmer count` text whose count is in [lo, hi] (hi None: no limit)."""
    hi = M if hi is None else hi
    return b"".join(ln for ln in text.splitlines(keepends=True) if lo <= int(ln.rsplit(b"\t", 1)[1]) <= hi)


def _upload(eng, recs, alphabet="IUPAC"):
    from kman_b200 import fasta

    return eng.upload(fasta.from_records(recs), alphabet=alphabet, with_names=False)


def _synth(n, seed):
    return ko.synth_bases(n, seed).decode()


def _mixed_records(n, seed):
    """Several records with N runs, IUPAC symbols, soft-masked stretches and a copied stretch."""
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
    t = t[: n // 2] + t[n // 10: n // 10 + 200_000] + t[n // 2:]
    cuts = [0, n // 3, n // 3 + 17, 2 * n // 3, len(t)]
    return [(f"chr{i}", t[cuts[i]:cuts[i + 1]]) for i in range(len(cuts) - 1)]


def _check_ranges(eng, recs, k, rc, alphabet="IUPAC", ranges=RANGES, oracle=True):
    """count_text(min, max) against the filtered count_text() and, with `oracle`, the filtered oracle text and
    the oracle's count column under the same mask."""
    d = _upload(eng, recs, alphabet)
    full = eng.count_text(d, k, rc)
    want_full = ko.count_text_np(recs, k, rc, alphabet) if oracle else full
    assert full == want_full, (k, rc, alphabet)
    counts = ko.count_np(recs, k, rc, alphabet)[1] if oracle else None
    for lo, hi in ranges:
        got = eng.count_text(d, k, rc, lo, hi)
        assert got == _keep(full, lo, hi), (k, rc, alphabet, lo, hi)
        if oracle:
            tabs = eng.count(d, k, rc, lo, hi)
            got_c = np.sort(np.concatenate([t.counts_host().astype(np.int64) for t in tabs]))
            mask = (counts >= lo) & (counts <= (M if hi is None else hi))
            assert np.array_equal(got_c, np.sort(counts[mask])), (k, rc, alphabet, lo, hi)
    return d, full


def _table(t):
    return bytes(t.keys[: t.n * t.key_bytes].cpu().numpy().tobytes()), t.counts_host().tobytes(), t.n


# ---- 1. golden texts -----------------------------------------------------------------------------------
def test_golden_texts_every_k(eng, golden):
    texts = {}
    for c in golden["cases"]:
        texts.setdefault(c["name"], c["fasta_text"])
    bad = []
    for name, text in sorted(texts.items()):
        recs = ko.parse_fasta_text(text)
        for alphabet in ("IUPAC", "ACGT"):
            d = _upload(eng, recs, alphabet)
            for k in K_GOLDEN:
                for rc in (False, True):
                    full = eng.count_text(d, k, rc)
                    want = ko.count_text_np(recs, k, rc, alphabet)
                    counts = ko.count_np(recs, k, rc, alphabet)[1]
                    for lo, hi in RANGES:
                        got = eng.count_text(d, k, rc, lo, hi)
                        tabs = eng.count(d, k, rc, lo, hi)
                        got_c = np.sort(np.concatenate([t.counts_host().astype(np.int64) for t in tabs]))
                        mask = (counts >= lo) & (counts <= (M if hi is None else hi))
                        if full != want or got != _keep(want, lo, hi) or not np.array_equal(got_c, np.sort(counts[mask])):
                            bad.append((name, alphabet, k, rc, lo, hi))
    assert not bad, (len(bad), bad[:5])


# ---- 2. mixed input on the fused pipeline ----------------------------------------------------------------
@pytest.mark.parametrize("pb", [16, 24])
@pytest.mark.parametrize("k,rc", [(31, False), (45, True)])
def test_fused_mixed_input(eng, pb, k, rc):
    eng.lib.kmg_set_option(b"hybrid_pb", pb)
    _check_ranges(eng, _mixed_records(3_000_000, 11), k, rc, ranges=((1, 1), (2, None), (2, 3)))


# ---- 3. EMIT 4 against EMIT 1 ----------------------------------------------------------------------------
def _genome_like(n):
    spec = importlib.util.spec_from_file_location("genome_like_bench", os.path.join(ROOT, "tools", "genome_like_bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.genome_like(n).tobytes().decode()


@pytest.mark.parametrize("case", ["cfg2", "genome_like", "k63"])
def test_range_that_keeps_everything_equals_count(eng, case):
    """(1, 2^32 - 2) takes EMIT 4 and keeps every row: kmg_extract_sort_count's table byte for byte."""
    if case == "cfg2":
        recs, k, alphabet = sc.cfg2(100_000_000), 31, "ACGT"
    elif case == "genome_like":
        recs, k, alphabet = [("g", _genome_like(100_000_000))], 31, "ACGT"
    else:
        recs, k, alphabet = [("r", _synth(20_000_000, 63))], 63, "ACGT"
    d = _upload(eng, recs, alphabet)
    want, n_other = eng.count_narrow(d, k, False)
    path = eng.lib.kmg_get_stat(b"hybrid_path")
    assert n_other == 0 and (path == 1 or case == "genome_like")
    got, _ = eng.count_narrow(d, k, False, min_count=1, max_count=M - 1)
    assert eng.lib.kmg_get_stat(b"hybrid_path") == path
    assert _table(got) == _table(want)
    kept, _ = eng.count_narrow(d, k, False, min_count=2)
    c = want.counts_host()
    assert kept.n == int((c >= 2).sum()) and np.array_equal(kept.counts_host(), c[c >= 2])


def test_full_range_through_sort_count_range_is_sort_count(eng):
    import ctypes as C

    import torch

    rng = np.random.default_rng(5)
    n = 3_000_000
    raw = rng.integers(0, 1 << 62, size=n, dtype=np.uint64)
    raw[1::4] = raw[::4]
    out = []
    for fn in ("kmg_sort_count", "kmg_sort_count_range"):
        keys = torch.from_numpy(raw.view(np.uint8).copy()).to(eng.device)
        alt = torch.empty_like(keys)
        counts = torch.zeros(n, dtype=torch.int32, device=eng.device)
        n_out = torch.zeros(1, dtype=torch.int64, device=eng.device)
        ws_bytes = eng.lib.kmg_sort_count_workspace_bytes(n, 8, 62)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=eng.device)
        sel = C.c_int(0)
        extra = (1, M) if fn == "kmg_sort_count_range" else ()
        rc = getattr(eng.lib, fn)(keys.data_ptr(), alt.data_ptr(), n, 8, 62, None, *extra, counts.data_ptr(),
                                  n_out.data_ptr(), C.byref(sel), ws.data_ptr(), ws_bytes, eng._stream())
        assert rc == 0 and eng.lib.kmg_ws_status(ws.data_ptr(), eng._stream()) == 0
        m = int(n_out.item())
        out.append(((alt if sel.value else keys)[: 8 * m].cpu().numpy().tobytes(), counts[:m].cpu().numpy().tobytes()))
    assert out[0] == out[1]


# ---- 4. (1, 1) against uniq ---------------------------------------------------------------------------------
@pytest.mark.parametrize("k,rc", [(31, False), (45, True)])
def test_singletons_are_uniq_keys(eng, k, rc):
    d = _upload(eng, _mixed_records(3_000_000, 13))
    tabs = eng.count(d, k, rc, 1, 1)
    sing = eng.uniq(d, k, rc)
    assert len(tabs) == len(sing)
    for t, s in zip(tabs, sing):
        assert t.n == s.n and np.array_equal(t.counts_host(), np.ones(t.n, np.uint32))
        assert t.keys[: t.n * t.key_bytes].cpu().numpy().tobytes() == s.keys[: s.n * s.key_bytes].cpu().numpy().tobytes()


# ---- 5. every path ----------------------------------------------------------------------------------------
def test_fused_path(eng):
    _check_ranges(eng, [("r", _synth(3_000_000, 3) + _synth(3_000_000, 3)[:400_000])], 31, False, "ACGT", oracle=False)
    assert eng.lib.kmg_get_stat(b"hybrid_path") == 1


def test_oversize_tiles_fall_back(eng):
    """Poly-A and copied stretches: the fused launch stands down, the sort re-sorts the flagged ranges
    (hybrid_path 2) and the table is compacted with kmg_filter_counts."""
    s = _synth(3_000_000, 21)
    recs = [("chrR", s[:1_500_000] + "A" * 30_000 + s[200_000:700_000] + s[1_500_000:] + "A" * 12_000 + s[:100_000])]
    d = _upload(eng, recs, "ACGT")
    full = eng.count_text(d, 31, False)
    for lo, hi in ((2, None), (1, 1), (10_000, None)):
        assert eng.count_text(d, 31, False, lo, hi) == _keep(full, lo, hi)
        assert eng.lib.kmg_get_stat(b"hybrid_path") == 2


def test_irregular_keys_beyond_the_gather_buffer(eng):
    s = _synth(1_300_000, 22)
    recs = [("chrA", s[:600_000] + "A" * 400_000 + s[600_000:] + "C" * 200_000)]
    d = _upload(eng, recs, "ACGT")
    full = eng.count_text(d, 31, False)
    for lo, hi in ((2, None), (1, 1)):
        assert eng.count_text(d, 31, False, lo, hi) == _keep(full, lo, hi)
        assert eng.lib.kmg_get_stat(b"hybrid_path") == 3


@pytest.mark.parametrize("lo,hi", [(2, None), (1, 1)])
def test_one_bucket_tiles_take_the_first_local_sort_kernel(eng, lo, hi):
    """72 M random 62-bit keys, a third repeating another; a 16-bit prefix and tiles of 2048 positions pick
    local_sort_kernel (see test_hybrid_one_bucket_tiles_take_the_first_local_sort_kernel)."""
    import torch

    from kman_b200.engine import KeyArray

    n, bits = 72_000_000, 62
    rng = np.random.default_rng(1099)
    raw = rng.integers(0, 1 << 62, size=n, dtype=np.uint64)
    raw[1::3] = raw[::3]
    eng.lib.kmg_set_option(b"hybrid_pb", 16)
    eng.lib.kmg_set_option(b"local_tile", 2048)
    keys = torch.from_numpy(raw.view(np.uint8)).to(eng.device)
    a = KeyArray(keys, torch.empty_like(keys), None, None, n, 8, 0, bits // 2, False)
    tab = eng.sort_count(a, bits, min_count=lo, max_count=hi)
    assert eng.lib.kmg_get_stat(b"hybrid_path") == 1 and eng.lib.kmg_get_stat(b"sort_passes") == 2
    wk, wc = np.unique(raw, return_counts=True)
    mask = (wc >= lo) & (wc <= (M if hi is None else hi))
    assert tab.n == int(mask.sum())
    assert np.array_equal(tab.keys[: tab.n * 8].cpu().numpy().view(np.uint64), wk[mask])
    assert np.array_equal(tab.counts_host().astype(np.int64), wc[mask])


def test_plain_passes(eng):
    """Fewer than 2^20 keys and k < 16: no hybrid finish, kmg_rle_count + kmg_filter_counts."""
    recs = _mixed_records(400_000, 6)
    for k in (31, 12):
        _check_ranges(eng, recs, k, True)
        assert eng.lib.kmg_get_stat(b"hybrid_path") == 0


def test_wide_32_byte_keys(eng):
    recs = _mixed_records(400_000, 5)
    for k, rc in ((40, True), (63, False), (64, True)):
        _check_ranges(eng, recs, k, rc)


# ---- 6. kmg_filter_counts ---------------------------------------------------------------------------------
@pytest.mark.parametrize("kb", [8, 16, 32])
@pytest.mark.parametrize("in_place", [True, False])
def test_filter_counts(eng, kb, in_place):
    import torch

    rng = np.random.default_rng(kb)
    stream = eng._stream()
    for n in (1, 2047, 2048, 2049, 4095, 4096, 4097, 3 * 4096 + 5, 1_000_003):
        keys = rng.integers(0, 1 << 63, size=n * kb // 8, dtype=np.uint64)
        counts = rng.integers(1, 6, size=n).astype(np.uint32)
        for lo, hi in ((2, 3), (1, M), (6, M), (1, 1), (5, 5)):
            dk = torch.from_numpy(keys.view(np.uint8).copy()).to(eng.device)
            dc = torch.from_numpy(counts.view(np.uint8).copy()).to(eng.device)
            ok = dk if in_place else torch.zeros_like(dk)
            oc = dc if in_place else torch.zeros_like(dc)
            n_out = torch.zeros(1, dtype=torch.int64, device=eng.device)
            ws_bytes = eng.lib.kmg_rle_workspace_bytes(n)
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=eng.device)
            rc = eng.lib.kmg_filter_counts(dk.data_ptr(), dc.data_ptr(), n, kb, lo, hi, ok.data_ptr(), oc.data_ptr(),
                                           n_out.data_ptr(), ws.data_ptr(), ws_bytes, stream)
            assert rc == 0 and eng.lib.kmg_ws_status(ws.data_ptr(), stream) == 0
            mask = (counts >= lo) & (counts <= hi)
            m = int(n_out.item())
            assert m == int(mask.sum()), (n, lo, hi)
            got_k = ok[: m * kb].cpu().numpy().view(np.uint64).reshape(m, kb // 8)
            assert np.array_equal(got_k, keys.reshape(n, kb // 8)[mask]), (n, lo, hi)
            assert np.array_equal(oc[: 4 * m].cpu().numpy().view(np.uint32), counts[mask]), (n, lo, hi)


def test_filter_counts_rejects_bad_ranges(eng):
    import torch

    from kman_b200 import _lib

    n_out = torch.zeros(1, dtype=torch.int64, device=eng.device)
    for lo, hi in ((0, 5), (3, 2)):
        assert eng.lib.kmg_filter_counts(None, None, 0, 8, lo, hi, None, None, n_out.data_ptr(), None, 0,
                                         eng._stream()) == _lib.KMG_ERR_ARG
    d = _upload(eng, [("r", "ACGTACGTAC")])
    with pytest.raises(AssertionError):
        eng.count_text(d, 4, False, 0, 3)
    with pytest.raises(AssertionError):
        eng.count_text(d, 4, False, 4, 3)


# ---- 7. long runs -----------------------------------------------------------------------------------------
def test_long_runs(eng):
    """A 300-base stretch copied 5 000 times: multiplicities >= 4096 kept or dropped by max_count."""
    s = _synth(1_000_000, 23)
    recs = [("chrB", s[:500_000] + s[600_000:600_300] * 5_000 + s[500_000:]), ("chrC", s[600_000:600_300] * 300)]
    for k, rc in ((31, False), (21, True), (40, False)):
        d, full = _check_ranges(eng, recs, k, rc, "ACGT", ranges=((4096, None), (1, 4095), (2, 5299), (5300, 5300)),
                                oracle=False)
        assert eng.count_text(d, k, rc, 4096) != b""


def test_count_limit_still_raises_under_a_range(eng):
    import torch

    from kman_b200.engine import KeyArray

    raw = np.repeat(np.arange(50, dtype=np.uint64), 2000)
    n = len(raw)
    t = torch.from_numpy(raw.view(np.uint8).copy()).to(eng.device)
    eng.lib.kmg_set_option(b"count_limit", 1500)
    for lo, hi in ((1, 10), (2, None), (3000, None)):
        a = KeyArray(t.clone(), torch.zeros(n * 8, dtype=torch.uint8, device=eng.device), None, None, n, 8, 0, 31, False)
        with pytest.raises(ValueError, match="count does not fit"):
            eng.sort_count(a, 62, min_count=lo, max_count=hi)
    eng.lib.kmg_set_option(b"count_limit", 0)
    a = KeyArray(t.clone(), torch.zeros(n * 8, dtype=torch.uint8, device=eng.device), None, None, n, 8, 0, 31, False)
    tab = eng.sort_count(a, 62, min_count=2000, max_count=2000)
    assert tab.n == 50


# ---- 8. forced passes ---------------------------------------------------------------------------------------
def _forced_budget(eng, d, k, rc, passes, chunk_rows):
    """A device budget under which plan_passes(mode="count") needs about `passes` passes."""
    from kman_b200.engine import pass_bytes

    narrow, wide = eng.part_counts(d, k, rc, 256)
    _, text_bytes = eng._text_plan(d, k, "count", chunk_rows)
    n_win = max(0, d.n_bases - k + 1)
    cost = lambda a, b: pass_bytes(k, "count", a, b, d.payload_bytes, text_bytes, n_win)  # noqa: E731
    target = cost(-(-int(narrow.sum()) // passes), -(-int(wide.sum()) // passes))
    biggest = max(cost(int(a), int(b)) for a, b in zip(narrow, wide))
    return max(target, biggest) + eng._resident_bytes(d)


def test_forced_passes_equal_one_pass(eng):
    recs = _mixed_records(3_000_000, 31)
    d = _upload(eng, recs)
    assert eng.plan_passes(d, 31, True, "count").n_passes == 1
    budget = _forced_budget(eng, d, 31, True, 4, 5000)
    full = eng.count_text(d, 31, True)
    for lo, hi in ((2, None), (1, 1)):
        one, multi = io.BytesIO(), io.BytesIO()
        eng.write_count(d, 31, True, one, min_count=lo, max_count=hi)
        p = eng.write_count(d, 31, True, multi, budget_bytes=budget, chunk_rows=5000, min_count=lo, max_count=hi)
        assert p.n_passes > 1
        assert multi.getvalue() == one.getvalue() == _keep(full, lo, hi)


# ---- 9. the command ---------------------------------------------------------------------------------------
def _cli(*argv):
    from click.testing import CliRunner

    from kman_b200.scripts import kmer

    return CliRunner().invoke(kmer.main, list(argv))


def test_cli_fasta_and_batches(eng, tmp_path, monkeypatch):
    monkeypatch.setenv("KMG_ALPHABET", "IUPAC")
    recs = _mixed_records(500_000, 41)
    recs.append(("rep", recs[0][1][:3000] * 3))
    inp = tmp_path / "in.fa"
    inp.write_bytes(ko.synth_fasta_bytes([(n, s.encode()) for n, s in recs]))
    full = tmp_path / "full.tsv"
    r = _cli("count", str(inp), str(full), "31")
    assert r.exit_code == 0, (r.output, r.exception)
    want = full.read_bytes()
    for opts, (lo, hi) in ((["--min-count", "2"], (2, None)), (["--max-count", "1"], (1, 1)),
                           (["--min-count", "2", "--max-count", "3"], (2, 3))):
        out = tmp_path / "out.tsv"
        r = _cli("count", str(inp), str(out), "31", *opts)
        assert r.exit_code == 0, (r.output, r.exception)
        assert out.read_bytes() == _keep(want, lo, hi), opts
    bdir = tmp_path / "batches"
    r = _cli("batch", str(inp), str(bdir), "25")
    assert r.exit_code == 0, (r.output, r.exception)
    r = _cli("count", "-B", str(bdir), str(inp), str(full), "25")
    assert r.exit_code == 0, (r.output, r.exception)
    want = full.read_bytes()
    out = tmp_path / "out_b.tsv"
    r = _cli("count", "-B", str(bdir), str(inp), str(out), "25", "--min-count", "2")
    assert r.exit_code == 0, (r.output, r.exception)
    assert out.read_bytes() == _keep(want, 2, None) != b""


def test_cli_empty_result(eng, tmp_path):
    inp, out = tmp_path / "in.fa", tmp_path / "out.tsv"
    inp.write_bytes(b">r1\nACGTTGCATGCAAGTC\n")
    r = _cli("count", str(inp), str(out), "8", "--min-count", "2")
    assert r.exit_code == 0, (r.output, r.exception)
    assert out.exists() and out.read_bytes() == b""
