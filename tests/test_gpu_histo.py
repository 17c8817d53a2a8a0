"""`kmer histo` / Engine.histogram: the k-mer multiplicity spectrum, bit-exact against the spectrum of the
oracle's count column (np.unique over oracle.kmer_oracle.count_np's counts)."""
import io
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import kmer_oracle as ko  # noqa: E402
import synth_configs as sc  # noqa: E402  (oracle/ is on sys.path, see conftest.py)

HISTO_BINS = 4096
K_GOLDEN = (2, 7, 12, 16, 25, 31, 32, 33, 45, 63, 64)


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


def _spectrum(counts):
    m, c = np.unique(np.asarray(counts), return_counts=True)
    return m.astype(np.uint64), c.astype(np.uint64)


def _want(recs, k, rc, alphabet):
    return _spectrum(ko.count_np(recs, k, rc, alphabet)[1])


def _upload(eng, recs, alphabet):
    from kman_b200 import fasta

    return eng.upload(fasta.from_records(recs), alphabet=alphabet, with_names=False)


def _same(got, want):
    return got[0].dtype == np.uint64 and got[1].dtype == np.uint64 and np.array_equal(got[0], want[0]) and \
        np.array_equal(got[1], want[1])


def _check(eng, recs, k, rc=False, alphabet="IUPAC", budget=None):
    got = eng.histogram(_upload(eng, recs, alphabet), k, rc, budget)
    want = _want(recs, k, rc, alphabet)
    assert _same(got, want), (k, rc, alphabet, got[0][:8], got[1][:8], want[0][:8], want[1][:8])
    return got


def _synth(n, seed):
    return ko.synth_bases(n, seed).decode()


def _mixed_records(n, seed):
    """Several records with N runs, IUPAC symbols, soft-masked stretches and a copied stretch."""
    rng = np.random.default_rng(seed)
    s = np.frombuffer(_synth(n, seed).encode(), np.uint8).copy()
    for _ in range(40):  # N runs
        a = int(rng.integers(0, n - 3000))
        s[a:a + int(rng.integers(1, 3000))] = ord("N")
    for a in rng.integers(0, n, size=300):  # single IUPAC symbols
        s[a] = ord("RYKMSWBDHV"[int(rng.integers(0, 10))])
    for _ in range(30):  # soft-masking
        a = int(rng.integers(0, n - 20000))
        seg = s[a:a + int(rng.integers(100, 20000))]
        seg[:] = np.where(seg < 97, seg + 32, seg)
    t = s.tobytes().decode()
    t = t[: n // 2] + t[n // 10: n // 10 + 200_000] + t[n // 2:]
    cuts = [0, n // 3, n // 3 + 17, 2 * n // 3, len(t)]
    return [(f"chr{i}", t[cuts[i]:cuts[i + 1]]) for i in range(len(cuts) - 1)]


# ---- small inputs ------------------------------------------------------------------------------------
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
                    got, want = eng.histogram(d, k, rc), _want(recs, k, rc, alphabet)
                    if not _same(got, want):
                        bad.append((name, alphabet, k, rc, got, want))
    assert not bad, (len(bad), bad[:3])


def test_golden_counts_agree(eng, golden):
    """The spectrum of every golden `kmer count` text."""
    for c in golden["cases"]:
        counts = [int(line.split(b"\t")[1]) for line in c["count"].encode("latin-1").splitlines()]
        got = eng.histogram(_upload(eng, ko.parse_fasta_text(c["fasta_text"]), c["alphabet"]), c["k"], c["rc"])
        assert _same(got, _spectrum(np.array(counts, np.int64))), c["name"]


def test_wide_32_byte_keys(eng):
    """k > 32 with N / IUPAC windows: the wide stream has 256-bit keys (kmg_sort256 + kmg_count_histogram)."""
    recs = _mixed_records(400_000, 5)
    for k, rc in ((40, True), (63, False), (64, True)):
        _check(eng, recs, k, rc)


# ---- the fused pipeline (about 3 Mbp) ---------------------------------------------------------------------
@pytest.mark.parametrize("pb", [16, 24])
@pytest.mark.parametrize("k,rc", [(31, False), (25, True), (45, False)])
def test_fused_mixed_input(eng, pb, k, rc):
    eng.lib.kmg_set_option(b"hybrid_pb", pb)
    _check(eng, _mixed_records(3_000_000, 11), k, rc)


def test_oversize_tiles_take_the_side_path(eng):
    """Poly-A and copied stretches: tiles too big for the local sort.  The fused histogram keeps running and
    the flagged ranges are re-sorted on the side (hybrid_path 2); count falls back for the same input."""
    s = _synth(3_000_000, 21)
    recs = [("chrR", s[:1_500_000] + "A" * 30_000 + s[200_000:700_000] + s[1_500_000:] + "A" * 12_000 + s[:100_000])]
    _check(eng, recs, 31, False, "ACGT")
    assert eng.lib.kmg_get_stat(b"hybrid_path") == 2
    assert eng.lib.kmg_get_stat(b"hybrid_irregular") > 0


def test_irregular_keys_beyond_the_gather_buffer(eng):
    """More than n / 8 keys in oversize tiles: the keys are sorted in full (hybrid_path 3)."""
    s = _synth(1_300_000, 22)
    recs = [("chrA", s[:600_000] + "A" * 400_000 + s[600_000:] + "C" * 200_000)]
    _check(eng, recs, 31, False, "ACGT")
    assert eng.lib.kmg_get_stat(b"hybrid_path") == 3


def test_multiplicities_beyond_the_bins(eng):
    """A 300-base stretch copied more than KMG_HISTO_BINS times: those k-mers go to the list."""
    s = _synth(1_000_000, 23)
    recs = [("chrB", s[:500_000] + s[600_000:600_300] * 5_000 + s[500_000:]), ("chrC", s[600_000:600_300] * 300)]
    for k, rc in ((31, False), (21, True), (40, False)):
        got = _check(eng, recs, k, rc, "ACGT")
        assert got[0][-1] >= HISTO_BINS


def test_one_bucket_tiles_take_the_first_local_sort_kernel(eng):
    """The regime of test_hybrid_one_bucket_tiles_take_the_first_local_sort_kernel: 72 M random 62-bit keys,
    a third of them repeating another, a 16-bit prefix and tiles of 2048 positions pick local_sort_kernel."""
    import torch

    from kman_b200.engine import KeyArray

    n, bits = 72_000_000, 62
    rng = np.random.default_rng(1099)
    raw = rng.integers(0, 1 << 62, size=n, dtype=np.uint64)
    raw[1::3] = raw[::3]
    eng.lib.kmg_set_option(b"hybrid_pb", 16)
    eng.lib.kmg_set_option(b"local_tile", 2048)
    acc = torch.zeros(8 * (HISTO_BINS + 1) + 4 * (n // HISTO_BINS + 1), dtype=torch.uint8, device=eng.device)
    keys = torch.from_numpy(raw.view(np.uint8)).to(eng.device)
    a = KeyArray(keys, torch.empty_like(keys), None, None, n, 8, 0, bits // 2, False)
    eng.sort_histo(a, (acc.data_ptr(), acc.data_ptr() + 8 * (HISTO_BINS + 1), acc.data_ptr() + 8 * HISTO_BINS))
    assert eng.lib.kmg_get_stat(b"hybrid_path") == 1
    assert eng.lib.kmg_get_stat(b"sort_passes") == 2
    h = acc[: 8 * (HISTO_BINS + 1)].cpu().numpy().view(np.uint64)
    want_m, want_c = _spectrum(np.unique(raw, return_counts=True)[1])
    assert h[HISTO_BINS] == 0
    assert np.array_equal(np.flatnonzero(h[:HISTO_BINS]), want_m.astype(np.int64))
    assert np.array_equal(h[want_m.astype(np.int64)], want_c)


def test_forced_passes_equal_one_pass(eng):
    recs = _mixed_records(3_000_000, 31)
    d = _upload(eng, recs, "IUPAC")
    one = eng.histogram(d, 31, True)
    plan = eng.plan_passes(d, 31, True, "histo")
    assert plan.n_passes == 1
    budget = plan.pass_bytes[0] // 3 + eng._resident_bytes(d)
    fh = io.BytesIO()
    plan = eng.write_histogram(d, 31, True, fh, budget_bytes=budget)
    assert plan.n_passes > 1
    multi = eng.histogram(d, 31, True, budget_bytes=budget)
    assert _same(multi, one) and _same(one, _want(recs, 31, True, "IUPAC"))
    assert fh.getvalue() == "".join("%d\t%d\n" % mc for mc in zip(one[0].tolist(), one[1].tolist())).encode()


# ---- the command --------------------------------------------------------------------------------------
def _cli(*argv):
    from click.testing import CliRunner

    from kman_b200.scripts import kmer

    return CliRunner().invoke(kmer.main, list(argv))


def test_cli_output_file(eng, tmp_path):
    recs = _mixed_records(500_000, 41)
    inp, out = tmp_path / "in.fa", tmp_path / "out.tsv"
    inp.write_bytes(ko.synth_fasta_bytes([(n, s.encode()) for n, s in recs]))
    for rc in (False, True):
        r = _cli("histo", str(inp), str(out), "31", *(["-r"] if rc else []))
        assert r.exit_code == 0, (r.output, r.exception)
        m, c = _want(ko.read_fasta(str(inp)), 31, rc, os.environ.get("KMG_ALPHABET", "IUPAC").upper())
        assert out.read_bytes() == "".join("%d\t%d\n" % mc for mc in zip(m.tolist(), c.tolist())).encode()


def test_cli_empty_result_and_k_errors(eng, tmp_path):
    inp, out = tmp_path / "in.fa", tmp_path / "out.tsv"
    inp.write_bytes(b">r1\nACGTACGTNNNN\n>r2\nACG\n")
    r = _cli("histo", str(inp), str(out), "20")
    assert r.exit_code == 0, (r.output, r.exception)
    assert out.exists() and out.read_bytes() == b""
    r = _cli("histo", str(inp), str(out), "1")
    assert isinstance(r.exception, AssertionError)
    r = _cli("histo", str(inp), str(out), "65")
    assert isinstance(r.exception, ValueError)


# ---- config 2 (100 Mbp, k = 31) ---------------------------------------------------------------------------
@pytest.mark.parametrize("dup", [False, True])
def test_cfg2_histogram_matches_count(eng, dup):
    recs = sc.cfg2(100_000_000, dup=dup)
    d = _upload(eng, recs, "ACGT")
    mult, n_kmers = eng.histogram(d, 31, False)
    n_keys, _ = eng.count_windows(d, 31, False)
    assert int((mult * n_kmers).sum()) == n_keys
    tabs = eng.count(d, 31, False)
    assert int(n_kmers.sum()) == sum(t.n for t in tabs)
    assert _same((mult, n_kmers), _spectrum(np.concatenate([t.counts_host() for t in tabs])))
