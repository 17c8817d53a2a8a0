"""Canonical k-mers (`--canonical`, rc = KMG_CANONICAL) without a GPU: the two oracle tiers against each other, the
oracle against the reference's own `-r` outputs (three identities), option parsing and rejection, the header
constant and the pass plan's key count."""
import os
import random
import re
from collections import Counter

import numpy as np
import pytest

import canonical_oracle as co

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cli(*argv):
    from click.testing import CliRunner

    from kman_b200.scripts import kmer

    return CliRunner().invoke(kmer.main, list(argv))


def _rand_records(rng, n_rec, length, symbols, lower=0.05):
    recs = []
    for r in range(n_rec):
        s = "".join(rng.choice(symbols) for _ in range(length))
        s = "".join(c.lower() if rng.random() < lower else c for c in s)
        recs.append((f"r{r} t", s))
    return recs


@pytest.mark.parametrize("alphabet,natype", [("IUPAC", "DNA"), ("IUPAC", "RNA"), ("ACGT", "DNA"), ("ACGT", "RNA")])
@pytest.mark.parametrize("k", [2, 3, 8, 16, 31, 32, 33, 45, 64])
def test_oracle_tiers_agree(alphabet, natype, k):
    import kmer_oracle as ko

    rng = random.Random(k * 7 + len(alphabet) + len(natype))
    plain = "ACG" + ("T" if natype == "DNA" else "U")
    # mostly plain bases, some IUPAC symbols and N, some bytes outside the alphabet, a palindrome-rich record
    symbols = plain * 12 + "NRYKMSWBDHV" + "X"
    recs = _rand_records(rng, 3, 300, symbols)
    pal = ("ACGT" if natype == "DNA" else "ACGU") * 40
    recs.append(("pal", pal + "GAATTC" * 10 + ("AATT" if natype == "DNA" else "AAUU") * 8))
    # a stretch pasted back as its reverse complement: canonical merging matters
    src = re.sub("[Xx]", "A", recs[0][1][:150])
    if alphabet == "ACGT":
        src = re.sub("[^ACGTUacgtu]", "C", src).replace("U" if natype == "DNA" else "T", "G")
    recs.append(("back", recs[0][1][:150] + ko.mkrc_py(src, ko.ALPHABETS[alphabet][natype])))
    for py_fn, np_fn in ((co.count_text_py, co.count_text_np), (co.uniq_text_py, co.uniq_text_np)):
        assert np_fn(recs, k, alphabet, natype) == py_fn(recs, k, alphabet, natype)


def _rc_of(golden_case):
    import kmer_oracle as ko

    ab = ko.ALPHABETS[golden_case["alphabet"]]["DNA"]
    return lambda s: ko.mkrc_py(s, ab)


def _rc_cases(golden):
    return [c for c in golden["cases"] if c["rc"] and "count" in c and "uniq" in c]


def test_identities_against_the_reference_rc_outputs(golden):
    """The reference's `-r` texts (tests/golden/golden.json) pin the canonical oracle:
    count: the -r table restricted to rows with seq <= rc(seq), palindrome counts halved;
    uniq: the -r records with seq <= rc(seq) (same coordinates and strand) plus the palindromes that occur once;
    histo: the spectrum of the canonical table, with sum(m * n(m)) = the number of valid windows."""
    import kmer_oracle as ko

    cases = _rc_cases(golden)
    assert len(cases) >= 10
    n_pal = 0
    for c in cases:
        recs = ko.parse_fasta_text(c["fasta_text"])
        k, alphabet, rc = c["k"], c["alphabet"], _rc_of(c)
        # count
        rows = []
        for line in c["count"].splitlines():
            seq, n = line.split("\t")
            r = rc(seq)
            if seq < r:
                rows.append((seq, int(n)))
            elif seq == r:
                assert int(n) % 2 == 0
                rows.append((seq, int(n) // 2))
                n_pal += 1
        want = "".join("%s\t%d\n" % x for x in rows).encode()
        assert co.count_text_np(recs, k, alphabet) == want, c["name"]
        assert co.count_text_py(recs, k, alphabet) == want, c["name"]
        # uniq
        lines = c["uniq"].splitlines()
        keep = [(lines[i], lines[i + 1]) for i in range(0, len(lines), 2) if lines[i + 1] < rc(lines[i + 1])]
        # palindromes seen exactly once in the canonical count are singletons: -r counts them twice
        once = {seq for seq, n in rows if n == 1 and seq == rc(seq)}
        if once:
            canon = co.uniq_text_py(recs, k, alphabet).decode().splitlines()
            pal = [(canon[i], canon[i + 1]) for i in range(0, len(canon), 2) if canon[i + 1] in once]
            assert len(pal) == len(once) and all(h.endswith(":+") for h, _ in pal)
            keep = sorted(keep + pal, key=lambda hs: hs[1])
        want = "".join(">%s\n%s\n" % (h[1:], s) for h, s in keep).encode()
        assert co.uniq_text_np(recs, k, alphabet) == want, c["name"]
        # histo: the spectrum of the canonical table; every valid window counted once
        ex = ko.extract_np(recs, k, alphabet=alphabet)
        n_valid = ex["narrow"]["pos"].size + ex["wide"]["pos"].size
        spectrum = Counter(n for _, n in rows)
        assert sum(m * nm for m, nm in spectrum.items()) == n_valid, c["name"]
    assert n_pal > 0  # even k goldens hold palindromes


def test_palindromes_count_once_with_strand_plus():
    recs = [("p", "ACGT" * 6), ("q", "GAATTC")]
    assert co.count_text_py(recs, 4) == b"AATT\t1\nACGT\t6\nATTC\t2\nCGTA\t10\nGTAC\t5\n"
    assert co.count_text_py(recs, 6) == b"ACGTAC\t10\nCGTACG\t5\nGAATTC\t1\nTACGTA\t4\n"
    assert co.uniq_text_py(recs, 6) == b">q:0-6:+\nGAATTC\n"
    # strand '-' exactly when the reverse complement is strictly smaller
    assert co.uniq_text_py([("m", "TTTG")], 4) == b">m:0-4:-\nCAAA\n"


def test_header_constant():
    from kman_b200 import _lib, engine

    hdr = open(os.path.join(ROOT, "include", "kmg.h")).read()
    assert int(re.search(r"#define KMG_CANONICAL (\d+)", hdr).group(1)) == _lib.KMG_CANONICAL == engine.CANONICAL
    assert [engine.keys_per_window(rc) for rc in (False, True, 0, 1, engine.CANONICAL)] == [1, 2, 1, 2, 1]


def test_cli_option_is_long_only():
    for cmd in ("count", "uniq", "histo"):
        r = _cli(cmd, "--help")
        assert r.exit_code == 0 and "--canonical" in r.output
        assert not re.search(r"-\w, --canonical", r.output)  # (-C is the reference's --compress)


@pytest.mark.parametrize("argv", [
    ["count", "-r", "--canonical"],
    ["uniq", "-r", "--canonical"],
    ["histo", "-r", "--canonical"],
    ["count", "--canonical", "-m", "VEC_COUNT"],
    ["count", "--canonical", "-m", "VEC_COUNT_MASKED"],
    ["count", "--canonical", "--min-count", "2", "-r"],
    ["count", "--canonical", "-B", "{batches}"],
    ["uniq", "--canonical", "-B", "{batches}"],
])
def test_cli_rejections_before_any_work(tmp_path, argv):
    inp, out, batches = tmp_path / "in.fa", tmp_path / "out", tmp_path / "batches"
    inp.write_bytes(b">r\nACGTACGT\n")
    batches.mkdir()
    (batches / "b0.fa").write_bytes(b">r:0-4:+\nACGT\n")
    argv = [a.format(batches=batches) for a in argv]
    r = _cli(argv[0], str(inp), str(out), "4", *argv[1:])
    assert isinstance(r.exception, AssertionError), (r.output, r.exception)
    assert not out.exists()


def test_batcher_and_engine_rejections():
    from kman_b200.batcher import FastaBatcher
    from kman_b200.engine import CANONICAL, Engine

    with pytest.raises(AssertionError):
        FastaBatcher(reverse=True, canonical=True)
    with pytest.raises(AssertionError):
        FastaBatcher(canonical=CANONICAL)  # the batcher takes a bool
    assert FastaBatcher(canonical=True).canonical and not FastaBatcher().canonical
    eng = object.__new__(Engine)  # (the checks come before any device work)
    for call in (lambda: Engine.abundance.__wrapped__(eng, None, 31, CANONICAL),
                 lambda: Engine.write_vectors.__wrapped__(eng, None, 31, CANONICAL, False, "/nonexistent"),
                 lambda: Engine.write_batch(eng, None, 31, CANONICAL, None)):
        with pytest.raises(AssertionError):
            call()
    from kman_b200.dist import DistributedCounter

    dc = object.__new__(DistributedCounter)
    for call in (lambda: dc.count(None, 31, CANONICAL), lambda: dc.uniq(None, 31, CANONICAL)):
        with pytest.raises(AssertionError):
            call()


def test_joiner_checks_canonical_consistency():
    from kman_b200.batch import DeviceBatch
    from kman_b200.join import KJoiner

    class DI:
        alphabet = "IUPAC"

    def batch(canonical):
        b = object.__new__(DeviceBatch)
        b.k, b.reverse, b.canonical, b.natype, b.device_input = 21, False, canonical, None, DI()
        return b

    with pytest.raises(AssertionError):
        KJoiner._merged_device_input([batch(True), batch(False)])
    with pytest.raises(AssertionError):
        DeviceBatch(None, None, 21, True, None, "/tmp", canonical=True)
    from kman_b200.engine import CANONICAL

    assert batch(True).strand_rule == CANONICAL and batch(False).strand_rule is False


@pytest.mark.parametrize("mode", ["count", "uniq", "histo"])
def test_plan_uses_one_key_per_window(mode):
    """plan_passes(..., CANONICAL): the totals, the one-pass bytes and every pass are sized for one key per window,
    as forward-only, and half of what -r plans."""
    from kman_b200 import _lib
    from kman_b200.engine import CANONICAL, Engine

    n_win, n_valid, n_wide = 3_000_000_000, 2_900_000_000, 1_000_000

    class D:
        n_bases = n_win + 30
        payload_bytes = 8

    class Stub:
        lib = _lib.load()
        seen = []

        def device_budget(self, d, budget_bytes=None):
            return budget_bytes

        def _text_plan(self, d, k, mode, chunk_rows):
            return 1 << 20, 64 << 20

        def count_windows(self, d, k, rc):
            return n_valid * (2 if rc is True else 1), n_wide

        def _one_pass_bytes(self, *a):
            return Engine._one_pass_bytes(self, *a)

        def part_counts(self, d, k, rc, n_parts):
            self.seen.append(rc)
            narrow = np.full(n_parts, n_valid * (2 if rc is True else 1) // n_parts, np.int64)
            return narrow, np.full(n_parts, n_wide * (2 if rc is True else 1) // n_parts, np.int64)

    plan = {}
    for rc in (False, True, CANONICAL):
        plan[rc] = Engine.plan_passes.__wrapped__(Stub(), D(), 31, rc, mode, 100 << 30)
    assert plan[CANONICAL].narrow.sum() == plan[False].narrow.sum() == n_valid // 256 * 256
    assert plan[CANONICAL].wide.sum() == plan[False].wide.sum()
    assert plan[CANONICAL].pass_bytes == plan[False].pass_bytes
    assert plan[True].narrow.sum() == 2 * plan[CANONICAL].narrow.sum()
    assert plan[CANONICAL].n_passes <= plan[True].n_passes
    assert Stub.seen.count(CANONICAL) == (plan[CANONICAL].n_parts > 1)
    s = Stub()
    one_c = Engine._one_pass_bytes(s, D(), 31, CANONICAL, mode, n_wide, 8, 0)
    assert one_c == Engine._one_pass_bytes(s, D(), 31, False, mode, n_wide, 8, 0)
    assert one_c < Engine._one_pass_bytes(s, D(), 31, True, mode, n_wide, 8, 0)


def test_workspace_queries_take_the_canonical_rule():
    from kman_b200 import _lib
    from kman_b200.engine import CANONICAL

    lib = _lib.load()
    for n in (1000, 1 << 22, 3_000_000_000):
        for k in (16, 31, 45):
            c = lib.kmg_pipeline_workspace_bytes(n, k, CANONICAL, 8)
            assert c == lib.kmg_pipeline_workspace_bytes(n, k, 0, 8) <= lib.kmg_pipeline_workspace_bytes(n, k, 1, 8)
            h = lib.kmg_pipeline_histo_workspace_bytes(n, k, CANONICAL)
            assert h == lib.kmg_pipeline_histo_workspace_bytes(n, k, 0) <= lib.kmg_pipeline_histo_workspace_bytes(n, k, 1)
