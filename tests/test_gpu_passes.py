"""Key-range passes on the GPU: kmg_extract_parts against kmg_extract filtered in numpy, per-pass tables
against the golden table hashes, write_count / write_uniq (and the command line) byte for byte against the
oracle and the reference's golden outputs under a forced multi-pass budget, and write_batch in chunks
against the oracle's batch file."""
import io
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import synth_configs as sc  # noqa: E402  (oracle/ is on sys.path, see conftest.py)

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
IUPAC_OTHER = np.frombuffer(b"RYKMSWBDHVN", np.uint8)


@pytest.fixture(scope="module")
def eng():
    from kman_b200.engine import get_engine

    return get_engine()


def iupac_records(n: int, seed: int):
    """Random ACGT (partly lower case) with isolated IUPAC symbols and N runs: many wide windows hold
    a non-plain symbol inside their first 4 positions, so their part is not that of a plain prefix."""
    rng = np.random.default_rng(seed)
    b = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n)].copy()
    at = rng.integers(0, n, n // 150)
    b[at] = IUPAC_OTHER[rng.integers(0, IUPAC_OTHER.size, at.size)]
    for s in rng.integers(0, n - 200, 12):
        b[s:s + rng.integers(1, 150)] = ord("N")
    low = rng.integers(0, n - 500, 20)
    for s in low:
        b[s:s + 300] |= 0x20
    cut = n // 3
    return [("chrA first", b[:cut].tobytes().decode()), ("chrB", b[cut:].tobytes().decode())]


def field(rows: np.ndarray, shift: int, width: int) -> np.ndarray:
    """Bits [shift, shift+width) of keys given as (n,) uint64 or (n, L) uint64 limbs, least significant first."""
    if width == 0:
        return np.zeros(rows.shape[0], np.int64)
    r = rows[:, None] if rows.ndim == 1 else rows
    w, o = divmod(shift, 64)
    v = r[:, w] >> np.uint64(o)
    if o + width > 64:
        v = v | (r[:, w + 1] << np.uint64(64 - o))
    return (v & np.uint64((1 << width) - 1)).astype(np.int64)


def parts_of(a, k: int, n_parts: int, rna: int) -> np.ndarray:
    from kman_b200.engine import wide_part_table

    keys = a.keys_host()
    b = n_parts.bit_length() - 1
    if not a.wide:
        return field(keys, 2 * k - b, b)
    return wide_part_table(rna, n_parts)[field(keys, 4 * k - 16, 16)].astype(np.int64)


IUPAC_RECS = iupac_records(300_000, 77)


@pytest.fixture(scope="module")
def dev_iupac(eng):
    from kman_b200 import fasta

    return eng.upload(fasta.from_records(IUPAC_RECS), alphabet="IUPAC")


@pytest.mark.parametrize("k", [12, 25, 31, 33, 45, 63])
@pytest.mark.parametrize("rc", [False, True])
@pytest.mark.parametrize("n_parts", [2, 16, 256])
def test_extract_parts_equals_filtered_extract(eng, dev_iupac, k, rc, n_parts):
    d = dev_iupac
    narrow_c, wide_c = eng.part_counts(d, k, rc, n_parts)
    for wide, want_c in ((False, narrow_c), (True, wide_c)):
        full = eng.extract(d, k, rc, wide=wide, val_bytes=4)
        assert full.n > 0
        fk, fv = full.keys_host(), full.vals_host()
        part = parts_of(full, k, n_parts, d.rna)
        assert np.array_equal(np.bincount(part, minlength=n_parts), want_c), "per-part counts"
        assert int(want_c.sum()) == full.n
        h = n_parts // 2
        ranges = {(0, 1), (n_parts - 1, n_parts), (h, h), (0, n_parts), (1, max(2, h + 1))}
        for lo, hi in sorted(ranges):
            sel = (part >= lo) & (part < hi)
            got = eng.extract_parts(d, k, rc, wide, 4, n_parts, lo, hi, int(sel.sum()))
            assert got.n == int(sel.sum())
            assert np.array_equal(got.keys_host(), fk[sel]), (wide, lo, hi)
            assert np.array_equal(got.vals_host(), fv[sel]), (wide, lo, hi)
        if n_parts > 16:
            continue
        # the parts one by one add up to the unfiltered stream, in part order after a stable sort by part
        order = np.argsort(part, kind="stable")
        cat = [eng.extract_parts(d, k, rc, wide, 4, n_parts, p, p + 1, int(want_c[p])) for p in range(n_parts)]
        assert np.array_equal(np.concatenate([c.vals_host() for c in cat]), fv[order])


def test_extract_parts_rejects_histograms_and_bad_ranges(eng, dev_iupac):
    from kman_b200 import _lib

    d = dev_iupac
    n_win = d.n_bases - 31 + 1
    ws_bytes = eng.lib.kmg_extract_workspace_bytes(n_win)
    ws = eng._new(ws_bytes)
    keys = eng._new(2 * n_win * 8)
    hist = eng._new(16 * 256 * 8)
    tab = eng._wide_parts(d.rna, 16)

    def call(lo, hi, h=None, n_parts=16):
        return eng.lib.kmg_extract_parts(d.bases.data_ptr(), d.n_bases, 0, n_win, 31, 0, 0, d.lut.data_ptr(),
                                         d.comp16.data_ptr(), n_parts, lo, hi, tab.data_ptr(), keys.data_ptr(), 8, None, 0,
                                         0, eng._small.data_ptr(), h, ws.data_ptr(), ws_bytes, eng._stream())

    assert call(0, 16, hist.data_ptr()) == _lib.KMG_ERR_ARG
    assert call(3, 2) == _lib.KMG_ERR_ARG
    assert call(0, 17) == _lib.KMG_ERR_ARG
    assert call(0, 12, n_parts=12) == _lib.KMG_ERR_ARG
    assert call(0, 16) == _lib.KMG_OK


def forced_budget(eng, d, k, rc, mode, passes=4, chunk_rows=None, slack=0):
    """A device budget under which plan_passes needs about `passes` passes (never below the largest part)."""
    from kman_b200.engine import pass_bytes

    narrow, wide = eng.part_counts(d, k, rc, 256)
    _, text_bytes = eng._text_plan(d, k, mode, chunk_rows)
    n_win = max(0, d.n_bases - k + 1)
    cost = lambda a, b: pass_bytes(k, mode, a, b, d.payload_bytes, text_bytes, n_win)  # noqa: E731
    target = cost(-(-int(narrow.sum()) // passes), -(-int(wide.sum()) // passes))
    biggest = max(cost(int(a), int(b)) for a, b in zip(narrow, wide))
    return max(target, biggest) + eng._resident_bytes(d) + slack


GOLD = json.load(open(os.path.join(HERE, "golden", "table_hashes.json")))
from test_gpu_golden_tables import MAKERS  # noqa: E402


@pytest.mark.parametrize("name", sorted(GOLD))
def test_pass_tables_match_golden_hashes(eng, name):
    import torch

    from kman_b200 import fasta

    g = GOLD[name]
    recs = MAKERS[name]()
    d = eng.upload(fasta.from_records(recs), alphabet=g["alphabet"], with_names=False)
    del recs
    k, rc, mode = g["k"], g["rc"], g["mode"]
    plan = eng.plan_passes(d, k, rc, mode, budget_bytes=forced_budget(eng, d, k, rc, mode))
    assert plan.n_parts == 256 and plan.n_passes >= 4, plan.parts
    cols = {"narrow": [[], []], "wide": [[], []]}
    for tabs in eng.pass_tables(d, k, rc, mode, plan):
        for sname, t in zip(("narrow", "wide"), tabs):
            cols[sname][0].append(np.ascontiguousarray(t.keys_host(), dtype=np.uint64))
            cols[sname][1].append(t.counts_host() if mode == "count" else t.vals_host().astype(np.uint64))
    for sname in ("narrow", "wide"):
        want = g[sname]
        ks, vs = cols[sname]
        if not ks:
            assert want["rows"] == 0, sname
            continue
        keys, vals = np.concatenate(ks), np.concatenate(vs)
        got = sc.count_digest(keys, vals) if mode == "count" else sc.uniq_digest(keys, vals)
        assert got == {kk: want[kk] for kk in got}, sname
    del d
    torch.cuda.empty_cache()


def _write(eng, d, k, rc, mode, **kw) -> bytes:
    fh = io.BytesIO()
    plan = (eng.write_count if mode == "count" else eng.write_uniq)(d, k, rc, fh, **kw)
    return fh.getvalue(), plan


@pytest.mark.parametrize("k,rc", [(12, True), (25, False), (31, True), (40, True), (63, False)])
@pytest.mark.parametrize("mode", ["count", "uniq"])
def test_write_multi_pass_equals_text(eng, dev_iupac, k, rc, mode):
    import kmer_oracle as ko

    d = dev_iupac
    want = (ko.count_text_np if mode == "count" else ko.uniq_text_np)(IUPAC_RECS, k, rc, "IUPAC")
    got, plan = _write(eng, d, k, rc, mode, chunk_rows=5000,
                       budget_bytes=forced_budget(eng, d, k, rc, mode, passes=6, chunk_rows=5000))
    assert plan.n_passes >= 4 and len(plan.pass_ms) == plan.n_passes
    assert got == want
    # one-pass plan, default budget, chunks: same bytes
    got1, plan1 = _write(eng, d, k, rc, mode, chunk_rows=7777)
    assert plan1.n_passes == 1 and got1 == want


def test_write_matches_reference_goldens(eng, golden):
    """The reference's own outputs: the small cases (both alphabets, +/- -r; k < 12, so one pass) in chunks
    of 3 rows, the synthetic ones (k >= 12) under a forced multi-pass budget."""
    import hashlib

    import kmer_oracle as ko

    from kman_b200 import fasta

    bad = []
    for c in golden["cases"]:
        d = eng.upload(fasta.parse_bytes(c["fasta_text"].encode("latin-1")), alphabet=c["alphabet"])
        for mode in ("count", "uniq"):
            got, plan = _write(eng, d, c["k"], c["rc"], mode, chunk_rows=3)
            if got != c[mode].encode("latin-1"):
                bad.append((c["name"], c["k"], c["alphabet"], c["rc"], mode, got[:80], c[mode][:80]))
    assert not bad, (len(bad), bad[:5])
    for ent in golden["synthetic"]:
        if ent["name"] == "syn_dup":
            data = ent["fasta_text"].encode()
        else:
            data = ko.synth_fasta_bytes([("chr1 synthetic seed=%d" % ent["seed"], ko.synth_bases(ent["n"], ent["seed"]))])
        d = eng.upload(fasta.parse_bytes(data))
        k, rc = ent["k"], ent.get("rc", False)
        for mode in ("count", "uniq"):
            kw = {"chunk_rows": 4000}
            if k >= 12:
                kw["budget_bytes"] = forced_budget(eng, d, k, rc, mode, passes=4, chunk_rows=4000)
            got, plan = _write(eng, d, k, rc, mode, **kw)
            assert plan.n_passes >= (2 if k >= 12 else 1), (ent["name"], k, rc, mode, plan.parts)
            assert (got.count(b"\n"), hashlib.sha256(got).hexdigest()) == (ent[mode + "_lines"], ent[mode + "_sha256"]), \
                (ent["name"], k, rc, mode, plan.n_passes)


def test_cli_multi_pass_output_file(eng, tmp_path):
    import kmer_oracle as ko

    from kman_b200 import fasta

    recs = iupac_records(200_000, 5)
    fa = tmp_path / "in.fa"
    fa.write_bytes(b"".join(b">%s\n%s\n" % (n.encode(), s.encode()) for n, s in recs))
    d = eng.upload(fasta.from_records(recs), alphabet="IUPAC")
    for mode, args, k, rc in (("count", [], 31, False), ("uniq", ["-r"], 27, True)):
        want = (ko.count_text_np if mode == "count" else ko.uniq_text_np)(recs, k, rc, "IUPAC")
        budget = forced_budget(eng, d, k, rc, mode, passes=4, slack=4 * fa.stat().st_size)
        out = tmp_path / f"out_{mode}.txt"
        env = dict(os.environ, PYTHONPATH=ROOT, KMG_ALPHABET="IUPAC", KMG_DEVICE_BUDGET=str(budget))
        subprocess.run([sys.executable, "-m", "kman_b200.scripts.kmer", mode, *args, str(fa), str(out), str(k)],
                       check=True, env=env, cwd=str(tmp_path), stdout=subprocess.DEVNULL)
        assert out.read_bytes() == want, mode
        plan = eng.plan_passes(d, k, rc, mode, budget_bytes=budget)
        assert plan.n_passes >= 2


@pytest.mark.parametrize("k", [7, 25, 40])
def test_write_batch_in_chunks_equals_oracle(eng, k):
    """`kmer batch`'s sorted export with N / IUPAC windows: in chunks of 3 and 1000 rows and in one chunk, the wide
    lines fall inside chunks, at chunk edges and after the last narrow row (windows starting with Y sort after T)."""
    import kmer_oracle as ko

    from kman_b200 import fasta

    rng = np.random.default_rng(500 + k)
    s1 = "".join(rng.choice(list("ACGT"), size=5000))
    s2 = "".join(rng.choice(list("ACGT"), size=3000))
    recs = [("chrA first", s1 + s1[:800].lower() + "NNNNNNNNNNRY" + s1[100:400]), ("chrB", s2 + "N" + s2[:500] + "ACGTN")]
    d = eng.upload(fasta.from_records(recs), alphabet="IUPAC")
    (want,) = ko.batch_text_py(recs, k, True, alphabet="IUPAC")
    for chunk_rows in (3, 1000, None):
        fh = io.BytesIO()
        eng.write_batch(d, k, True, fh, chunk_rows=chunk_rows)
        assert fh.getvalue() == want, chunk_rows


def test_empty_result_leaves_empty_output(eng):
    from kman_b200 import fasta

    d = eng.upload(fasta.from_records([("r", "ACGTNACGT")]), alphabet="IUPAC")
    for mode in ("count", "uniq"):
        got, plan = _write(eng, d, 31, False, mode)
        assert got == b"" and plan.n_passes == 1


def test_budget_below_largest_part_raises(eng, dev_iupac):
    from kman_b200.engine import pass_bytes

    d = dev_iupac
    k, rc = 31, True
    narrow, wide = eng.part_counts(d, k, rc, 256)
    _, text_bytes = eng._text_plan(d, k, "count", None)
    biggest = max(pass_bytes(k, "count", int(a), int(b), 4, text_bytes, d.n_bases - k + 1) for a, b in zip(narrow, wide))
    with pytest.raises(ValueError, match="needs"):
        eng.write_count(d, k, rc, io.BytesIO(), budget_bytes=biggest - 1 + eng._resident_bytes(d))
    with pytest.raises(ValueError, match="k >= 12"):
        eng.write_count(d, 11, rc, io.BytesIO(), budget_bytes=eng._resident_bytes(d) + 1000)
