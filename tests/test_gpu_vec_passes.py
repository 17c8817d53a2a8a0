"""Abundance vectors (`kmer count -m VEC_COUNT / VEC_COUNT_MASKED`) in key-range passes with device text:
Engine.write_vectors under forced multi-pass budgets against the oracle, kmg_format_vector against
abundance.vector_text, kmg_vector_extents against numpy, the command line with KMG_DEVICE_BUDGET, and the
errors and directory semantics of the writer."""
import gzip
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
IUPAC_OTHER = np.frombuffer(b"RYKMSWBDHVN", np.uint8)


@pytest.fixture(scope="module")
def eng():
    from kman_b200.engine import get_engine

    return get_engine()


def vec_records(n: int, seed: int):
    """Random ACGT with isolated IUPAC symbols, N runs and soft-masked stretches; stretches copied inside a record
    and across records (counts above 1, masked groups spanning records); a record shorter than k, an empty one."""
    rng = np.random.default_rng(seed)
    b = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n)].copy()
    at = rng.integers(0, n, n // 300)
    b[at] = IUPAC_OTHER[rng.integers(0, IUPAC_OTHER.size, at.size)]
    for s in rng.integers(0, n - 200, 6):
        b[s:s + rng.integers(1, 120)] = ord("N")
    cut1, cut2 = n // 3, 2 * n // 3
    b[cut1 + 1000:cut1 + 4000] = b[2000:5000]        # record A -> record B
    b[cut2 + 500:cut2 + 2500] = b[cut1 + 5000:cut1 + 7000]  # record B -> record C
    b[7000:8500] = b[12000:13500]                    # inside record A
    b[cut2 + 9000:cut2 + 9600] = b[cut2 + 500:cut2 + 1100] | 0x20  # soft-masked copy inside record C
    for s in rng.integers(0, n - 500, 8):
        b[s:s + 200] |= 0x20
    txt = b.tobytes().decode()
    return [("chrA first", txt[:cut1]), ("chrB", txt[cut1:cut2]), ("tiny", "ACGTNAC"), ("chrC", txt[cut2:] + "NNNN"),
            ("void", "")]


VEC_RECS = vec_records(120_000, 31)


@pytest.fixture(scope="module")
def dev_vec(eng):
    from kman_b200 import fasta

    return eng.upload(fasta.from_records(VEC_RECS), alphabet="IUPAC")


def forced_budget(eng, d, k, rc, passes=4, chunk_rows=None, slack=0):
    """A device budget under which plan_passes(mode="vec") needs about `passes` passes (never below the
    largest part): the resident input and the vector pair plus the cost of 1/passes of the keys."""
    from kman_b200.engine import pass_bytes

    narrow, wide = eng.part_counts(d, k, rc, 256)
    _, text_bytes = eng._text_plan(d, k, "vec", chunk_rows)
    n_win = max(0, d.n_bases - k + 1)
    cost = lambda a, b: pass_bytes(k, "vec", a, b, d.payload_bytes, text_bytes, n_win)  # noqa: E731
    target = cost(-(-int(narrow.sum()) // passes), -(-int(wide.sum()) // passes))
    biggest = max(cost(int(a), int(b)) for a, b in zip(narrow, wide))
    return max(target, biggest) + eng._resident_bytes(d) + 8 * (d.n_bases + 1) + slack


def read_dir(path) -> dict:
    return {f: gzip.open(os.path.join(path, f), "rb").read() for f in sorted(os.listdir(path))}


@pytest.mark.parametrize("k", [12, 25, 31, 40, 63])
@pytest.mark.parametrize("rc", [False, True])
@pytest.mark.parametrize("masked", [False, True])
def test_write_vectors_multi_pass_equals_oracle(eng, dev_vec, tmp_path, k, rc, masked):
    import kmer_oracle as ko

    d = dev_vec
    want = ko.vec_count_np(VEC_RECS, k, rc, masked, "IUPAC")
    assert want and (not masked or len(want) < 2 * len(VEC_RECS))
    budget = forced_budget(eng, d, k, rc, passes=5, chunk_rows=777)
    plan = eng.write_vectors(d, k, rc, masked, str(tmp_path / "vec.txt"), budget_bytes=budget, chunk_rows=777)
    assert plan.n_parts == 256 and plan.n_passes >= 4 and len(plan.pass_ms) == plan.n_passes
    assert max(plan.pass_bytes) <= budget - eng._resident_bytes(d) - 8 * (d.n_bases + 1)
    assert read_dir(tmp_path / "vec") == want
    # the pass loop gives the vectors of the one-pass plan
    assert eng.plan_passes(d, k, rc, "vec").n_passes == 1
    assert eng.plan_passes(d, k, rc, "vec", budget, text=False).n_passes >= 3
    one = eng.abundance(d, k, rc, masked)
    multi = eng.abundance(d, k, rc, masked, budget_bytes=budget)
    assert np.array_equal(one[0], multi[0]) and np.array_equal(one[1], multi[1])
    # one pass, default chunks: the same files
    plan1 = eng.write_vectors(d, k, rc, masked, str(tmp_path / "one"))
    assert plan1.n_passes == 1 and read_dir(tmp_path / "one") == want


def test_format_vector_equals_vector_text(eng):
    import torch

    from kman_b200.abundance import vector_text

    rng = np.random.default_rng(3)
    special = [0, 1, 9, 10, 99, 100, 2**32 - 1]
    digits = [rng.integers(10**i, min(10**(i + 1), 2**32), 200, dtype=np.int64) for i in range(10)]
    vals = np.concatenate([np.array(special * 20, np.int64), *digits])
    vals = vals[rng.permutation(vals.size)].astype(np.uint32)
    dev = torch.from_numpy(vals.view(np.int32)).to(eng.device)

    def want(a: np.ndarray) -> bytes:
        return vector_text(a, 7)[len(b"# k=7\n"):]

    assert eng.format_vector(dev[:0]).numel() == 0
    for v in special:
        one = torch.tensor([v], dtype=torch.int64).to(torch.int32).to(eng.device) if v < 2**31 else \
            torch.from_numpy(np.array([v], np.uint32).view(np.int32)).to(eng.device)
        assert eng.format_vector(one).cpu().numpy().tobytes() == b"%d\n" % v
    for a, b in ((0, vals.size), (3, 1030), (1, 2), (1025, 3000), (1023, 1024), (5, vals.size - 7)):
        assert eng.format_vector(dev[a:b]).cpu().numpy().tobytes() == want(vals[a:b]), (a, b)
    for chunk in (1, 3, 1000, vals.size):
        got = b"".join(eng.format_vector(dev[i:i + chunk]).cpu().numpy().tobytes() for i in range(0, vals.size, chunk))
        assert got == want(vals), chunk
    # into a caller's buffer
    buf = eng._new(11 * vals.size)
    text = eng.format_vector(dev, buf)
    assert text.data_ptr() == buf.data_ptr() and text.cpu().numpy().tobytes() == want(vals)


def test_vector_extents_against_numpy(eng):
    """Records of 0 .. 12000 positions (tiles of 4096 positions inside one record and across records), vectors
    all zero, sparse, dense, with their last entry set and with only their first entry set."""
    import torch

    from kman_b200 import fasta

    lens = [0, 1, 5000, 4095, 4096, 9000, 3, 0, 12000, 2]
    d = eng.upload(fasta.from_records([("r%d" % i, "A" * n) for i, n in enumerate(lens)]), alphabet="ACGT")
    starts = d.flat.rec_starts.astype(np.int64)
    rng = np.random.default_rng(9)
    vec = np.zeros((2, d.n_bases + 1), np.uint32)
    for r, n in enumerate(lens):
        for s in (0, 1):
            b = int(starts[r])
            kind = (r + 3 * s) % 5
            if n == 0 or kind == 0:
                continue
            if kind == 1:
                vec[s, b + rng.integers(0, n, max(1, n // 50))] = rng.integers(1, 1000, max(1, n // 50))
            elif kind == 2:
                vec[s, b:b + n] = rng.integers(0, 3, n)
            elif kind == 3:
                vec[s, b + n - 1] = 4_000_000_000
            else:
                vec[s, b] = 1
    plus, minus = (torch.from_numpy(v.view(np.int32).copy()).to(eng.device) for v in vec)
    got = eng.vector_extents(d, plus, minus)
    want = np.zeros((len(lens), 2), np.int64)
    for r in range(len(lens)):
        for s in (0, 1):
            nz = np.flatnonzero(vec[s, starts[r]:starts[r + 1] - 1])
            want[r, s] = nz[-1] + 1 if nz.size else 0
    assert np.array_equal(got, want), (got, want)


def test_vector_files_trimmed_and_skipped(eng, tmp_path):
    """No file for an all-zero vector ('-' without -r; masked, a record that shares nothing), trailing zeros
    trimmed (a record ending in N, invalid in the ACGT alphabet), a record exactly k long, empty records; in
    chunks of 1 and 3 entries and in one chunk."""
    import kmer_oracle as ko

    from kman_b200 import fasta

    k = 21
    rng = np.random.default_rng(21)
    s1, s2, s3 = ("".join(rng.choice(list("ACGT"), size=n)) for n in (600, 400, 300))
    recs = [("plain", s1), ("endsN", s2 + "NNNNN"), ("exact", s3[:k]), ("empty", ""), ("short", "ACG"),
            ("shared", s1[100:400] + s3[50:250] + "NN"), ("alone", s3[:250][::-1])]
    d = eng.upload(fasta.from_records(recs), alphabet="ACGT")
    for rc in (False, True):
        for masked in (False, True):
            want = ko.vec_count_np(recs, k, rc, masked, "ACGT")
            if not rc:
                assert not any(f.endswith("___-.gz") for f in want)
            if masked:
                assert "alone___+.gz" not in want and "plain___+.gz" in want
            else:
                assert want["exact___+.gz"] == b"# k=21\n1\n"
            assert "empty___+.gz" not in want and "short___+.gz" not in want
            for chunk_rows in (1, 3, None):
                out = tmp_path / f"v_{rc}_{masked}_{chunk_rows}"
                eng.write_vectors(d, k, rc, masked, str(out) + ".txt", chunk_rows=chunk_rows)
                assert read_dir(out) == want, (rc, masked, chunk_rows)
    assert read_dir(tmp_path / "v_False_False_None")["endsN___+.gz"].count(b"\n") == 1 + len(s2) - k + 1


@pytest.mark.parametrize("mode,rc,k", [("VEC_COUNT", False, 31), ("VEC_COUNT", True, 25),
                                       ("VEC_COUNT_MASKED", False, 40), ("VEC_COUNT_MASKED", True, 31)])
def test_cli_vectors_multi_pass(eng, tmp_path, mode, rc, k):
    import kmer_oracle as ko

    from kman_b200 import fasta

    recs = vec_records(90_000, 8)
    fa = tmp_path / "in.fa"
    fa.write_bytes(b"".join(b">%s\n%s\n" % (n.encode(), s.encode()) for n, s in recs))
    d = eng.upload(fasta.from_records(recs), alphabet="IUPAC")
    budget = forced_budget(eng, d, k, rc, passes=4, slack=1 << 16)  # (the CLI's input buffer holds the FASTA's bytes)
    assert eng.plan_passes(d, k, rc, "vec", budget_bytes=budget).n_passes >= 2
    env = dict(os.environ, PYTHONPATH=ROOT, KMG_ALPHABET="IUPAC", KMG_DEVICE_BUDGET=str(budget))
    subprocess.run([sys.executable, "-m", "kman_b200.scripts.kmer", "count", "-m", mode, *(["-r"] if rc else []), str(fa),
                    str(tmp_path / "vec.txt"), str(k)], check=True, env=env, cwd=str(tmp_path), stdout=subprocess.DEVNULL)
    want = ko.vec_count_np(recs, k, rc, mode == "VEC_COUNT_MASKED", "IUPAC")
    assert sorted(os.listdir(tmp_path / "vec")) == sorted(want)
    for f, text in want.items():
        with gzip.open(tmp_path / "vec" / f, "rb") as fh:  # valid gzip, one stream
            assert fh.read() == text, f


def test_vec_errors_and_directory(eng, dev_vec, tmp_path, capsys):
    from kman_b200 import fasta
    from kman_b200.engine import pass_bytes

    d = dev_vec
    extra = eng._resident_bytes(d) + 8 * (d.n_bases + 1)
    with pytest.raises(ValueError, match="k >= 12"):
        eng.write_vectors(d, 11, False, False, str(tmp_path / "a"), budget_bytes=extra + 1000)
    with pytest.raises(ValueError, match="k >= 12"):
        eng.abundance(d, 11, False, False, budget_bytes=extra + 1000)
    k, rc = 31, True
    narrow, wide = eng.part_counts(d, k, rc, 256)
    _, text_bytes = eng._text_plan(d, k, "vec", None)
    biggest = max(pass_bytes(k, "vec", int(a), int(b), d.payload_bytes, text_bytes, d.n_bases - k + 1)
                  for a, b in zip(narrow, wide))
    with pytest.raises(ValueError, match="needs"):
        eng.write_vectors(d, k, rc, False, str(tmp_path / "b"), budget_bytes=biggest - 1 + extra)
    # two records of one name
    dup = eng.upload(fasta.from_records([("x one", "ACGT" * 10), ("x two", "TTGCA" * 9)]), alphabet="ACGT")
    with pytest.raises(AssertionError):
        eng.write_vectors(dup, 12, False, False, str(tmp_path / "c"))
    # the output directory is an existing file
    (tmp_path / "taken").write_bytes(b"")
    with pytest.raises(AssertionError):
        eng.write_vectors(d, 31, False, False, str(tmp_path / "taken.txt"))
    # nothing to write: the directory exists and is empty
    none = eng.upload(fasta.from_records([("r", "ACGTNACGT"), ("s", "")]), alphabet="ACGT")
    capsys.readouterr()
    plan = eng.write_vectors(none, 31, True, False, str(tmp_path / "empty.txt"))
    assert plan.n_passes == 1 and (tmp_path / "empty").is_dir() and not os.listdir(tmp_path / "empty")
    assert capsys.readouterr().out == 'Writing output in "%s"\n' % (tmp_path / "empty")
