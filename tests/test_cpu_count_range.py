"""`kmer count --min-count / --max-count` pieces that need no GPU: option parsing and rejection, the range
helper and the pass plan of a filtered count."""
import pytest

M = 2**32 - 1


def _cli(*argv):
    from click.testing import CliRunner

    from kman_b200.scripts import kmer

    return CliRunner().invoke(kmer.main, list(argv))


def test_count_range_helper():
    from kman_b200.engine import count_range

    assert count_range() is None and count_range(1, M) is None and count_range(1, None) is None
    assert count_range(2) == (2, M) and count_range(1, 1) == (1, 1) and count_range(1, M - 1) == (1, M - 1)
    for lo, hi in ((0, None), (0, 5), (3, 2), (1, M + 1), (M + 1, None), (-1, 4)):
        with pytest.raises(AssertionError):
            count_range(lo, hi)


def test_options_are_long_only():
    r = _cli("count", "--help")
    assert r.exit_code == 0 and "--min-count" in r.output and "--max-count" in r.output


@pytest.mark.parametrize("opts", [["--min-count", "0"], ["--min-count", "5", "--max-count", "4"],
                                  ["--max-count", "0"], ["--max-count", str(M + 1)], ["--min-count", "-3"]])
def test_bad_ranges_are_rejected_before_any_work(tmp_path, opts):
    inp, out = tmp_path / "in.fa", tmp_path / "out"
    inp.write_bytes(b">r\nACGTACGT\n")
    r = _cli("count", str(inp), str(out), "4", *opts)
    assert isinstance(r.exception, AssertionError), (r.output, r.exception)
    assert not out.exists()


@pytest.mark.parametrize("mode", ["VEC_COUNT", "VEC_COUNT_MASKED"])
@pytest.mark.parametrize("opts", [["--min-count", "2"], ["--max-count", "3"]])
def test_vector_modes_reject_a_range(tmp_path, mode, opts):
    inp, out = tmp_path / "in.fa", tmp_path / "out"
    inp.write_bytes(b">r\nACGTACGT\n")
    r = _cli("count", "-m", mode, str(inp), str(out), "4", *opts)
    assert isinstance(r.exception, AssertionError), (r.output, r.exception)
    assert not out.exists()


def test_joiner_carries_the_range():
    from kman_b200.join import KJoiner, KJoinerThreading

    j = KJoinerThreading(KJoiner.MODE.SEQ_COUNT)
    assert j.count_range == (1, None)
    j.count_range = (2, 7)
    assert j.count_range == (2, 7)
    with pytest.raises(AssertionError):
        j.count_range = (0, 7)
    j = KJoinerThreading(KJoiner.MODE.UNIQUE)
    j.count_range = (1, None)  # the full range is no restriction
    with pytest.raises(AssertionError):
        j.count_range = (2, None)


def test_host_batches_skip_lines_outside_the_range(tmp_path):
    """The reference protocol (host batches): the lines of the unfiltered join whose count is in range."""
    from kman_b200.batch import Batch
    from kman_b200.join import KJoiner, KJoinerThreading
    from kman_b200.seq import KMer

    a, b = Batch(KMer, str(tmp_path), 4), Batch(KMer, str(tmp_path), 4)
    a.add_all([KMer("c", 0, 4, "ACGT"), KMer("c", 1, 5, "CGTA"), KMer("c", 2, 6, "TTTT"), KMer("c", 3, 7, "ACGT")])
    b.add_all([KMer("d", 0, 4, "ACGT"), KMer("d", 1, 5, "TTTT")])
    a.write(doSort=True)
    b.write(doSort=True)
    outs = {}
    for rng in ((1, None), (2, None), (1, 1), (3, 3), (4, None)):
        j = KJoinerThreading(KJoiner.MODE.SEQ_COUNT)
        j.count_range = rng
        out = tmp_path / f"out_{rng[0]}_{rng[1]}.tsv"
        j.join([a, b], str(out))
        outs[rng] = out.read_text()
    assert outs[(1, None)] == "ACGT\t3\nCGTA\t1\nTTTT\t2\n"
    assert outs[(2, None)] == "ACGT\t3\nTTTT\t2\n"
    assert outs[(1, 1)] == "CGTA\t1\n"
    assert outs[(3, 3)] == "ACGT\t3\n"
    assert outs[(4, None)] == ""


def test_filtered_count_takes_the_count_plan():
    """write_count with a range plans with mode "count": the filtered tables and workspaces are never larger."""
    import io

    from kman_b200.engine import Engine

    calls = []

    class Stub:
        def _write_passes(self, d, k, rc, fh, mode, budget_bytes, chunk_rows, rng=None):
            calls.append((mode, budget_bytes, chunk_rows, rng))

    Engine.write_count(Stub(), None, 31, False, io.BytesIO(), 123, 45, min_count=2)
    Engine.write_count(Stub(), None, 31, False, io.BytesIO(), 123, 45, min_count=1, max_count=9)
    Engine.write_count(Stub(), None, 31, False, io.BytesIO(), 123, 45)
    assert calls == [("count", 123, 45, (2, M)), ("count", 123, 45, (1, 9)), ("count", 123, 45, None)]
