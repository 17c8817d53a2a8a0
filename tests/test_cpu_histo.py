"""`kmer histo` pieces that need no GPU: the command's registration and argument checks, the pass model."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_histo_bins_match_the_header():
    from kman_b200 import _lib

    hdr = open(os.path.join(ROOT, "include", "kmg.h")).read()
    assert int(re.search(r"#define KMG_HISTO_BINS (\d+)", hdr).group(1)) == _lib.KMG_HISTO_BINS


def test_histo_command_is_registered(tmp_path):
    from click.testing import CliRunner

    from kman_b200.scripts import kmer

    r = CliRunner().invoke(kmer.main, ["--help"])
    assert r.exit_code == 0 and "histo" in r.output
    r = CliRunner().invoke(kmer.main, ["histo", "--help"])
    assert r.exit_code == 0 and "INPUT OUTPUT K" in r.output
    inp = tmp_path / "in.fa"
    inp.write_bytes(b">r\nACGTACGT\n")
    r = CliRunner().invoke(kmer.main, ["histo", str(inp), str(tmp_path / "out"), "1"])  # before any device work
    assert isinstance(r.exception, AssertionError)
    assert not (tmp_path / "out").exists()


def test_histo_pass_bytes_model():
    from kman_b200 import _lib
    from kman_b200.engine import pass_bytes

    lib = _lib.load()
    n, m, n_win = 50_000_000, 2_000_000, 100_000_000
    for k in (31, 45):
        kb, kw = (8, 16) if k <= 32 else (16, 32)
        h = pass_bytes(k, "histo", n, m, 4, 0, n_win)
        assert h >= 2 * n * kb + lib.kmg_sort_histo_workspace_bytes(n, kb, 2 * k)
        assert h >= 2 * m * kw
        assert h < pass_bytes(k, "count", n, m, 4, 0, n_win)  # no counts, no merge ranks
        assert pass_bytes(k, "histo", 2 * n, m, 4, 0, n_win) > h and pass_bytes(k, "histo", n, 40 * m, 4, 0, n_win) > h


@pytest.mark.parametrize("n", [0, 1, 4095, 4096, 1 << 20, 100_000_000])
def test_histo_workspaces_cover_the_sort(n):
    from kman_b200 import _lib

    lib = _lib.load()
    for kb, end_bit in ((8, 62), (16, 90)):
        assert lib.kmg_sort_histo_workspace_bytes(n, kb, end_bit) >= lib.kmg_radix_sort_workspace_bytes(n, kb, 0, 0, end_bit)
    assert lib.kmg_pipeline_histo_workspace_bytes(n, 31, 1) > 0
    assert lib.kmg_pipeline_histo_workspace_bytes(n, 65, 0) == 0
