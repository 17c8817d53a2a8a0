"""bench.py on the device: --steps sets the number of timed steps, and --dump-outputs writes the same
sample of the last step's (k-mer, count) table on every run of the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "0",
                        "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-3000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, p.stdout
    return json.loads(lines[0])


def test_bench_dump_outputs_is_reproducible(tmp_path):
    runs = [_bench(tmp_path / "a"), _bench(tmp_path / "b")]
    assert all(d["steps"] == 2 and d["verify"]["ok"] for d in runs)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b")) == ["counts.npy", "keys_hi.npy", "keys_lo.npy", "n_rows.npy", "rows.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in names) <= 64 << 20
    a = {f[:-4]: np.load(tmp_path / "a" / f) for f in names}
    for f in names:
        assert np.array_equal(a[f[:-4]], np.load(tmp_path / "b" / f)), f
    assert a["n_rows"].tolist() == [runs[0]["verify"]["distinct"]]
    keys = a["keys_hi"].astype(np.uint64) << np.uint64(31) | a["keys_lo"].astype(np.uint64)
    assert keys.size == a["rows"].size > 0 and (np.diff(keys.astype(np.int64)) > 0).all() and keys.max() < 1 << 62
    assert (a["counts"] >= 1).all()
