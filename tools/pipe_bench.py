#!/usr/bin/env python
"""Device timings of the fused device path (kmg_extract_sort_count / kmg_extract_sort_uniq) next to
the stage path (kmg_extract -> kmg_sort_count) on one GPU, with the per-kernel event timings the
library keeps under kmg_set_option("time_passes", 1); a development tool.
usage: python tools/pipe_bench.py [--n 100000000] [--k 31] [--rc]"""
import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from kman_b200 import fasta  # noqa: E402
from kman_b200.engine import get_engine  # noqa: E402


def timed(fn, reps=7, warm=2):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), float(np.min(ts))


def kernel_split(lib, fn, reps=5):
    lib.kmg_set_option(b"time_passes", 1)
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    out = []
    for nm in ("prepass", "scatter", "sort_pass", "local_sort"):
        ns, c = lib.kmg_get_stat((nm + "_ns").encode()), lib.kmg_get_stat((nm + "_count").encode())
        if c:
            out.append(f"{nm} {ns / 1e6 / reps:.3f} ms ({c // reps} launches)")
    lib.kmg_set_option(b"time_passes", 0)
    return ", ".join(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=100_000_000)
    ap.add_argument("--k", type=int, default=31)
    ap.add_argument("--rc", action="store_true")
    args = ap.parse_args()
    eng = get_engine(0)
    lib = eng.lib
    rng = np.random.default_rng(1234)
    bases = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, size=args.n, dtype=np.uint8)]
    flat = fasta.FlatInput(np.concatenate([bases, np.array([10], np.uint8)]), np.array([0, args.n + 1], np.uint64), ["chr1"], ["chr1"])
    d = eng.upload(flat, alphabet="ACGT", with_names=False)
    k, rc = args.k, args.rc
    N = (args.n - k + 1) * (2 if rc else 1)

    def stage_count():
        return eng.sort_count(eng.extract(d, k, rc, val_bytes=0, reuse="b_", want_hist=True), reuse="b_")

    def pipe_count():
        return eng.count_narrow(d, k, rc, reuse="b_")[0]

    def stage_uniq():
        return eng.sort_uniq(eng.extract(d, k, rc, val_bytes=4, reuse="u_", want_hist=True))

    def pipe_uniq():
        return eng.uniq_narrow(d, k, rc, reuse="u_", val_bytes=4)[0]

    for name, fn in (("count, stage calls ", stage_count), ("count, fused path  ", pipe_count),
                     ("uniq,  stage calls ", stage_uniq), ("uniq,  fused path  ", pipe_uniq)):
        med, mn = timed(fn)
        r = fn()
        print(f"{name}: {med:8.3f} ms (min {mn:.3f})  {N / med / 1e6:8.2f} G k-mers/s  rows {r.n}  passes "
              f"{lib.kmg_get_stat(b'sort_passes')} path {lib.kmg_get_stat(b'hybrid_path')}")
        print("    kernels per call:", kernel_split(lib, fn))
    for pb in (16, 24):
        lib.kmg_set_option(b"hybrid_pb", pb)
        med, mn = timed(pipe_count)
        print(f"count, fused path, pb {pb}: {med:8.3f} ms (min {mn:.3f})  {N / med / 1e6:8.2f} G k-mers/s")
        print("    kernels per call:", kernel_split(lib, pipe_count))
    lib.kmg_set_option(b"hybrid_pb", 0)


if __name__ == "__main__":
    main()
