#!/usr/bin/env python
"""Device timings (CUDA events) of the extraction entry points that size and feed the multi-GPU range
partition, on one GPU: kmg_extract_dest_counts (its 4-mer pre-pass over the bases plus the
per-destination sums), kmg_extract_scatter_checked with every destination buffer on this GPU, and the
stage path's kmg_extract with its digit histograms.  Prints a checksum of the results so that two
builds can be compared; a development tool.
usage: python tools/extract_bench.py [--n 387500030] [--k 31] [--parts 8]"""
import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from kman_b200 import _lib, fasta  # noqa: E402
from kman_b200.engine import get_engine  # noqa: E402
from pipe_bench import timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=387_500_030, help="bases (default: 387.5 M windows at k=31)")
    ap.add_argument("--k", type=int, default=31)
    ap.add_argument("--parts", type=int, default=8)
    args = ap.parse_args()
    eng = get_engine(0)
    lib = eng.lib
    rng = np.random.default_rng(1234)
    bases = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, size=args.n, dtype=np.uint8)]
    flat = fasta.FlatInput(np.concatenate([bases, np.array([10], np.uint8)]), np.array([0, args.n + 1], np.uint64), ["chr1"], ["chr1"])
    d = eng.upload(flat, alphabet="ACGT", with_names=False)
    k, G = args.k, args.parts
    n_win = d.n_bases - k + 1
    kb = 8 if k <= 32 else 16
    st = eng._stream()
    print(f"n_windows {n_win}  k {k}  n_parts {G}")
    ws_bytes = lib.kmg_dest_counts_workspace_bytes()
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=eng.device)
    counts = torch.zeros(G + 1, dtype=torch.int64, device=eng.device)
    for rc in (0, 1):
        def dest_counts():
            _lib.check(lib.kmg_extract_dest_counts(d.bases.data_ptr(), d.n_bases, 0, n_win, k, rc, d.lut.data_ptr(), G,
                                                   counts.data_ptr(), ws.data_ptr(), ws_bytes, st))

        med, mn = timed(dest_counts, reps=21, warm=3)
        c = counts.cpu().numpy()
        print(f"dest_counts rc={rc}: {med:.4f} ms (min {mn:.4f})  counts {list(c)}")

        cap = int(c[:G].max())
        keys = torch.empty((G, cap * kb), dtype=torch.uint8, device=eng.device)
        vals = torch.empty((G, cap * 8), dtype=torch.uint8, device=eng.device)
        kptr = torch.tensor([keys[g].data_ptr() for g in range(G)], dtype=torch.int64, device=eng.device)
        vptr = torch.tensor([vals[g].data_ptr() for g in range(G)], dtype=torch.int64, device=eng.device)
        cursors = torch.zeros(G, dtype=torch.int64, device=eng.device)
        status = torch.zeros(2, dtype=torch.int32, device=eng.device)

        def scatter():
            cursors.zero_()
            _lib.check(lib.kmg_extract_scatter_checked(d.bases.data_ptr(), d.n_bases, 0, n_win, k, rc, d.lut.data_ptr(), G,
                                                       kptr.data_ptr(), vptr.data_ptr(), kb, 8, 0, cursors.data_ptr(), cap,
                                                       status.data_ptr(), st))

        med, mn = timed(scatter, reps=11, warm=2)
        torch.cuda.synchronize()
        # keys of a destination arrive in no fixed order: sum them (mod 2^64) as the checksum
        ks = [int(keys[g, : int(c[g]) * kb].view(torch.int64).sum()) & (2**64 - 1) for g in range(G)]
        print(f"scatter_checked rc={rc}: {med:.4f} ms (min {mn:.4f})  cursors {list(cursors.cpu().numpy())} "
              f"status {list(status.cpu().numpy())} key sums {ks}")
        del keys, vals
        torch.cuda.empty_cache()

        def stage_extract():
            return eng.extract(d, k, bool(rc), val_bytes=0, reuse="b_", want_hist=True)

        med, mn = timed(stage_extract, reps=11, warm=2)
        a = stage_extract()
        print(f"stage kmg_extract rc={rc}: {med:.4f} ms (min {mn:.4f})  keys {a.n}  key sum "
              f"{int(a.keys[: a.n * kb].view(torch.int64).sum()) & (2**64 - 1)}")
        eng._scratch.clear()
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
