#!/usr/bin/env python
"""Per-stage device timings (CUDA events) of the hot path on one GPU; a development tool.
usage: python tools/stage_bench.py [--n 100000000] [--k 31] [--local-tiles 4096,7936] [--yardstick]"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from kman_b200 import fasta  # noqa: E402
from kman_b200.engine import get_engine  # noqa: E402


def timed(fn, reps=5, warm=2, flush=None):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(reps):
        if flush is not None:
            flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), float(np.min(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=100_000_000)
    ap.add_argument("--k", type=int, default=31)
    ap.add_argument("--vb", type=int, default=0)
    ap.add_argument("--yardstick", action="store_true")
    ap.add_argument("--local-tiles", default="")
    args = ap.parse_args()
    eng = get_engine(0)
    rng = np.random.default_rng(1234)
    bases = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, size=args.n, dtype=np.uint8)]
    flat = fasta.FlatInput(np.concatenate([bases, np.array([10], np.uint8)]), np.array([0, args.n + 1], np.uint64), ["chr1"], ["chr1"])
    d = eng.upload(flat, alphabet="ACGT", with_names=False)
    k = args.k
    N = args.n - k + 1
    peak = 6552.6
    try:
        peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        pass
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    res = {}
    med, mn = timed(lambda: eng.extract(d, k, False, val_bytes=args.vb, reuse="b_", want_hist=True), flush=flush)
    W = 8 if k <= 32 else 16
    print(f"extract        : {med:8.3f} ms (min {mn:.3f})  {N/med/1e6:8.2f} G kmers/s   alg {(1+W+args.vb)*N/med/1e6:8.1f} GB/s")
    res["extract_ms"] = med
    P8 = (2 * k + 7) // 8

    def run():
        a = eng.extract(d, k, False, val_bytes=args.vb, reuse="b_", want_hist=True)
        return eng.sort(a)

    med_all, _ = timed(run, flush=flush)
    srt = med_all - res["extract_ms"]
    alg = N * (W * (2 * P8 + 1) + 2 * P8 * args.vb)
    print(f"sort           : {srt:8.3f} ms  {N/srt/1e6:8.2f} G keys/s  model {alg/srt/1e6:8.1f} GB/s = {alg/srt/1e6/peak:5.3f} of measured peak")
    res["sort_ms"] = srt
    for hy, pb in ((0, 0), (1, 16), (1, 24), (1, 0)):
        eng.lib.kmg_set_option(b"hybrid", hy)
        eng.lib.kmg_set_option(b"hybrid_pb", pb)
        med_all, _ = timed(run, flush=flush)
        srt = med_all - res["extract_ms"]
        print(f"hybrid {hy} pb {pb:2d}: sort {srt:8.3f} ms  {N/srt/1e6:8.2f} G keys/s  passes {eng.lib.kmg_get_stat(b'sort_passes')} irregular {eng.lib.kmg_get_stat(b'hybrid_irregular')}")
        res[f"sort_hy{hy}_pb{pb}_ms"] = srt
    eng.lib.kmg_set_option(b"hybrid_pb", 0)

    def full():
        return eng.sort_count(eng.extract(d, k, False, val_bytes=0, reuse="b_", want_hist=True), reuse="b_")

    for pbv in (0, 24):
        eng.lib.kmg_set_option(b"hybrid_pb", pbv)
        for lt in [int(x) for x in args.local_tiles.split(",") if x]:
            eng.lib.kmg_set_option(b"local_tile", lt)
            med_full, mn_full = timed(full, flush=flush)
            print(f"pb {pbv:2d} local_tile {lt}: full count {med_full:8.3f} ms  {N/med_full/1e6:8.2f} G kmers/s")
    eng.lib.kmg_set_option(b"hybrid_pb", 0)
    eng.lib.kmg_set_option(b"local_tile", 7936)
    eng.lib.kmg_set_option(b"count_fused", 0)
    med_full, mn_full = timed(full, flush=flush)
    print(f"full count (sort, then rle): {med_full:8.3f} ms (min {mn_full:.3f})  {N/med_full/1e6:8.2f} G kmers/s")
    eng.lib.kmg_set_option(b"count_fused", 1)
    med_full, mn_full = timed(full, flush=flush)
    print(f"full count     : {med_full:8.3f} ms (min {mn_full:.3f})  {N/med_full/1e6:8.2f} G kmers/s")
    res["full_ms"] = med_full

    def full_uniq():
        return eng.sort_uniq(eng.extract(d, k, False, val_bytes=4, reuse="u_", want_hist=True))

    eng.lib.kmg_set_option(b"hybrid", 0)
    med_u, mn_u = timed(full_uniq, flush=flush)
    print(f"full uniq (u32 payload, plain LSD passes): {med_u:8.3f} ms (min {mn_u:.3f})  {N/med_u/1e6:8.2f} G kmers/s")
    eng.lib.kmg_set_option(b"hybrid", 1)
    med_u, mn_u = timed(full_uniq, flush=flush)
    print(f"full uniq (u32 payload): {med_u:8.3f} ms (min {mn_u:.3f})  {N/med_u/1e6:8.2f} G kmers/s  passes {eng.lib.kmg_get_stat(b'sort_passes')} path {eng.lib.kmg_get_stat(b'hybrid_path')}")
    res["full_uniq_ms"] = med_u
    if args.yardstick:
        a = eng.extract(d, k, False, val_bytes=0, reuse="b_", want_hist=True)
        keys = a.keys[: a.n * 8].view(torch.int64)
        med, mn = timed(lambda: torch.sort(keys), flush=flush)
        print(f"torch.sort (library yardstick): {med:8.3f} ms  {N/med/1e6:8.2f} G keys/s")
        src = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")
        dst = torch.empty_like(src)
        med, mn = timed(lambda: dst.copy_(src))
        print(f"copy 1 GiB     : {med:8.3f} ms  {2*(1<<30)/med/1e6:8.1f} GB/s")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
