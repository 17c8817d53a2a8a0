#!/usr/bin/env python
"""`kmer count --min-count / --max-count` against `kmer count` on one GPU, the sides alternated in one process:
  1. kmg_extract_sort_count against kmg_extract_sort_count_range at (2, 2^32-1), (1, 1) and (1, 2^32-2)
     (Engine.count_narrow with reused buffers), CUDA events around each call (every call synchronises the host
     internally), on config 2 (synth_configs.cfg2: 100 Mbp random ACGT, one record) at k = 31 and k = 63, and on
     tools/genome_like_bench.py's input (4 records with interspersed repeats, poly-A tails, microsatellites,
     soft-masking, N gaps), where the fused count falls back to sort + run-length stage (+ kmg_filter_counts);
  2. with --cfg3 N: Engine.write_count with and without min_count=2 on synth_configs.cfg3(N) already on the
     device (the text goes to a sink that only counts bytes), wall time.
The card's name, power limit and SM clock are read in the same run.  Every filtered table is checked against
the count table of the same input with the same mask (keys and counts).
usage: python tools/count_range_bench.py [--n 100000000] [--reps 10] [--cfg3 3100000000]"""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

M = 2**32 - 1
SIDES = (("count", 1, M), ("range_2_inf", 2, M), ("range_1_1", 1, 1), ("range_1_max-1", 1, M - 1))


class NullSink:
    """Binary file object that keeps nothing but the byte count."""

    def __init__(self):
        self.bytes = 0

    def write(self, b) -> int:
        n = memoryview(b).nbytes
        self.bytes += n
        return n


def table(t):
    keys = t.keys[: t.n * t.key_bytes].cpu().numpy().view(np.uint64).reshape(t.n, t.key_bytes // 8)
    return keys, t.counts_host()


def compare(eng, d, k, reps, label):
    """count_narrow at every side of SIDES on one input, alternated; median ms of each, output checks."""
    n_keys, _ = eng.count_windows(d, k, False)
    stats = {}

    def run(lo, hi):
        tab, _ = eng.count_narrow(d, k, False, reuse="rb_", min_count=lo, max_count=None if hi == M else hi)
        return tab

    want_k, want_c = table(run(1, M))
    same = {}
    for name, lo, hi in SIDES:
        gk, gc = table(run(lo, hi))
        mask = (want_c >= lo) & (want_c <= hi)
        same[name] = bool(np.array_equal(gk, want_k[mask]) and np.array_equal(gc, want_c[mask]))
        stats[name] = (eng.lib.kmg_get_stat(b"hybrid_path"), int(mask.sum()))
    del want_k, want_c
    for _ in range(2):  # warm-up of every side
        for _, lo, hi in SIDES:
            run(lo, hi)
    ms = {name: [] for name, _, _ in SIDES}
    for _ in range(reps):
        for name, lo, hi in SIDES:
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            run(lo, hi)
            t1.record()
            t1.synchronize()
            ms[name].append(t0.elapsed_time(t1))
    print(json.dumps({
        "input": label, "k": k, "keys": n_keys, "reps": reps, "same_as_filtered_count": same,
        "median_ms": {n_: round(float(np.median(v)), 3) for n_, v in ms.items()},
        "ms_all": {n_: [round(x, 3) for x in v] for n_, v in ms.items()},
        "hybrid_path_rows": stats,
    }), flush=True)
    eng._scratch.clear()
    torch.cuda.empty_cache()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=100_000_000)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--cfg3", type=int, default=0, help="bases of synth_configs.cfg3 (0: skip the genome-size run)")
    args = ap.parse_args()

    import synth_configs as sc

    from kman_b200 import fasta
    from kman_b200.engine import get_engine

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print(f"# {gpu}", flush=True)
    eng = get_engine(0)

    d = eng.upload(fasta.from_records(sc.cfg2(args.n)), alphabet="ACGT", with_names=False)
    compare(eng, d, 31, args.reps, f"cfg2 {args.n} bp")
    compare(eng, d, 63, args.reps, f"cfg2 {args.n} bp")
    del d

    spec = importlib.util.spec_from_file_location("genome_like_bench", os.path.join(ROOT, "tools", "genome_like_bench.py"))
    gl = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gl)
    per = args.n // 4
    parts, starts, pos = [], [0], 0
    for r in range(4):
        parts += [gl.genome_like(per, seed=7 + r), np.array([10], np.uint8)]
        pos += per + 1
        starts.append(pos)
    names = ["chr%d" % i for i in range(4)]
    flat = fasta.FlatInput(np.concatenate(parts), np.array(starts, np.uint64), names, names)
    d = eng.upload(flat, alphabet="ACGT", with_names=False)
    compare(eng, d, 31, args.reps, f"genome_like {args.n} bp")
    del d, flat, parts

    if args.cfg3:
        t0 = time.perf_counter()
        d = eng.upload(fasta.from_records(sc.cfg3(args.cfg3, 24)), alphabet="ACGT", with_names=False)
        print(f"# cfg3 {args.cfg3} bp uploaded in {time.perf_counter() - t0:.1f} s", flush=True)
        res = {}
        for name, lo in (("count", 1), ("min_count_2", 2), ("count", 1), ("min_count_2", 2)):
            sink = NullSink()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            plan = eng.write_count(d, 31, False, sink, min_count=lo)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            res.setdefault(name, []).append(round(wall, 2))
            print(json.dumps({"cmd": f"Engine.write_count k=31 min_count={lo}", "bases": d.n_bases, "passes": plan.n_passes,
                              "pass_ms": [round(x, 1) for x in plan.pass_ms], "wall_s": round(wall, 2),
                              "bytes_written": sink.bytes, "hybrid_path_last_call": eng.lib.kmg_get_stat(b"hybrid_path")}),
                  flush=True)
            eng._scratch.clear()
            torch.cuda.empty_cache()
        print(json.dumps({"cfg3_wall_s": res}), flush=True)


if __name__ == "__main__":
    main()
