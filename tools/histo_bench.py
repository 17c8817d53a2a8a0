#!/usr/bin/env python
"""`kmer histo` against `kmer count` on one GPU, the two sides alternated in one process:
  1. kmg_extract_sort_histo against kmg_extract_sort_count (Engine.histo_narrow / count_narrow with reused
     buffers) on config 2 (synth_configs.cfg2: 100 Mbp random ACGT, one record, k = 31), CUDA events around
     each call (both calls synchronise the host internally);
  2. the same pair on tools/genome_like_bench.py's input (4 records, interspersed repeats with poly-A tails,
     microsatellites, soft-masking, N gaps), where the fused count falls back to sort + run-length stage;
  3. with --cfg3 N: Engine.write_histogram against Engine.write_count (the text goes to a sink that only
     counts bytes) on synth_configs.cfg3(N) already on the device, wall time.
The card's name, power limit and SM clock are read in the same run.  The histogram of every pair is checked
against the spectrum of the count table of the same call.
usage: python tools/histo_bench.py [--n 100000000] [--k 31] [--reps 10] [--cfg3 3100000000]"""
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

BINS = 4096


class NullSink:
    """Binary file object that keeps nothing but the byte count."""

    def __init__(self):
        self.bytes = 0

    def write(self, b) -> int:
        n = memoryview(b).nbytes
        self.bytes += n
        return n


def spectrum_of_counts(counts: np.ndarray):
    m, c = np.unique(counts, return_counts=True)
    return m.astype(np.uint64), c.astype(np.uint64)


def read_histo(acc: torch.Tensor):
    raw = acc.cpu().numpy()
    bins = raw[: 8 * (BINS + 1)].view(np.uint64)
    big = raw[8 * (BINS + 1):].view(np.uint32)[: int(bins[BINS])]
    mult = np.flatnonzero(bins[:BINS]).astype(np.uint64)
    cnt = bins[:BINS][mult.astype(np.int64)]
    if big.size:
        bm, bc = np.unique(big, return_counts=True)
        mult, cnt = np.concatenate([mult, bm.astype(np.uint64)]), np.concatenate([cnt, bc.astype(np.uint64)])
    return mult, cnt


def pair(eng, d, k, reps, label):
    """histo_narrow vs count_narrow on one input, alternated; median ms of each and the two stats."""
    n_keys, _ = eng.count_windows(d, k, False)
    acc = torch.zeros(8 * (BINS + 1) + 4 * (n_keys // BINS + 1), dtype=torch.uint8, device=eng.device)
    out = (acc.data_ptr(), acc.data_ptr() + 8 * (BINS + 1), acc.data_ptr() + 8 * BINS)
    stats = {}

    def histo():
        acc.zero_()
        eng.histo_narrow(d, k, False, out, reuse="hb_")
        stats["histo"] = (eng.lib.kmg_get_stat(b"hybrid_path"), eng.lib.kmg_get_stat(b"hybrid_irregular"))

    def count():
        tab, _ = eng.count_narrow(d, k, False, reuse="hb_")
        stats["count"] = (eng.lib.kmg_get_stat(b"hybrid_path"), eng.lib.kmg_get_stat(b"hybrid_irregular"))
        return tab

    tab = count()
    want = spectrum_of_counts(tab.counts_host())
    del tab
    histo()
    same = all(np.array_equal(a, b) for a, b in zip(read_histo(acc), want))
    for _ in range(2):  # warm-up of both sides
        histo()
        count()
    ms = {"histo": [], "count": []}
    for _ in range(reps):
        for name, fn in (("histo", histo), ("count", count)):
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            fn()
            t1.record()
            t1.synchronize()
            ms[name].append(t0.elapsed_time(t1))
    med = {k_: float(np.median(v)) for k_, v in ms.items()}
    print(json.dumps({
        "input": label, "k": k, "keys": n_keys, "reps": reps, "same_spectrum": same,
        "kmg_extract_sort_histo_ms": round(med["histo"], 3), "kmg_extract_sort_count_ms": round(med["count"], 3),
        "histo_ms_all": [round(x, 3) for x in ms["histo"]], "count_ms_all": [round(x, 3) for x in ms["count"]],
        "histo_hybrid_path_irregular": stats["histo"], "count_hybrid_path_irregular": stats["count"],
        "histo_g_kmers_per_s": round(n_keys / med["histo"] / 1e6, 2), "count_g_kmers_per_s": round(n_keys / med["count"] / 1e6, 2),
    }), flush=True)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=100_000_000)
    ap.add_argument("--k", type=int, default=31)
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
    pair(eng, d, args.k, args.reps, f"cfg2 {args.n} bp")
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
    pair(eng, d, args.k, args.reps, f"genome_like {args.n} bp")
    del d, flat, parts
    eng._scratch.clear()
    torch.cuda.empty_cache()

    if args.cfg3:
        t0 = time.perf_counter()
        d = eng.upload(fasta.from_records(sc.cfg3(args.cfg3, 24)), alphabet="ACGT", with_names=False)
        print(f"# cfg3 {args.cfg3} bp uploaded in {time.perf_counter() - t0:.1f} s", flush=True)
        res = {}
        for name in ("histo", "count", "histo"):
            sink = NullSink()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            if name == "histo":
                plan = eng.write_histogram(d, args.k, False, sink)
            else:
                plan = eng.write_count(d, args.k, False, sink)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            res.setdefault(name, []).append(round(wall, 2))
            print(json.dumps({"cmd": f"Engine.write_{'histogram' if name == 'histo' else 'count'} k={args.k}", "bases": d.n_bases,
                              "passes": plan.n_passes, "pass_ms": [round(x, 1) for x in plan.pass_ms], "wall_s": round(wall, 2),
                              "bytes_written": sink.bytes, "hybrid_path_last_call": eng.lib.kmg_get_stat(b"hybrid_path")}),
                  flush=True)
            eng._scratch.clear()
            torch.cuda.empty_cache()
        print(json.dumps({"cfg3_wall_s": res}), flush=True)


if __name__ == "__main__":
    main()
