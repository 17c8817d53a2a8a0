#!/usr/bin/env python
"""Genome-scale `kmer count -m VEC_COUNT / VEC_COUNT_MASKED` on one GPU through Engine.write_vectors: the real
REF___STRAND.gz files are written to a scratch directory, read back and removed at the end.

Reports per command: passes and their planned bytes, torch.cuda.max_memory_allocated, time per pass (CUDA
events), the text stage's time (device formatting and copies, waits for a free chunk buffer included), the wall
time of write_vectors and the host's peak RSS, with the card's name and power limit.

For VEC_COUNT it checks two invariants without an oracle, on the decompressed files: the number of non-zero
entries equals the number of k-mers, and the sum of all entries equals the sum of count^2 over the count table
of the same input (Engine.pass_tables(..., "count", plan)): every k-mer's position holds its group's size.

`--shared` copies stretches between neighbouring records (1/50 of each record from the one before it), so the
masked vectors are not empty.

usage: python tools/vec_bench.py [--n 3100000000] [--runs vec-r:31,vec:40] [--shared] [--budget BYTES] [--dir DIR]"""
import argparse
import gzip
import json
import os
import resource
import shutil
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def peak_rss_gb() -> float:
    return resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 1e6


def file_stats(path: str):
    """(non-zero entries, sum of entries) of one decompressed vector file ("# k=K" line, then one count per line)."""
    nonzero = total = 0
    rest = b""
    with gzip.open(path, "rb") as fh:
        fh.readline()
        while True:
            block = fh.read(64 << 20)
            if not block:
                break
            a = np.frombuffer(rest + block, np.uint8)
            nl = np.flatnonzero(a == 10)
            rest = a[nl[-1] + 1:].tobytes() if nl.size else a.tobytes()
            if not nl.size:
                continue
            starts = np.concatenate(([0], nl[:-1] + 1))
            ndig = nl - starts
            val = np.zeros(nl.size, np.int64)
            scale = 1
            for j in range(int(ndig.max())):
                has = ndig > j
                val[has] += (a[nl[has] - 1 - j].astype(np.int64) - 48) * scale
                scale *= 10
            nonzero += int(np.count_nonzero(val))
            total += int(val.sum())
    assert not rest, f"{path}: unterminated last line"
    return nonzero, total


def count_squares(eng, d, k: int, rc: bool):
    """(k-mers, sum of count^2) from the count table of the input, pass by pass."""
    plan = eng.plan_passes(d, k, rc, "count")
    n = sq = 0
    for tabs in eng.pass_tables(d, k, rc, "count", plan):
        for t in tabs:
            c = t.counts[: t.n * 4].view(torch.int32).to(torch.int64) & 0xFFFFFFFF
            n += int(c.sum())
            sq += int((c * c).sum())
        del tabs
    return n, sq


def records(n: int, shared: bool):
    import synth_configs as sc

    recs = sc.cfg3(n, 24)
    if shared:
        out = [recs[0]]
        for (_, prev), (title, seq) in zip(recs, recs[1:]):
            m = len(seq) // 50
            at = len(seq) // 3
            out.append((title, seq[:at] + prev[:m] + seq[at + m:]))
        recs = out
    return recs


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=3_100_000_000, help="bases of synth_configs.cfg3 (24 records)")
    ap.add_argument("--runs", default="vec-r:31,vec:40", help="vec[-r]:k or masked[-r]:k, comma-separated")
    ap.add_argument("--shared", action="store_true", help="copy stretches between neighbouring records")
    ap.add_argument("--budget", type=int, default=None, help="device budget in bytes (default: free memory)")
    ap.add_argument("--dir", default=None, help="where the scratch output directory goes (default: TMPDIR)")
    args = ap.parse_args()

    from kman_b200 import fasta
    from kman_b200.engine import get_engine

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    eng = get_engine(0)
    t0 = time.perf_counter()
    recs = records(args.n, args.shared)
    d = eng.upload(fasta.from_records(recs), alphabet="ACGT")
    del recs
    print(f"# {gpu}; cfg3{' shared' if args.shared else ''} {args.n} bp uploaded in {time.perf_counter() - t0:.1f} s",
          flush=True)
    scratch = tempfile.mkdtemp(prefix="kmg_vec_", dir=args.dir)
    try:
        for run in args.runs.split(","):
            mode, k = run.split(":")
            rc, masked, k = mode.endswith("-r"), mode.startswith("masked"), int(k)
            out = os.path.join(scratch, f"{mode}_{k}")
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            t0 = time.perf_counter()
            plan = eng.write_vectors(d, k, rc, masked, out, budget_bytes=args.budget)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            files = sorted(os.listdir(out))
            res = {
                "gpu": gpu, "cmd": f"kmer count -m VEC_COUNT{'_MASKED' if masked else ''}{' -r' if rc else ''} k={k}",
                "bases": d.n_bases, "passes": plan.n_passes, "parts": plan.parts if plan.n_parts > 1 else None,
                "planned_pass_gb": [round(b / 1e9, 2) for b in plan.pass_bytes],
                "max_memory_allocated_gb": round(torch.cuda.max_memory_allocated() / 1e9, 2),
                "pass_ms": [round(x, 1) for x in plan.pass_ms], "text_ms": round(plan.text_ms, 1), "wall_s": round(wall, 2),
                "host_peak_rss_gb": round(peak_rss_gb(), 2), "files": len(files),
                "gz_gb": round(sum(os.path.getsize(os.path.join(out, f)) for f in files) / 1e9, 3),
            }
            print(json.dumps(res), flush=True)
            t0 = time.perf_counter()
            with ThreadPoolExecutor(min(16, os.cpu_count() or 1)) as pool:
                stats = list(pool.map(file_stats, [os.path.join(out, f) for f in files]))
            res = {"cmd": res["cmd"], "nonzero_entries": sum(s[0] for s in stats), "sum_entries": sum(s[1] for s in stats)}
            if not masked:
                kmers, squares = count_squares(eng, d, k, rc)
                res.update(kmers=kmers, sum_count_squared=squares, nonzero_equals_kmers=res["nonzero_entries"] == kmers,
                           sum_equals_sum_count_squared=res["sum_entries"] == squares)
            res["check_s"] = round(time.perf_counter() - t0, 1)
            print(json.dumps(res), flush=True)
            shutil.rmtree(out)
    finally:
        shutil.rmtree(scratch, ignore_errors=True)


if __name__ == "__main__":
    main()
