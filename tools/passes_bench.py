#!/usr/bin/env python
"""Genome-scale `kmer count` / `kmer uniq` on one GPU through the key-range pass writers
(Engine.write_count / write_uniq), streamed into a sink that hashes the bytes (sha256) and counts
lines instead of writing a file.  The sink also checks that the rows ascend across pass and chunk
boundaries and, for count, that the counts add up to the number of k-mers.

Reports per command: passes, torch.cuda.max_memory_allocated, time per pass (CUDA events), wall time
and the host's peak RSS.

usage: python tools/passes_bench.py [--n 3100000000] [--runs count:31,uniq-r:40] [--budget BYTES]"""
import argparse
import hashlib
import json
import os
import resource
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402


class CheckingSink:
    """Binary file object that keeps nothing: sha256 and line count of the bytes, and checks on the rows.
    Every write ends at a row boundary, and rows inside a write come from one sorted table slice, so the
    order check compares the first k-mer of each write with the last one of the write before: that is
    every chunk and pass boundary.  For count, the counts must add up to the number of k-mers.  The
    line checks run on a second thread while the calling thread hashes."""

    def __init__(self, mode: str, k: int):
        self.h = hashlib.sha256()
        self.mode, self.k = mode, k
        self.bytes = self.lines = self.total = self.out_of_order = 0
        self.unterminated = 0
        self.prev = b""
        self.pool = ThreadPoolExecutor(1)

    def _seq_at(self, a: np.ndarray, line_start: int) -> bytes:
        return a[line_start:line_start + self.k].tobytes()

    def _check(self, a: np.ndarray) -> None:
        if a[-1] != 10:
            self.unterminated += 1
        if self.mode == "uniq":  # ">NAME:START-END:STRAND\nSEQ\n" records: the SEQ lines
            self.lines += int(np.count_nonzero(a == 10))
            head = a[:4096].tobytes()
            first = head.index(b"\n") + 1
            tail_at = max(0, a.size - 4096)
            tail = a[tail_at:-1].tobytes()
            last = tail_at + tail.rindex(b"\n") + 1
        else:  # "SEQ\tCOUNT\n": also add up the counts (digits between the tab and the newline)
            nl = np.flatnonzero(a == 10)
            self.lines += int(nl.size)
            starts = np.concatenate(([0], nl[:-1] + 1))
            first, last = 0, int(starts[-1])
            ndig = nl - (starts + self.k + 1)
            val = np.zeros(nl.size, np.int64)
            scale = 1
            for j in range(int(ndig.max())):
                has = ndig > j
                val[has] += (a[nl[has] - 1 - j].astype(np.int64) - 48) * scale
                scale *= 10
            self.total += int(val.sum())
        self.out_of_order += int(self._seq_at(a, first) <= self.prev)
        self.prev = self._seq_at(a, last)

    def write(self, b) -> int:
        mv = memoryview(b).cast("B")
        if mv.nbytes == 0:
            return 0
        job = self.pool.submit(self._check, np.frombuffer(mv, np.uint8))
        self.h.update(mv)
        job.result()
        self.bytes += mv.nbytes
        return mv.nbytes


def peak_rss_gb() -> float:
    return resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 1e6


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=3_100_000_000, help="bases of synth_configs.cfg3 (24 records)")
    ap.add_argument("--runs", default="count:31,uniq-r:40", help="mode[-r]:k, comma-separated")
    ap.add_argument("--budget", type=int, default=None, help="device budget in bytes (default: free memory)")
    args = ap.parse_args()

    import synth_configs as sc

    from kman_b200 import fasta
    from kman_b200.engine import get_engine

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    eng = get_engine(0)
    t0 = time.perf_counter()
    recs = sc.cfg3(args.n, 24)
    d = eng.upload(fasta.from_records(recs), alphabet="ACGT")
    del recs
    print(f"# {gpu}; cfg3 {args.n} bp uploaded in {time.perf_counter() - t0:.1f} s", flush=True)
    for run in args.runs.split(","):
        mode, k = run.split(":")
        rc = mode.endswith("-r")
        mode, k = mode.replace("-r", ""), int(k)
        sink = CheckingSink(mode, k)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        t0 = time.perf_counter()
        writer = eng.write_count if mode == "count" else eng.write_uniq
        plan = writer(d, k, rc, sink, budget_bytes=args.budget)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        n_win = d.n_bases - 24 * k  # windows inside the 24 records (each followed by one separator byte)
        res = {
            "gpu": gpu, "cmd": f"kmer {mode}{' -r' if rc else ''} k={k}", "bases": d.n_bases, "passes": plan.n_passes,
            "parts": plan.parts if plan.n_parts > 1 else None, "max_memory_allocated_gb": torch.cuda.max_memory_allocated() / 1e9,
            "pass_ms": [round(x, 1) for x in plan.pass_ms], "wall_s": round(wall, 2), "host_peak_rss_gb": round(peak_rss_gb(), 2),
            "planned_pass_gb": [round(b / 1e9, 2) for b in plan.pass_bytes],
        }
        n_keys = n_win * (2 if rc else 1)
        res.update(sha256=sink.h.hexdigest(), bytes=sink.bytes, lines=sink.lines, rows_out_of_order=sink.out_of_order,
                   writes_not_ending_a_row=sink.unterminated)
        if mode == "count":
            res.update(count_total=sink.total, kmers=n_keys, counts_add_up=sink.total == n_keys)
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
