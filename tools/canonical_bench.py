#!/usr/bin/env python
"""Canonical k-mers (rc = KMG_CANONICAL) against forward-only (rc 0) and `-r` (rc 1) on one GPU, in one process:
  1. kmg_extract_sort_count / _histo / _uniq (Engine.count_narrow / histo_narrow / uniq_narrow with reused buffers)
     with rc 0, 1 and 2, alternated call by call, CUDA events around each call (every call synchronises the host
     internally), on config 2 (synth_configs.cfg2: 100 Mbp random ACGT, one record) at k = 31 and k = 63, and on
     tools/genome_like_bench.py's input at k = 31;
  2. with --cfg3 N: Engine.write_histogram and Engine.write_count (text into a sink that only counts bytes),
     canonical against -r, on synth_configs.cfg3(N) already on the device: wall time and passes of each plan.
Every canonical result is checked against the identities with the `-r` result of the same input: the count table
is the -r table restricted to keys <= their reverse complement with palindrome counts halved, the spectrum is that
table's, the singletons are its count-1 keys.  The card's name, power limit and SM clock are read in the same run.
usage: python tools/canonical_bench.py [--n 100000000] [--reps 10] [--cfg3 3100000000]"""
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


def rc_rows(keys: np.ndarray, k: int) -> np.ndarray:
    """Reverse complements of narrow keys: (n,) uint64 (k <= 32) or (n, 2) uint64 limbs, least significant first."""
    if keys.ndim == 1:
        x, out = ~keys, np.zeros_like(keys)
        for i in range(k):
            out = (out << np.uint64(2)) | ((x >> np.uint64(2 * i)) & np.uint64(3))
        return out
    lo, hi = ~keys[:, 0], ~keys[:, 1]
    rlo, rhi = np.zeros_like(lo), np.zeros_like(lo)
    for i in range(k):
        c = ((lo >> np.uint64(2 * i)) if i < 32 else (hi >> np.uint64(2 * i - 64))) & np.uint64(3)
        rhi = (rhi << np.uint64(2)) | (rlo >> np.uint64(62))
        rlo = (rlo << np.uint64(2)) | c
    return np.stack([rlo, rhi], axis=1)


def le(a: np.ndarray, b: np.ndarray):
    """(a <= b, a == b) row-wise for the key layouts of rc_rows."""
    if a.ndim == 1:
        return a <= b, a == b
    eq = (a[:, 1] == b[:, 1]) & (a[:, 0] == b[:, 0])
    return (a[:, 1] < b[:, 1]) | ((a[:, 1] == b[:, 1]) & (a[:, 0] <= b[:, 0])), eq


def run_input(eng, d, k, reps, label):
    from kman_b200.engine import CANONICAL

    n_win = d.n_bases - k + 1
    acc = torch.zeros(8 * (BINS + 1) + 4 * (2 * n_win // BINS + 1), dtype=torch.uint8, device=eng.device)
    out = (acc.data_ptr(), acc.data_ptr() + 8 * (BINS + 1), acc.data_ptr() + 8 * BINS)
    rules = {"fwd": False, "rc": True, "canonical": CANONICAL}

    def count(rc):
        return eng.count_narrow(d, k, rc, reuse="cb_")[0]

    def histo(rc):
        acc.zero_()
        eng.histo_narrow(d, k, rc, out, reuse="cb_")

    def uniq(rc):
        return eng.uniq_narrow(d, k, rc, reuse="cb_", val_bytes=8)[0]

    # identities, from one call of each
    t = count(True)
    rk, rcnt = t.keys_host().copy(), t.counts_host().astype(np.int64)
    t = count(CANONICAL)
    ck, ccnt = t.keys_host().copy(), t.counts_host().astype(np.int64)
    keep, pal = le(rk, rc_rows(rk, k))
    want_c = np.where(pal[keep], rcnt[keep] // 2, rcnt[keep])
    ok_count = np.array_equal(ck, rk[keep]) and np.array_equal(ccnt, want_c)
    histo(CANONICAL)
    wm, wn = np.unique(want_c, return_counts=True)
    gm, gn = read_histo(acc)
    ok_histo = np.array_equal(gm, wm.astype(np.uint64)) and np.array_equal(gn, wn.astype(np.uint64))
    s = uniq(CANONICAL)
    ok_uniq = np.array_equal(s.keys_host(), rk[keep][want_c == 1])
    del t, s, rk, rcnt, ck, ccnt
    ms = {(op, name): [] for op in ("count", "histo", "uniq") for name in rules}
    for op, fn in (("count", count), ("histo", histo), ("uniq", uniq)):
        for rc in rules.values():  # warm-up
            fn(rc)
        for _ in range(reps):
            for name, rc in rules.items():
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record()
                fn(rc)
                t1.record()
                t1.synchronize()
                ms[(op, name)].append(t0.elapsed_time(t1))
    eng._scratch.clear()
    torch.cuda.empty_cache()
    med = {f"{op}_{name}_ms": round(float(np.median(v)), 3) for (op, name), v in ms.items()}
    print(json.dumps({"input": label, "k": k, "windows": n_win, "reps": reps, "identity_count": bool(ok_count),
                      "identity_histo": bool(ok_histo), "identity_uniq": bool(ok_uniq), **med}), flush=True)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=100_000_000)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--cfg3", type=int, default=0, help="bases of synth_configs.cfg3 (0: skip the genome-size run)")
    args = ap.parse_args()

    import synth_configs as sc

    from kman_b200 import fasta
    from kman_b200.engine import CANONICAL, get_engine

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print(f"# {gpu}", flush=True)
    eng = get_engine(0)

    d = eng.upload(fasta.from_records(sc.cfg2(args.n)), alphabet="ACGT", with_names=False)
    for k in (31, 63):
        run_input(eng, d, k, args.reps, f"cfg2 {args.n} bp")
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
    run_input(eng, d, 31, args.reps, f"genome_like {args.n} bp")
    del d, flat, parts
    eng._scratch.clear()
    torch.cuda.empty_cache()

    if args.cfg3:
        t0 = time.perf_counter()
        d = eng.upload(fasta.from_records(sc.cfg3(args.cfg3, 24)), alphabet="ACGT", with_names=False)
        print(f"# cfg3 {args.cfg3} bp uploaded in {time.perf_counter() - t0:.1f} s", flush=True)
        for name, rc in (("canonical", CANONICAL), ("rc", True), ("canonical", CANONICAL), ("rc", True)):
            for what in ("histogram", "count"):
                sink = NullSink()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                plan = (eng.write_histogram if what == "histogram" else eng.write_count)(d, 31, rc, sink)
                torch.cuda.synchronize()
                wall = time.perf_counter() - t0
                print(json.dumps({"cmd": f"Engine.write_{what} k=31 {name}", "bases": d.n_bases, "passes": plan.n_passes,
                                  "pass_ms": [round(x, 1) for x in plan.pass_ms], "wall_s": round(wall, 2),
                                  "bytes_written": sink.bytes}), flush=True)
                eng._scratch.clear()
                torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
