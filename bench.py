#!/usr/bin/env python
"""Benchmark of the k-mer hot path (extract + sort + count, k=31) -- BASELINE.json's metric.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload cfg2|cfg3]
                  [--dump-outputs DIR]
  (N>1: launched by torchrun, one rank per GPU; rank 0 prints ONE JSON line)

A "step" is one pass of the hot path over one synthetic input (--workload auto):
  N=1 : config 2 of BASELINE.json -- 100 Mbp random-ACGT single record, k=31, count
  N>1 : config 3 -- 3.1 Gbp synthetic genome of 24 records (lengths proportional to the human
        chromosomes), k=31, count, STRONG scaling: every rank holds 1/N of the flat base buffer (k-1
        base overlap, chunk boundaries fall anywhere, also inside and next to record separators),
        keys are range-partitioned by their top bits and exchanged over NVLink
        (--workload cfg2 keeps the round-1 weak-scaling workload: one 100 Mbp chunk per GPU;
         --workload cfg3 runs config 3 on any N, one GPU included)
`verify`  : checked outside the timed region on every N: counts sum to the number of windows, distinct
           keys strictly ascending inside every rank and across rank boundaries, and sum(key * count)
           == sum of all extracted keys (mod 2^64, all-reduced)
`value`  : whole-job k-mers/s with the bases already resident in HBM (device-timed, max over ranks)
`e2e`    : the same metric through the host-buffer C-ABI call kmg_count_host (N=1) or the
           distributed Python API (N>1), pinned host memory, H2D of the bases and D2H of the
           (k-mer, count) table inside the timed region
`roofline`: onesweep pass kernel, algorithmic bytes 2*W per key per launch, live CUDA-event
           timing of every launch inside the timed region; `local_sort` is the same for the hybrid
           finish's kernel; `sort_model_frac` = 2*W bytes per key per launch over the whole sort,
           `sort_lsd8_model_frac` = SURVEY.md §8d's fixed 8-bit LSD model N*W*(2*P8+1) over the same time
`cpu_baseline` / --impl reference: the oracle's numpy port of the reference algorithm on the
           host cores (bounded sample) -- a reported baseline, not the target.
--dump-outputs DIR: after the timed steps, the (k-mer, count) table of the last one is written to
           DIR as float64 .npy files (see dump_outputs; `bench_outputs/` is ignored by git).  The
           inputs are seeded, so two builds run with the same arguments can be compared file by file.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

K = 31
CFG2_BASES = 100_000_000
CFG3_BASES = 3_100_000_000
METRIC = "k-mers/sec (extract+sort+count, k=31)"
CFG3_RECORDS = 24
HUMAN_MBP = [248, 242, 198, 190, 182, 171, 159, 145, 138, 134, 135, 133, 114, 107, 102, 90, 83, 80, 59, 64, 47, 51, 156, 57]


def cfg3_layout(total=CFG3_BASES):
    """Flat buffer of config 3: `total` bytes, record r followed by one '\n' separator.  Returns
    (separator positions, number of windows = sum over records of max(0, len - K + 1))."""
    w = np.array(HUMAN_MBP, np.float64)
    ends = np.floor(np.cumsum(w) / w.sum() * total).astype(np.int64)
    ends[-1] = total
    seps = ends - 1  # last byte of every record's slot is its separator
    starts = np.concatenate(([0], ends[:-1]))
    lens = seps - starts
    return seps, int(np.maximum(0, lens - K + 1).sum())


def cfg3_slice(b: int, e: int) -> np.ndarray:
    """Bytes [b, e) of config 3's flat buffer: block i of 100 Mbp comes from seed 1234+i, so every
    rank builds only its own slice."""
    blk = 100_000_000
    parts = []
    for i in range(b // blk, (e + blk - 1) // blk):
        x = synth_bases(blk, 1234 + i)
        parts.append(x[max(b - i * blk, 0) : min(e - i * blk, blk)])
    out = np.concatenate(parts)
    seps, _ = cfg3_layout()
    inside = seps[(seps >= b) & (seps < e)]
    out[inside - b] = 10
    return out


def synth_bases(n: int, seed: int) -> np.ndarray:
    """SURVEY.md §8d generator: uniform random ACGT."""
    rng = np.random.default_rng(seed)
    out = np.empty(n, np.uint8)
    step = 1 << 26
    lut = np.frombuffer(b"ACGT", np.uint8)
    for s in range(0, n, step):
        m = min(step, n - s)
        out[s : s + m] = lut[rng.integers(0, 4, size=m, dtype=np.uint8)]
    return out


def peak_hbm_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock + throttle reasons sampled every ~10 ms WHILE the timed region runs (NVML in a
    thread; falls back to one `nvidia-smi` query if NVML is unavailable)."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index: int):
        import threading

        self.index = index
        self.samples, self.reason_bits, self.max_mhz = [], 0, None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml

            pynvml.nvmlInit()
            # honour CUDA_VISIBLE_DEVICES-style remapping when the UUID is available through torch
            import torch

            uuid = str(torch.cuda.get_device_properties(index).uuid)
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.nv = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.reason_bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:
                pass
            self._stop.wait(0.01)

    def stop(self):
        if self._thread is not None:
            self._stop.set()
            self._thread.join(timeout=2)
            sm = sorted(self.samples)
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz,
                    "reasons": sorted(v for b, v in self.REASONS.items() if self.reason_bits & b),
                    "samples": len(sm), "source": "nvml, 10 ms period, timed region only"}
        try:
            out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=clocks.sm,clocks.max.sm",
                                  "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10).stdout
            a, b = [float(x) for x in out.strip().split(",")[:2]]
            return {"sm_mhz": a, "sm_max_mhz": b, "reasons": [], "samples": 1, "source": "nvidia-smi after the run"}
        except Exception:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"], "samples": 0}


# ---- reference arm / cpu baseline -------------------------------------------------------------------
def host_threads() -> int:
    return len(os.sched_getaffinity(0))


def cpu_port_rate(sample_bases: int, steps: int, warmup: int, budget_s: float = 240.0):
    """k-mers/s of the oracle's numpy port of the same stages the GPU arm times (extract -> stable
    sort -> run-length grouping into the binary (k-mer, count) table) on ALL host threads this process
    may use: chunks with k-1 overlap extracted and sorted by a thread each, merge + grouping split by
    key range (oracle/kmer_oracle.py: count_table_np_threads -- the shape of `kmer batch --threads N`
    followed by the join).  Stops after `budget_s` seconds.  Returns (rate, seconds per pass, threads, passes timed)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import kmer_oracle as ko

    threads = host_threads()
    seq = synth_bases(sample_bases, 1234).tobytes().decode()
    recs = [("chr1 synthetic seed=1234", seq)]
    ts = []
    t_start = time.perf_counter()
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        keys, counts = ko.count_table_np_threads(recs, K, False, "ACGT", threads=threads)
        dt = time.perf_counter() - t0
        if i >= warmup:
            ts.append(dt)
        if ts and time.perf_counter() - t_start + dt > budget_s:
            break  # (the caller reports len(ts) as the number of steps timed)
    n_win = sample_bases - K + 1
    assert int(counts.sum()) == n_win
    return n_win / (sum(ts) / len(ts)), sum(ts) / len(ts), threads, len(ts)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # N=1: the FULL configuration (config 2, 100 Mbp).  N>1: config 3 is 3.1 Gbp -- the port would need
    # > 100 GB of host memory; its step is a 100 Mbp sample of the same generator.  Either way a step is
    # one pass over 100 Mbp (~10 s on 16 threads); --steps / --warmup are honoured as far as a 4-minute
    # budget allows (one warm-up pass at most), and `steps` reports the passes actually timed.
    sample = int(os.environ.get("KMG_BENCH_REF_BASES", CFG2_BASES))  # (the CPU test-suite shrinks it)
    warm = min(args.warmup, 1)
    rate, sec, threads, steps = cpu_port_rate(sample, max(1, args.steps), warm)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": "k-mers/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": workload_config(args, sample_note=("the full configuration" if args.workload == "cfg2" and args.gpus == 1 and sample == CFG2_BASES
                                                      else f"bounded sample: {sample} bases of the same generator per step")),
        "cpu_baseline": {"value": rate, "unit": "k-mers/s", "cores": threads, "kind": "port",
                         "sample": f"{sample} bp random ACGT, k={K}, count; oracle numpy port on {threads} threads "
                                   f"(chunked extract + sort per thread, merge + grouping split by key range)",
                         "host_cores_available": os.cpu_count()},
        "e2e": {"value": rate, "unit": "k-mers/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def workload_config(args, sample_note=None, p2p=None, shared=None):
    n = args.gpus
    if p2p is None:
        p2p = os.environ.get("KMG_DIST_P2P", "1") != "0"
    if args.workload == "cfg3":
        wl = (f"config 3: {CFG3_BASES} bp synthetic random-ACGT genome in {CFG3_RECORDS} records (lengths proportional to "
              f"the human chromosomes), k={K}, count, strong scaling over {n} GPU(s): 1/{n} of the flat base buffer per GPU "
              "with k-1 overlap, range partition by the top key bits"
              + ("" if n == 1 else ("; exchange: fused extract+partition kernel storing into the owners' buffers over NVLink "
                                     "(CUDA IPC peer memory)" if p2p else "; exchange: range partition pass + NCCL all-to-all")))
    elif n == 1:
        wl = f"config 2: {CFG2_BASES} bp synthetic random-ACGT single record (seed 1234), k={K}, count"
    else:
        wl = (f"config 2 x {n} (weak): {n}x{CFG2_BASES} bp synthetic random-ACGT genome, one {CFG2_BASES} bp chunk per GPU "
              f"with k-1 overlap, range partition by the top key bits, k={K}, count; exchange: "
              + (("fused extract+partition kernel storing into the owners' buffers over NVLink (CUDA IPC peer memory), "
                  + ("one launch, shared per-destination cursors" if shared else "count-only launch + exact regions"))
                 if p2p else "range partition pass + NCCL all-to-all of the partitioned keys"))
    cfg = {"workload": wl, "k": K, "mode": "count", "alphabet": "ACGT",
           "l2": "working set per step (>= 0.8 GB of keys written and re-read + a 1.2 GB table per 100 M k-mers per GPU) "
                 ">> 126 MB L2; no explicit flush"}
    if sample_note:
        cfg["reference_sample"] = sample_note
    return cfg


def verify_table(eng, d, tab, n_win_global, world, rank):
    """Outside the timed region: size-independent properties of the result of ONE step, over all ranks.
    (kmermaid/join.py:95-130: every window lands in exactly one group; batch.py:156-168 + join.py:63-93:
    groups come out in ascending key order; rank r owns key range r.)"""
    import torch
    import torch.distributed as dist

    keys = tab.keys[: tab.n * 8].view(torch.int64)
    counts = tab.counts[: tab.n * 4].view(torch.int32).to(torch.int64)
    asc = bool((keys[1:] > keys[:-1]).all()) if tab.n > 1 else True  # 62-bit keys: signed compare is exact
    a = eng.extract(d, K, False, val_bytes=0)  # this rank's windows, extraction order
    sum_in = a.keys[: a.n * 8].view(torch.int64).sum() if a.n else torch.zeros((), dtype=torch.int64, device=eng.device)
    n_in = a.n
    del a
    red = torch.stack([counts.sum(), (keys * counts).sum(), sum_in, torch.tensor(n_in, device=eng.device),
                       torch.tensor(tab.n, device=eng.device), torch.tensor(0 if asc else 1, device=eng.device)])
    edge = torch.stack([keys[0], keys[-1]]) if tab.n else torch.tensor([-1, -1], dtype=torch.int64, device=eng.device)
    cross = True
    if world > 1:
        dist.all_reduce(red)  # (int64 sums wrap modulo 2^64 on every path alike)
        edges = torch.empty(2 * world, dtype=torch.int64, device=eng.device)
        dist.all_gather_into_tensor(edges, edge)
        prev = -1
        for r, (first, last) in enumerate(edges.view(world, 2).tolist()):
            if first < 0:
                continue
            cross = cross and first > prev
            prev = last
    total, kc, ks, n_keys, rows, bad = (int(x) for x in red.tolist())
    ok = total == n_win_global and n_keys == n_win_global and kc == ks and bad == 0 and cross
    return {"ok": bool(ok), "windows": n_win_global, "counts_sum": total, "keys_extracted": n_keys, "distinct": rows,
            "ascending_within_ranks": bad == 0, "ascending_across_ranks": bool(cross),
            "sum_key_times_count_eq_sum_keys_mod_2_64": kc == ks}


DUMP_ROWS = 1 << 20  # 4 float64 arrays of this many rows: 32 MB


def dump_rows(n: int) -> np.ndarray:
    """Rows of an n-row table that --dump-outputs writes: all of them up to DUMP_ROWS, else a fixed
    seeded sample; ascending."""
    if n <= DUMP_ROWS:
        return np.arange(n, dtype=np.int64)
    return np.sort(np.random.default_rng(1234).choice(n, DUMP_ROWS, replace=False))


def dump_outputs(out_dir, eng, tab, world, rank):
    """Writes the (k-mer, count) table of one step -- the rank-order concatenation of every rank's slice,
    i.e. the whole job's table, so the files do not depend on N for the same workload -- as float64 .npy
    files in `out_dir`: `n_rows` (the table's length), the sampled `rows` (dump_rows) and their `keys_hi`,
    `keys_lo` (the 2k-bit k-mer code split at bit 31, so both halves are exact in float64) and `counts`."""
    import torch
    import torch.distributed as dist

    ns = [tab.n]
    if world > 1:
        ns = [None] * world
        dist.all_gather_object(ns, tab.n)
    off = sum(ns[:rank])
    rows = dump_rows(sum(ns))
    mine = torch.from_numpy(rows[(rows >= off) & (rows < off + tab.n)] - off).to(eng.device)
    keys = tab.keys[: tab.n * 8].view(torch.int64)[mine].cpu().numpy().view(np.uint64)
    counts = tab.counts[: tab.n * 4].view(torch.int32)[mine].cpu().numpy().view(np.uint32)
    parts = [(keys, counts)]
    if world > 1:
        parts = [None] * world if rank == 0 else None
        dist.gather_object((keys, counts), parts, dst=0)
    if rank != 0:
        return
    keys = np.concatenate([p[0] for p in parts])
    counts = np.concatenate([p[1] for p in parts])
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"n_rows": np.array([sum(ns)]), "rows": rows, "keys_hi": keys >> np.uint64(31),
              "keys_lo": keys & np.uint64((1 << 31) - 1), "counts": counts}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


# ---- GPU arm --------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="kmg", choices=["kmg", "reference"])
    ap.add_argument("--workload", default="auto", choices=["auto", "cfg2", "cfg3"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's table to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's table; it is not available with --impl reference")
    if args.workload == "auto":
        # N=1: the configuration the single-GPU path is quoted on; N>1: BASELINE.json's scaling configuration
        args.workload = "cfg2" if args.gpus == 1 else "cfg3"
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist

    from kman_b200 import _lib, alphabet as ab, fasta
    from kman_b200.engine import get_engine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torchrun for N>1)"
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    eng = get_engine(local_rank)
    lib = eng.lib

    # ---- synthetic input (this rank's chunk only) ---------------------------------------------
    if args.workload == "cfg3":
        from kman_b200.dist import chunk_bases

        total = CFG3_BASES
        b, e = chunk_bases(total, K, world)[rank]
        chunk = cfg3_slice(b, e)  # every rank generates only its slice
        n_win_global = cfg3_layout()[1]
    else:
        total = CFG2_BASES * world
        # weak scaling: rank r owns block r (+ k-1 bases of block r+1)
        chunk = synth_bases(CFG2_BASES, 1234 + rank)
        if rank + 1 < world:
            chunk = np.concatenate([chunk, synth_bases(CFG2_BASES, 1234 + rank + 1)[: K - 1]])
        b = rank * CFG2_BASES
        n_win_global = total - K + 1
    flat = fasta.FlatInput(chunk, np.array([0, chunk.size + 1], np.uint64), ["chr1"], ["chr1"])
    d = eng.upload(flat, alphabet="ACGT", with_names=False)
    d.pos_offset = b
    n_local = d.n_bases - K + 1

    if world > 1:
        from kman_b200.dist import DistributedCounter

        dc = DistributedCounter(eng)

        def step():
            return dc.count(d, K, False)
    else:
        def step():
            # ONE native call: histogram pre-pass over the bases, extraction fused with the first prefix
            # pass, remaining prefix pass(es), local sort emitting the (k-mer, count) table
            return eng.count_narrow(d, K, False, reuse="bench_")[0]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        tab = step()
    verify = verify_table(eng, d, tab, n_win_global, world, rank)
    assert verify["ok"], verify

    lib.kmg_set_option(b"time_passes", 1)
    lib.kmg_get_stat(b"reset_launches")
    sampler = ClockSampler(local_rank) if rank == 0 else None
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    t_wall0 = time.perf_counter()
    for i in range(args.steps):
        ev[i][0].record()
        tab = step()
        ev[i][1].record()
    barrier()
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop() if sampler else None
    launches = int(lib.kmg_get_stat(b"launches"))
    pass_ns = int(lib.kmg_get_stat(b"sort_pass_ns"))
    pass_cnt = int(lib.kmg_get_stat(b"sort_pass_count"))
    ls_ns = int(lib.kmg_get_stat(b"local_sort_ns"))
    ls_cnt = int(lib.kmg_get_stat(b"local_sort_count"))
    lib.kmg_set_option(b"time_passes", 0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, eng, tab, world, rank)  # before the N>1 e2e steps overwrite `tab`
    dev_ms = sum(a.elapsed_time(b_) for a, b_ in ev)
    tmax = torch.tensor([dev_ms], dtype=torch.float64, device=eng.device)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    dev_ms = float(tmax.item())
    ms_per_step = dev_ms / args.steps
    value = n_win_global / (ms_per_step / 1e3)

    # ---- roofline of the dominant kernel (rank 0's launches) ------------------------------------
    peak, peak_src = peak_hbm_gbs()
    W = 8
    P8 = (2 * K + 7) // 8
    roofline = None
    if pass_cnt:
        avg_pass_ms = pass_ns / 1e6 / pass_cnt
        n_keys = n_local if world == 1 else n_win_global / world
        passes_per_sort = pass_cnt / args.steps
        local_per_sort = ls_cnt / args.steps
        avg_local_ms = ls_ns / 1e6 / ls_cnt if ls_cnt else 0.0
        # plain LSD: P8 passes (a sort of more than 2^30 keys runs every pass in several launches);
        # hybrid finish: 2-3 prefix passes + one local-sort launch, every one a read + write of the keys
        n_passes = int(lib.kmg_get_stat(b"sort_passes")) or P8  # passes of the last sort (2-3 with the hybrid finish)
        launches_per_pass = max(1.0, passes_per_sort / n_passes)
        alg_bytes = 2 * W * n_keys / launches_per_pass
        achieved = alg_bytes / (avg_pass_ms / 1e3) / 1e9
        sort_ms = avg_pass_ms * passes_per_sort + avg_local_ms * local_per_sort
        model_launches = passes_per_sort / launches_per_pass + local_per_sort
        roofline = {
            "bound": "hbm", "kernel": "kmg::onesweep_kernel (one radix pass: read + write of every key)",
            "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": achieved / peak,
            "traffic": None, "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": avg_pass_ms,
            "launches_per_step": passes_per_sort,
            "sort_model_bytes_per_kmer": 2 * W * model_launches,
            "sort_model_frac": (2 * W * model_launches * n_keys) / (sort_ms / 1e3) / 1e9 / peak,
            "sort_ms_per_step": sort_ms,
            # SURVEY.md 8d's fixed 8-bit LSD model (W*(2*P8+1) bytes per key) over the same time: above 1
            # means the sort moved fewer bytes than that model (the hybrid finish does)
            "sort_lsd8_model_bytes_per_kmer": W * (2 * P8 + 1),
            "sort_lsd8_model_frac": (W * (2 * P8 + 1) * n_keys) / (sort_ms / 1e3) / 1e9 / peak,
        }
        if ls_cnt:
            # fused count: reads every key once, writes one (key, count) pair per distinct k-mer
            n_distinct = int(tab.n)
            ls_bytes = W * n_keys + (W + 4) * n_distinct
            ls_ach = ls_bytes / (avg_local_ms / 1e3) / 1e9
            local = {"bound": "hbm", "kernel": "kmg::local_sort_fine_kernel<uint64_t, EMIT=count, VB=0> (hybrid finish + run-length count: reads every "
                     "key, writes the (k-mer, count) table)",
                     "achieved": ls_ach, "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": ls_ach / peak,
                     "traffic": None, "algorithmic_bytes_per_launch": ls_bytes, "avg_launch_ms": avg_local_ms,
                     "launches_per_step": local_per_sort}
            if avg_local_ms * local_per_sort > avg_pass_ms * passes_per_sort:
                # the local sort is the larger share of the step: it is the kernel the roofline is quoted on
                for key in ("sort_model_bytes_per_kmer", "sort_model_frac", "sort_ms_per_step",
                            "sort_lsd8_model_bytes_per_kmer", "sort_lsd8_model_frac"):
                    local[key] = roofline.pop(key)
                local["onesweep"] = roofline
                roofline = local
            else:
                roofline["local_sort"] = local
        prof = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(prof):
            try:
                tj = json.load(open(prof))
                if "onesweep" in roofline:
                    roofline["traffic"] = tj.get("local_sort_dram_bytes_per_launch")
                    roofline["onesweep"]["traffic"] = tj.get("onesweep_dram_bytes_per_launch")
                else:
                    roofline["traffic"] = tj.get("onesweep_dram_bytes_per_launch")
            except Exception:
                pass

    # ---- e2e: host buffers in, host table out ------------------------------------------------------
    e2e = None
    if not args.no_e2e:
        e2e_steps = max(1, min(args.steps, 5))
        h_bases = torch.from_numpy(chunk).pin_memory()
        if world == 1:
            lut, _ = ab.lut_tables("ACGT", ab.NATYPES.DNA)
            cap = n_local
            h_keys = torch.empty(cap, dtype=torch.int64).pin_memory()
            h_counts = torch.empty(cap, dtype=torch.int32).pin_memory()
            n_out = C.c_uint64(0)
            ctx = C.c_void_p()
            _lib.check(lib.kmg_ctx_create(local_rank, C.byref(ctx)))

            def e2e_step():
                _lib.check(lib.kmg_count_host(ctx, h_bases.data_ptr(), chunk.size, K, 0, lut.ctypes.data,
                                              h_keys.data_ptr(), h_counts.data_ptr(), cap, C.byref(n_out)))
                return chunk.size, n_out.value * 12

            e2e_step()
        else:
            h_keys = h_counts = None

            def e2e_step():
                nonlocal h_keys, h_counts
                d.bases[: chunk.size].copy_(h_bases, non_blocking=True)
                t = dc.count(d, K, False)
                if h_keys is None or h_keys.numel() < t.n * 8:
                    h_keys = torch.empty(int(t.n * 8 * 1.05), dtype=torch.uint8).pin_memory()
                    h_counts = torch.empty(int(t.n * 4 * 1.05), dtype=torch.uint8).pin_memory()
                h_keys[: t.n * 8].copy_(t.keys[: t.n * 8], non_blocking=True)
                h_counts[: t.n * 4].copy_(t.counts[: t.n * 4], non_blocking=True)
                torch.cuda.synchronize()
                return chunk.size, t.n * 12

            e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            h2d, d2h = e2e_step()
        barrier()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=eng.device)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e = {"value": n_win_global / (float(tt.item()) / e2e_steps), "unit": "k-mers/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(d2h), "steps": e2e_steps,
               "api": "kmg_count_host (C ABI, pinned host buffers)" if world == 1 else "kman_b200.dist.DistributedCounter.count + pinned copies (per rank bytes)"}
        if world == 1:
            lib.kmg_ctx_destroy(ctx)

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # (a bounded sample: half of config 2, one pass; ~5 s on 8-16 threads)
        rate, sec, threads, _ = cpu_port_rate(50_000_000, 1, 0)
        cpu_baseline = {"value": rate, "unit": "k-mers/s", "cores": threads, "kind": "port",
                        "sample": f"50000000 bp of the same generator, k={K}, count; oracle numpy port on {threads} threads, "
                                  f"{sec:.1f} s per pass",
                        "host_cores_available": os.cpu_count()}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "k-mers/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong" if args.workload == "cfg3" else "weak", "vs_baseline": None, "dtype": "u64",
            "data": "synthetic", "config": workload_config(args, p2p=(dc.p2p if world > 1 else None), shared=(dc.shared if world > 1 else None)), "clocks": clocks,
            "e2e": e2e, "verify": verify,
            "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu_baseline,
            "wall_ms_per_step": t_wall / args.steps * 1e3, "kmers_per_step": n_win_global,
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
