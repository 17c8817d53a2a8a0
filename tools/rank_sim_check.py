#!/usr/bin/env python
"""One rank's share of config 3 on 8 GPUs, on ONE GPU: 387.5 M random 62-bit keys that agree in their top
three bits, counted over the low 59 bits (what DistributedCounter hands to sort_count after the range
partition).  This is the one-bucket-per-tile regime of the local sort (16-bit prefix, buckets of ~5900 keys,
~8 % of the tiles own no bucket start) that smaller inputs never reach.  Checks: counts sum to n, keys strictly
ascending, sum(key * count) = sum(keys) mod 2^64.  usage: rank_sim_check.py [--n 387500000] [--rank 5] [--reps 3]"""
import argparse
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from kman_b200.engine import KeyArray, get_engine  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--n", type=int, default=387_500_000)
ap.add_argument("--rank", type=int, default=5)
ap.add_argument("--world", type=int, default=8)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--pb", type=int, default=0)
args = ap.parse_args()
eng = get_engine(0)
eng.lib.kmg_set_option(b"time_passes", 1)
eng.lib.kmg_set_option(b"hybrid_pb", args.pb)
n, key_bits = args.n, 62
part_bits = (args.world - 1).bit_length()
end_bit = key_bits - part_bits
gen = torch.Generator(device="cuda")
gen.manual_seed(99)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
for rep in range(args.reps):
    keys = torch.randint(0, 1 << end_bit, (n,), dtype=torch.int64, device="cuda", generator=gen) | (args.rank << end_bit)
    want_sum = int(keys.sum().item()) & (2**64 - 1)
    a = KeyArray(keys.view(torch.uint8), torch.empty(n * 8, dtype=torch.uint8, device="cuda"), None, None, n, 8, 0, 31, False)
    del keys
    torch.cuda.synchronize()
    e0.record()
    tab = eng.sort_count(a, end_bit)
    e1.record()
    torch.cuda.synchronize()
    k = tab.keys[: tab.n * 8].view(torch.int64)
    c = tab.counts[: tab.n * 4].view(torch.int32).to(torch.int64)
    assert int(c.sum().item()) == n, (int(c.sum().item()), n)
    assert bool((k[1:] > k[:-1]).all().item()), "keys not strictly ascending"
    got_sum = int((k * c).sum().item()) & (2**64 - 1)
    assert got_sum == want_sum, (got_sum, want_sum)
    kt = {nm: (eng.lib.kmg_get_stat((nm + "_ns").encode()), eng.lib.kmg_get_stat((nm + "_count").encode())) for nm in ("sort_pass", "local_sort")}
    print(f"rep {rep}: kernels (cumulative ns, launches) {kt}")
    print(f"rep {rep}: n {n} distinct {tab.n} sort_count {e0.elapsed_time(e1):.3f} ms  passes {eng.lib.kmg_get_stat(b'sort_passes')} "
          f"path {eng.lib.kmg_get_stat(b'hybrid_path')} irregular {eng.lib.kmg_get_stat(b'hybrid_irregular')}", flush=True)
    del a, tab, k, c
print("RANK_SIM_OK")
