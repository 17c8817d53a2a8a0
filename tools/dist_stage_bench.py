#!/usr/bin/env python
"""Per-stage wall-clock of the distributed count step (synchronising between stages; run under
torchrun with KMG_DIST_TIMING=1).  A development tool: the sum is larger than the pipelined step."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ["KMG_DIST_TIMING"] = "1"
from kman_b200 import fasta  # noqa: E402
from kman_b200.dist import DistributedCounter  # noqa: E402
from kman_b200.engine import get_engine  # noqa: E402

rank, world, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(lr)
dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
eng = get_engine(lr)
dc = DistributedCounter(eng)
n, k = int(os.environ.get("KMG_STAGE_N", "100000000")), 31  # bases per rank (config 3 on 8 GPUs: 387500000)
rng = np.random.default_rng(1234 + rank)
chunk = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, size=n, dtype=np.uint8)]
flat = fasta.FlatInput(chunk, np.array([0, n + 1], np.uint64), ["chr1"], ["chr1"])
d = eng.upload(flat, alphabet="ACGT", with_names=False)
d.pos_offset = rank * n
for it in range(8):
    if it == 3:
        dc._timing.clear()
        dc._t_last = None
        eng.lib.kmg_set_option(b"time_passes", 1)
    tab = dc.count(d, k, False)
if rank == 0:
    print(f"world {world}, {n} bases per rank, k={k}; shared cursors {dc.shared}; rows on rank 0: {tab.n}; sort passes "
          f"{eng.lib.kmg_get_stat(b'sort_passes')} path {eng.lib.kmg_get_stat(b'hybrid_path')}")
    for nm in ("sort_pass", "local_sort"):
        ns, c = eng.lib.kmg_get_stat((nm + "_ns").encode()), eng.lib.kmg_get_stat((nm + "_count").encode())
        if c:
            print(f"   kernel {nm:12s} {ns / 1e6 / 5:8.3f} ms per step ({c // 5} launches)")
    tot = sum(v for kk, v in dc._timing.items() if kk != "(outside)")
    for kk, v in dc._timing.items():
        print(f"{kk:36s} {v / 5 * 1e3:8.3f} ms")
    print(f"{'sum (serialised)':36s} {tot / 5 * 1e3:8.3f} ms")
dist.barrier()
dist.destroy_process_group()
