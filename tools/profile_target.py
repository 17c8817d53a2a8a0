#!/usr/bin/env python
"""Minimal profiling target: two passes of the config-2 count path on cuda:0 -- the fused device path
(kmg_extract_sort_count; KMG_PROF_STAGE=1: the stage calls extract -> sort -> rle).  Run plain first,
then under ncu (B200_PROFILING.md).  KMG_PROF_N / _K / _VB."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from kman_b200 import fasta  # noqa: E402
from kman_b200.engine import get_engine  # noqa: E402

n = int(os.environ.get("KMG_PROF_N", "100000000"))
k = int(os.environ.get("KMG_PROF_K", "31"))
vb = int(os.environ.get("KMG_PROF_VB", "0"))
eng = get_engine(0)
rng = np.random.default_rng(1234)
bases = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, size=n, dtype=np.uint8)]
flat = fasta.FlatInput(np.concatenate([bases, np.array([10], np.uint8)]), np.array([0, n + 1], np.uint64), ["chr1"], ["chr1"])
d = eng.upload(flat, alphabet="ACGT", with_names=False)
stage = os.environ.get("KMG_PROF_STAGE") == "1"
for it in range(2):
    if stage:
        a = eng.extract(d, k, False, val_bytes=vb, reuse="p_", want_hist=True)
        r = eng.singletons(eng.sort(a)) if vb else eng.sort_count(a, reuse="p_")
    elif vb:
        r, _ = eng.uniq_narrow(d, k, False, reuse="p_", val_bytes=vb)
    else:
        r, _ = eng.count_narrow(d, k, False, reuse="p_")
torch.cuda.synchronize()
print("profile target done", r.n)
