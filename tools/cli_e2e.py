#!/usr/bin/env python
"""Wall-clock of the drop-in command line on a synthetic FASTA (file in, file out), per mode: `kmer count`,
`kmer uniq`, `kmer batch` (sorted batch files in an output folder) and `kmer count -m VEC_COUNT` (one gzipped
abundance vector per record and strand in an output folder).
usage: python tools/cli_e2e.py [--n 20000000] [--k 31]"""
import argparse
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ap = argparse.ArgumentParser()
ap.add_argument("--n", type=int, default=20_000_000)
ap.add_argument("--k", type=int, default=31)
args = ap.parse_args()
tmp = tempfile.mkdtemp(prefix="kmg_cli_")
fa = os.path.join(tmp, "genome.fa")
rng = np.random.default_rng(11)
seq = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, size=args.n, dtype=np.uint8)]
with open(fa, "wb") as fh:
    fh.write(b">chr1 synthetic\n")
    lines = seq.reshape(-1, 80) if args.n % 80 == 0 else None
    if lines is not None:
        fh.write(np.concatenate([lines, np.full((lines.shape[0], 1), 10, np.uint8)], axis=1).tobytes())
    else:
        fh.write(seq.tobytes() + b"\n")
env = dict(os.environ, PYTHONPATH=ROOT, KMG_ALPHABET="ACGT", TMPDIR=tmp)
try:
    for mode, opts in (("count", []), ("uniq", []), ("batch", []), ("count", ["-m", "VEC_COUNT"])):
        name = " ".join([mode, *opts])
        out = os.path.join(tmp, "out_" + "_".join([mode, *opts]))
        t0 = time.perf_counter()
        subprocess.run([sys.executable, "-m", "kman_b200.scripts.kmer", mode, *opts, fa, out, str(args.k)], check=True,
                       env=env, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        dt = time.perf_counter() - t0
        files = [os.path.join(out, f) for f in os.listdir(out)] if os.path.isdir(out) else [out]
        sz = sum(os.path.getsize(f) for f in files)
        print(f"kmer {name}: {args.n} bp, k={args.k}: {dt:.2f} s wall (python start + CUDA init + FASTA load + GPU + {sz/1e6:.0f} MB written) "
              f"= {(args.n - args.k + 1)/dt/1e6:.1f} M k-mers/s")
finally:
    shutil.rmtree(tmp)
