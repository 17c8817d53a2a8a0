"""CPU-side tests: the C-ABI library loads and exports every symbol include/kmg.h declares,
host logic (FASTA loader, alphabets, LUT builder, chunk planning) and the N>1 plumbing over
gloo.  No compute call is made here -- there is no GPU and no CPU fallback."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import kmer_oracle as ko

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from kman_b200 import _lib

    lib = _lib.load()
    hdr = open(os.path.join(ROOT, "include", "kmg.h")).read()
    declared = set(re.findall(r"\b(kmg_[a-z0-9_]+)\s*\(", hdr))
    declared.discard("kmg_build_lut's")
    assert len(declared) >= 20
    for name in sorted(declared):
        assert hasattr(lib, name), f"libkmg.so lacks {name} declared in include/kmg.h"
    assert set(_lib.SIGNATURES) == declared, set(_lib.SIGNATURES) ^ declared
    assert lib.kmg_version() == 100


def test_compute_fails_loudly_without_gpu():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from kman_b200 import _lib
    from kman_b200.engine import get_engine

    with pytest.raises(_lib.KmgError):
        get_engine()
    lib = _lib.load()
    ctx = C.c_void_p()
    rc = lib.kmg_ctx_create(0, C.byref(ctx))
    assert rc == _lib.KMG_ERR_CUDA and lib.kmg_last_error()


def test_product_never_imports_the_oracle():
    bad = []
    for dp, _, files in os.walk(os.path.join(ROOT, "kman_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dp, f), errors="replace").read()
                if re.search(r"kmer_oracle|from oracle|import oracle|oracle/", txt):
                    bad.append(os.path.join(dp, f))
    assert not bad, bad


def test_lut_builder_matches_alphabet_tables():
    from kman_b200 import alphabet as ab

    for name in ("IUPAC", "ACGT"):
        for nat in ab.NATYPES:
            lut, comp = ab.lut_tables(name, nat)
            sym, cmp_row = ab.rows(name, nat)
            for c in range(256):
                ch = chr(c).upper()
                if ch in sym and chr(c).isalpha():
                    e = int(lut[c])
                    assert not e & 0x80
                    assert (e >> 2) & 0xF == ab.SYMBOLS16.index(ch)
                    assert bool(e & 0x40) == (sym.index(ch) >= 4)
                    if sym.index(ch) < 4:
                        assert e & 3 == sym.index(ch)
                    assert ab.SYMBOLS16[comp[(e >> 2) & 0xF]] == cmp_row[sym.index(ch)]
                else:
                    assert lut[c] == 0x80, (name, nat, c)
    with pytest.raises(AssertionError):
        ab.rows("XYZ", ab.NATYPES.DNA)


def test_fasta_loader_follows_reference_text_rules(golden, tmp_path):
    from kman_b200 import fasta

    seen = set()
    for c in golden["cases"]:
        if c["name"] in seen:
            continue
        seen.add(c["name"])
        recs = ko.parse_fasta_text(c["fasta_text"])
        fl = fasta.parse_bytes(c["fasta_text"].encode("latin-1"))
        b, st, names = ko.concat_records(recs)
        assert (fl.bases == b).all() and (fl.rec_starts.astype(np.int64) == st).all() and fl.names == names
        for k in (2, 4, 7):
            assert fl.n_windows(k) == sum(max(0, len(s) - k + 1) for _, s in recs)
    # tabs / control characters take the slow path: trailing ones stripped, inner ones kept
    txt = ">a\tb c\nACG\tT \t\nAC GT\x0b\n>e\n>f\nAC\n"
    fl = fasta.parse_bytes(txt.encode())
    recs = ko.parse_fasta_text(txt)
    assert fl.names == ["a\tb", "e", "f"] and [t for t, _ in recs] == fl.titles
    assert bytes(fl.bases) == b"ACG\tTACGT\n\nAC\n"
    # gz and plain files, missing file, empty file
    import gzip

    p = tmp_path / "x.fa"
    p.write_text(">r\nACGT\nAC\n")
    with gzip.open(str(p) + ".gz", "wt") as fh:
        fh.write(">r\nACGT\nAC\n")
    assert bytes(fasta.read_fasta(str(p)).bases) == bytes(fasta.read_fasta(str(p) + ".gz").bases) == b"ACGTAC\n"
    with pytest.raises(AssertionError):
        fasta.read_fasta(str(tmp_path / "missing.fa"))
    (tmp_path / "empty.fa").write_text("no header here\n")
    with pytest.raises(AssertionError):
        fasta.read_fasta(str(tmp_path / "empty.fa"))


def test_chunking_is_the_reference_batcher_rule():
    """dist.chunk_* against Sequence.batcher's known answer (tests/test_seq.py:136-138)."""
    from kman_b200.dist import chunk_bases, chunk_windows, sort_bits_after_partition

    seq = "ACGATCGATCG"
    # reference: batcher(seq, k=3, size=5) -> chunks starting 0, 3, 6 of 5 bases = 3 windows each
    got = chunk_bases(len(seq), 3, 3)
    assert [seq[b:e] for b, e in got] == [c for c, _ in ko.batcher_py(seq, 3, 5)]
    assert [b for b, _ in got] == [o for _, o in ko.batcher_py(seq, 3, 5)]
    for n, k, w in ((1000, 31, 8), (17, 5, 4), (3, 5, 2), (100, 2, 7)):
        wins = chunk_windows(n, k, w)
        assert wins[0][0] == 0 and wins[-1][1] == max(0, n - k + 1)
        assert all(a[1] == b[0] for a, b in zip(wins, wins[1:]))
        for (wb, we), (bb, be) in zip(wins, chunk_bases(n, k, w)):
            assert bb == wb and (be == we + k - 1 if we > wb else be == bb)
    assert sort_bits_after_partition(62, 8) == 59 and sort_bits_after_partition(62, 1) == 62
    assert sort_bits_after_partition(62, 3) == 62


_WORKER = r'''
import os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, "oracle"))
import kmer_oracle as ko
from kman_b200.dist import chunk_bases, exchange, part_of_keys, sort_bits_after_partition
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo")
k = 13
seq = ko.synth_bases(20000, 3).decode()
seq = seq[:12000] + seq[:8000]          # duplicates -> counts > 1
b, e = chunk_bases(len(seq), k, world)[rank]
# stand-in for the device kernels (tests only): oracle extraction of this rank's chunk
ex = ko.extract_np([("chr", seq[b:e])], k, False, "ACGT")
keys = ex["narrow"]["keys"][0]
part = part_of_keys(keys >> np.uint64(2 * k - 16), world).astype(np.int64)
order = np.argsort(part, kind="stable")
send = torch.from_numpy(keys[order].view(np.int64).copy())
counts = np.bincount(part, minlength=world)
recv, rc = exchange(send, counts, 1)
mine = np.sort(recv.numpy().view(np.uint64))
u, c = np.unique(mine, return_counts=True)
out = [None] * world
dist.all_gather_object(out, (u, c))
if rank == 0:
    gu = np.concatenate([x[0] for x in out]); gc = np.concatenate([x[1] for x in out])
    _, cw, det = ko.count_np([("chr", seq)], k, False, "ACGT")
    assert (gu == det["narrow"]["keys"][0]).all() and (gc == det["narrow"]["counts"]).all()
    assert (np.diff(gu.astype(np.int64)) > 0).all()      # rank-order concatenation is globally sorted
    print("DIST_OK", world, gu.size)
dist.destroy_process_group()
'''


@pytest.mark.parametrize("world", [2, 3])
def test_exchange_plumbing_over_gloo(world, tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT))
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    p = subprocess.run(
        [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr",
         "127.0.0.1", "--master-port", str(29500 + world + os.getpid() % 1000), str(script)],
        capture_output=True, text=True, timeout=300, env=env)
    assert p.returncode == 0 and "DIST_OK" in p.stdout, p.stdout[-2000:] + p.stderr[-3000:]


def test_bench_reference_arm_contract():
    sys.path.insert(0, ROOT)
    import bench

    rate, sec, threads, steps = bench.cpu_port_rate(200_000, 2, 0)
    assert rate > 0 and sec > 0 and steps == 2
    assert threads == len(os.sched_getaffinity(0))  # every host thread the process may use
    # the time budget cuts a long run short and says so
    assert bench.cpu_port_rate(200_000, 5, 0, budget_s=0.0)[3] == 1


@pytest.mark.parametrize("gpus", [1, 4])
def test_bench_reference_arm_prints_the_contract_line(gpus):
    """`bench.py --impl reference` (the driver's reference arm): one JSON line on stdout with the arm's own
    metric / unit / config, `impl`, `cpu_baseline` (kind, cores, sample) and an `e2e` that repeats the value."""
    import json
    import subprocess

    env = dict(os.environ, KMG_BENCH_REF_BASES="300000", RANK="0", WORLD_SIZE=str(gpus))
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", str(gpus), "--steps", "2",
                        "--warmup", "1"], capture_output=True, text=True, timeout=300, env=env)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, p.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "k-mers/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("k-mers/sec") and d["n_gpus"] == gpus and d["steps"] == 2 and d["warmup"] == 1
    assert d["value"] > 0 and d["e2e"] == {"value": d["value"], "unit": "k-mers/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] == len(os.sched_getaffinity(0)) and cb["value"] == d["value"] and cb["sample"]
    assert ("config 2" if gpus == 1 else "config 3") in d["config"]["workload"]
    # the other ranks of a torchrun launch exit 0 without work
    env["RANK"] = "1"
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", str(gpus)],
                       capture_output=True, text=True, timeout=300, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_bench_rejects_zero_steps_and_a_reference_dump(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=300)
        assert p.returncode == 2 and "error:" in p.stderr, p.stderr[-2000:]


def test_bench_dump_outputs_writes_a_fixed_sample_of_the_table(tmp_path):
    """bench.py --dump-outputs on a host-resident stand-in for a device table: the same seeded rows every
    time, float64 files, k-mer codes recovered exactly from their two halves, at most 64 MB."""
    import types

    import torch

    sys.path.insert(0, ROOT)
    import bench

    for n in (1000, 3 * bench.DUMP_ROWS):
        keys = np.sort(np.random.default_rng(0).integers(0, 1 << 62, n, dtype=np.uint64))
        counts = np.random.default_rng(1).integers(1, 1 << 31, n).astype(np.uint32)
        tab = types.SimpleNamespace(n=n, keys=torch.from_numpy(keys.view(np.uint8).copy()),
                                    counts=torch.from_numpy(counts.view(np.uint8).copy()))
        bench.dump_outputs(str(tmp_path / str(n)), types.SimpleNamespace(device=torch.device("cpu")), tab, 1, 0)
        files = {f[:-4]: tmp_path / str(n) / f for f in os.listdir(tmp_path / str(n))}
        assert set(files) == {"n_rows", "rows", "keys_hi", "keys_lo", "counts"}
        assert sum(os.path.getsize(f) for f in files.values()) <= 64 << 20
        a = {name: np.load(f) for name, f in files.items()}
        assert all(v.dtype == np.float64 for v in a.values()) and a["n_rows"].tolist() == [n]
        rows = a["rows"].astype(np.int64)
        assert rows.size == min(n, bench.DUMP_ROWS) and (np.diff(rows) > 0).all()
        assert np.array_equal(rows, bench.dump_rows(n))
        got = a["keys_hi"].astype(np.uint64) << np.uint64(31) | a["keys_lo"].astype(np.uint64)
        assert np.array_equal(got, keys[rows]) and np.array_equal(a["counts"], counts[rows])


def test_every_option_and_stat_is_documented_in_the_header():
    """kmg_set_option / kmg_get_stat names handled in api.cu must appear in include/kmg.h's
    tuning section (and nothing documented may be unknown to the library)."""
    import re

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    api = open(os.path.join(root, "kman_b200", "csrc", "api.cu")).read()
    hdr = open(os.path.join(root, "include", "kmg.h")).read()
    doc = hdr[hdr.index("tuning / introspection"):]
    set_body = api[api.index('extern "C" int kmg_set_option'):api.index('extern "C" int64_t kmg_get_stat')]
    get_body = api[api.index('extern "C" int64_t kmg_get_stat'):]
    get_body = get_body[: get_body.index("\n}\n")]
    options = set(re.findall(r'strcmp\(name, "([a-z_]+)"\)', set_body))
    stats = set(re.findall(r'strcmp\(name, "([a-z_]+)"\)', get_body))
    assert options and stats
    documented = set(re.findall(r'"([a-z_]+)"', doc))
    assert options <= documented, sorted(options - documented)
    assert stats <= documented, sorted(stats - documented)
    assert documented <= options | stats, sorted(documented - options - stats)
