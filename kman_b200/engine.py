"""Device pipeline: drives libkmg's stage API with torch-owned buffers.

torch is plumbing only (device memory, streams, torch.distributed); every byte of the hot
path is produced by the CUDA kernels behind include/kmg.h.  There is no CPU fallback: the
constructor raises if the shared library or a CUDA device is missing.

Stage -> reference mapping (see DESIGN.md):
  extract()        seq.py:284-328 (+ rc :245-282)           K1+K2
  sort()           batch.py:156-168 + join.py:63-93         K3
  rle_count()      join.py:95-130 + :265-285                K4
  singletons()     join.py:95-130 + :243-263                K4
  format_counts()/format_uniq()  join.py:262,284; seq.py:103-104  K6
  _write_text()    join.py:262,284; batch.py:281-296        K6 in chunks (+ narrow/wide rank merge): the one text
                   writer behind write_count()/write_uniq()/write_batch() and count_text()/uniq_text()
  write_vectors()  join.py:287-335 + abundance.py:104-172      vectors filled pass by pass, trimmed and formatted on
                   the device, gzipped on host threads (abundance() returns the same vectors as host arrays)
  histogram()      `kmer histo`: the spectrum of count()'s count column, summed on the device pass by pass
                   (write_histogram() writes it as text)

Strand rule: every method's `rc` is False / 0 (forward k-mers), True / 1 (`-r`: each k-mer and its reverse
complement, two keys per window) or CANONICAL (`--canonical`: one key per window, the smaller of the k-mer and its
reverse complement; see kmg.h).  Abundance vectors, batch files and the multi-GPU path take 0 / 1 only.
"""
from __future__ import annotations

import ctypes as C
import io
import os
from concurrent.futures import ThreadPoolExecutor
from dataclasses import dataclass, field
from typing import BinaryIO, Callable, Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np
import torch

from kman_b200 import _lib, alphabet as ab
from kman_b200.fasta import FlatInput

CANONICAL = _lib.KMG_CANONICAL  # `rc` of the canonical strand rule


def keys_per_window(rc) -> int:
    """Keys an extraction emits per valid window under the strand rule `rc`: 2 with `-r`, else 1."""
    return 1 if rc == CANONICAL else (2 if rc else 1)


def per_strand(rc) -> None:
    """AssertionError for CANONICAL where the output is defined per strand (vectors, batch files) or the path
    has no canonical keys (the multi-GPU exchange)."""
    if rc == CANONICAL:
        raise AssertionError("canonical k-mers are not available here: use rc = False / True")


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _on_device(fn):
    """Run an Engine method with the engine's GPU current: libkmg launches on the current device
    (kernel attributes, workspaces and streams are per device), and one process may own several
    engines (get_engine(device))."""
    import functools

    @functools.wraps(fn)
    def wrapper(self, *args, **kwargs):
        if torch.cuda.current_device() == self.device.index:
            return fn(self, *args, **kwargs)
        with torch.cuda.device(self.device):
            return fn(self, *args, **kwargs)

    return wrapper


@dataclass
class DeviceInput:
    """Flat base buffer resident in HBM."""

    bases: torch.Tensor  # uint8[n_bases (+pad)]
    n_bases: int
    flat: FlatInput
    alphabet: str
    natype: ab.NATYPES
    lut: torch.Tensor
    comp16: torch.Tensor
    rec_starts: Optional[torch.Tensor] = None  # uint64 as int64 [n_rec+1]
    names_buf: Optional[torch.Tensor] = None
    name_offs: Optional[torch.Tensor] = None
    pos_offset: int = 0  # global position of bases[0] (multi-GPU chunks)

    @property
    def rna(self) -> int:
        return 1 if self.natype == ab.NATYPES.RNA else 0

    @property
    def payload_bytes(self) -> int:
        """Bytes of a (global position << 1 | strand) payload: 4 while every position of the input fits."""
        return 4 if ((self.pos_offset + self.n_bases) << 1) < (1 << 32) else 8


def key_bytes(k: int, wide: bool) -> int:
    """Bytes of one key: narrow 2-bit codes take 8 / 16 bytes, wide 4-bit codes 16 / 32 (k <= 32 / k <= 64)."""
    return (16 if k <= 32 else 32) if wide else (8 if k <= 32 else 16)


def window_range(d: DeviceInput, k: int, win_begin: int = 0, win_end: Optional[int] = None) -> Tuple[int, int]:
    """[win_begin, win_end) clamped to the windows of the input; AssertionError for k <= 1 and ValueError for
    k > 64, the reference's check and this build's limit."""
    if k <= 1:
        raise AssertionError(f"k must be >= 1, got {k} instead.")  # batcher.py:477-478
    if k > 64:
        raise ValueError(f"k={k}: this build supports k <= 64 (no CPU fallback)")
    n_win_total = max(0, d.n_bases - k + 1)
    win_end = n_win_total if win_end is None else min(win_end, n_win_total)
    return min(win_begin, win_end), win_end


@dataclass
class KeyArray:
    """n keys (+ optional payload) in `keys`/`vals`; `keys_alt`/`vals_alt` are same-sized scratch."""

    keys: torch.Tensor  # uint8 bytes
    keys_alt: Optional[torch.Tensor]
    vals: Optional[torch.Tensor]
    vals_alt: Optional[torch.Tensor]
    n: int
    key_bytes: int
    val_bytes: int
    k: int
    wide: bool
    n_other: int = 0  # narrow extraction: windows that belong to the wide stream
    is_sorted: bool = False
    hist: Optional[torch.Tensor] = None  # digit histograms of exactly these keys (from kmg_extract)

    @property
    def key_bits(self) -> int:
        return self.k * (4 if self.wide else 2)

    def keys_host(self) -> np.ndarray:
        raw = self.keys[: self.n * self.key_bytes].cpu().numpy()
        return raw.view(np.uint64) if self.key_bytes == 8 else raw.view(np.uint64).reshape(-1, self.key_bytes // 8)

    def vals_host(self) -> Optional[np.ndarray]:
        if self.vals is None:
            return None
        raw = self.vals[: self.n * self.val_bytes].cpu().numpy()
        return raw.view(np.uint32 if self.val_bytes == 4 else np.uint64)


@dataclass
class CountTable:
    keys: torch.Tensor
    counts: torch.Tensor  # uint32 as bytes
    n: int
    key_bytes: int
    k: int
    wide: bool

    def keys_host(self) -> np.ndarray:
        raw = self.keys[: self.n * self.key_bytes].cpu().numpy()
        return raw.view(np.uint64) if self.key_bytes == 8 else raw.view(np.uint64).reshape(-1, self.key_bytes // 8)

    def counts_host(self) -> np.ndarray:
        return self.counts[: self.n * 4].cpu().numpy().view(np.uint32)


# ---- key-range passes (write_count / write_uniq) ------------------------------------------------------
PASS_PARTS = 256  # parts of a multi-pass plan: the top 8 key bits (first 4 bases)
DEVICE_HEADROOM = 2 << 30  # bytes of free device memory a default budget leaves alone (allocator, context)
TEXT_CHUNK_BYTES = 256 << 20  # device text of one chunk (two of them on the device, two pinned on the host)
VEC_CHUNK_ROWS = 1 << 20  # vector entries per text chunk of write_vectors (at most 11 bytes each)
VEC_GZIP_THREADS = min(16, os.cpu_count() or 1)  # write_vectors: files compressed at once (two chunk buffers each)


def wide_part_table(rna: int, n_parts: int) -> np.ndarray:
    """uint8[65536]: part of a wide-stream key from its top 16 bits (first 4 symbols), see
    kmg_wide_part_table in include/kmg.h.  Host only."""
    t = np.zeros(65536, np.uint8)
    _lib.check(_lib.load().kmg_wide_part_table(int(rna), int(n_parts), t.ctypes.data_as(_lib.u8p)))
    return t


def plan_parts(narrow: Sequence[int], wide: Sequence[int], pass_bytes: Callable[[int, int], int],
               budget: int) -> List[Tuple[int, int]]:
    """Group contiguous parts [lo, hi) greedily into passes whose pass_bytes(narrow keys, wide keys) stays
    within `budget` (pass_bytes grows with both, so greedy gives the fewest passes).  ValueError if one
    part alone does not fit."""
    out: List[Tuple[int, int]] = []
    lo, n_parts = 0, len(narrow)
    while lo < n_parts:
        need = pass_bytes(int(narrow[lo]), int(wide[lo]))
        if need > budget:
            raise ValueError(f"part {lo} of {n_parts} needs {need} device bytes, more than the {budget} available")
        hi, n, m = lo + 1, int(narrow[lo]), int(wide[lo])
        while hi < n_parts and pass_bytes(n + int(narrow[hi]), m + int(wide[hi])) <= budget:
            n, m = n + int(narrow[hi]), m + int(wide[hi])
            hi += 1
        out.append((lo, hi))
        lo = hi
    return out


COUNT_MAX = 2**32 - 1  # the largest count a table holds (uint32)


def count_range(min_count: int = 1, max_count: Optional[int] = None) -> Optional[Tuple[int, int]]:
    """(min_count, max_count) of a count restricted to min_count <= count <= max_count (max_count None: no upper
    limit), or None for the full range [1, 2^32-1]: the plain count table.  A bad range raises AssertionError."""
    hi = COUNT_MAX if max_count is None else int(max_count)
    lo = int(min_count)
    assert 1 <= lo <= hi <= COUNT_MAX, f"bad count range: need 1 <= min_count <= max_count <= {COUNT_MAX}, got [{lo}, {hi}]"
    return None if (lo, hi) == (1, COUNT_MAX) else (lo, hi)


def pass_bytes(k: int, mode: str, n: int, m: int, val_bytes: int, text_bytes: int, n_win: int) -> int:
    """Device bytes of one pass over n narrow and m wide keys: key (+ payload) buffers and their alternates,
    counts, the sort workspace from the library's own *_workspace_bytes (one buffer the engine keeps and
    grows, so the wide stage sees the larger of the two), the merge ranks, the extraction workspace and the
    text chunk buffers (`text_bytes`).

    mode "vec" (abundance vectors): keys + payload and their alternates and the stable payload sort's workspace
    per stream.  The narrow buffers are freed before the wide stream is extracted, so a pass costs the larger
    stage, not their sum, and there is no merge term; the text stage comes after the passes, with only the
    (kept) sort workspaces beside it.

    mode "histo" (multiplicity spectrum): keys and their alternates and kmg_sort_histo's workspace per stream
    (32-byte wide keys: kmg_sort256 + kmg_rle_count and the counts), the larger stage as in "vec"; no counts,
    merge ranks or text.  The histogram arrays themselves (a few MB) are not counted.

    A count restricted to a multiplicity range (write_count(min_count=, max_count=)) takes the "count" plan:
    its tables, counts and workspaces (kmg_sort_count_range, kmg_filter_counts in place) are never larger than
    the unfiltered ones, so the count plan is an upper bound for it."""
    lib = _lib.load()
    kb, kw = key_bytes(k, False), key_bytes(k, True)
    if mode == "histo":
        ws_n = lib.kmg_sort_histo_workspace_bytes(n, kb, 2 * k)
        if kw == 32:
            ws = ws_n + lib.kmg_sort256_workspace_bytes(m) + lib.kmg_rle_workspace_bytes(m) + 4 * m
        else:
            ws = max(ws_n, lib.kmg_sort_histo_workspace_bytes(m, kw, 4 * k))
        return int(max(2 * n * kb + ws_n, 2 * m * kw + ws) + lib.kmg_extract_workspace_bytes(n_win))
    if mode == "vec":
        ws_n = lib.kmg_radix_sort_workspace_bytes(n, kb, val_bytes, 0, 2 * k)
        if kw == 32:  # kmg_sort256 has a workspace of its own, next to the narrow sort's
            ws = ws_n + lib.kmg_sort256_workspace_bytes(m)
        else:
            ws = max(ws_n, lib.kmg_radix_sort_workspace_bytes(m, kw, val_bytes, 0, 4 * k))
        stages = max(2 * n * (kb + val_bytes) + ws_n, 2 * m * (kw + val_bytes) + ws, ws + text_bytes)
        return int(stages + lib.kmg_extract_workspace_bytes(n_win))
    item = 4 if mode == "count" else val_bytes  # count / payload bytes per key
    if mode == "count":
        ws_n = lib.kmg_sort_count_workspace_bytes(n, kb, 2 * k)
        ws_w = lib.kmg_sort_count_workspace_bytes(m, kw, 4 * k)
    else:
        ws_n = lib.kmg_sort_uniq_workspace_bytes(n, kb, val_bytes, 2 * k)
        ws_w = lib.kmg_sort_uniq_workspace_bytes(m, kw, val_bytes, 4 * k)
    if kw == 32:
        ws_w = lib.kmg_sort256_workspace_bytes(m) + lib.kmg_rle_workspace_bytes(m)
    stages = 2 * n * (kb + item) + ws_n
    if m:  # the narrow table is held while the wide stream is extracted, sorted and ranked against it
        merge = 8 * (n + m) + (16 * m if k > 32 else 0)
        stages = max(stages, n * (kb + item) + 2 * m * (kw + item) + max(ws_n, ws_w) + merge)
    return int(stages + lib.kmg_extract_workspace_bytes(n_win) + text_bytes)


@dataclass
class PassPlan:
    """How write_count / write_uniq / write_vectors split the key space.  n_parts == 1: one pass on the
    whole-input path (count() / uniq() / unfiltered extraction); otherwise parts[i] = (lo, hi) of pass i over
    `n_parts` parts with `narrow[p]` / `wide[p]` keys in part p, and pass_bytes[i] its modelled device bytes.
    pass_ms[i]: time of pass i between CUDA events (filled in by the writers).  text_ms: write_vectors' text
    stage (device formatting and copies, waits for a free chunk buffer included)."""

    n_parts: int
    parts: List[Tuple[int, int]]
    narrow: np.ndarray
    wide: np.ndarray
    pass_bytes: List[int] = field(default_factory=list)
    pass_ms: List[float] = field(default_factory=list)
    text_ms: float = 0.0

    @property
    def n_passes(self) -> int:
        return len(self.parts)


def make_plan(k: int, budget: int, one_pass_bytes: int, totals: Tuple[int, int],
              part_counts: Callable[[], Tuple[np.ndarray, np.ndarray]], cost: Callable[[int, int], int]) -> PassPlan:
    """One pass when the whole-input path fits `budget` (or there is nothing to do); otherwise group the
    parts of part_counts() (narrow, wide keys per part) into passes by `cost` (plan_parts).  Key-range
    passes need the per-part counts of the 4-mer histogram, so k < 12 that does not fit is a ValueError."""
    n, m = totals
    if one_pass_bytes <= budget or n + m == 0:
        return PassPlan(1, [(0, 1)], np.array([n], np.int64), np.array([m], np.int64), [one_pass_bytes])
    if k < 12:
        raise ValueError(f"k={k}: the input needs {one_pass_bytes} device bytes, more than the {budget} available, "
                         f"and key-range passes need k >= 12")
    narrow, wide = part_counts()
    parts = plan_parts(narrow, wide, cost, budget)
    return PassPlan(len(narrow), parts, narrow, wide,
                    [cost(int(narrow[lo:hi].sum()), int(wide[lo:hi].sum())) for lo, hi in parts])


class _ChunkSink:
    """Device text -> pinned host buffer -> file through `slots` buffer pairs: the copy of a chunk runs on a
    copy stream and its file write on one of `workers` threads while the GPU formats the next chunks.  Every
    submit names its file (default `fh`); writes to one file keep their submission order, writes to different
    files run in parallel.  With the defaults (two slots, one worker, one file) this is plain double buffering."""

    def __init__(self, eng: "Engine", fh: Optional[BinaryIO], nbytes: int, slots: int = 2, workers: int = 1):
        self.fh = fh
        self.dev = [eng._new(nbytes) for _ in range(slots)]
        self.pinned = [torch.empty(max(nbytes, 16), dtype=torch.uint8, pin_memory=True) for _ in range(slots)]
        self.stream = torch.cuda.Stream(eng.device)
        self.pool = ThreadPoolExecutor(workers)
        self.pending = [None] * slots
        self.last: dict = {}  # file -> future of the latest task submitted for it
        self.slot = 0

    def buffer(self) -> torch.Tensor:
        """Device buffer of the next chunk (free once the write of the chunk `slots` submits back is done)."""
        s = self.slot
        if self.pending[s] is not None:
            self.pending[s].result()
            self.pending[s] = None
        return self.dev[s]

    def submit(self, text: torch.Tensor, pieces: Optional[List[Tuple[Optional[np.ndarray], int, int]]],
               fh: Optional[BinaryIO] = None) -> None:
        """Write `text` (a prefix of buffer()) to `fh`; pieces: (None, a, b) = text[a:b], (arr, a, b) = arr[a:b]
        in this order, or None for the whole text."""
        fh = self.fh if fh is None else fh
        s, nb = self.slot, int(text.numel())
        ready = torch.cuda.Event()
        ready.record()
        self.stream.wait_event(ready)
        done = torch.cuda.Event()
        with torch.cuda.stream(self.stream):
            if nb:
                self.pinned[s][:nb].copy_(text, non_blocking=True)
            done.record()
        host = self.pinned[s].numpy()
        # FIFO workers: the task a write waits for was taken up before it, so the wait always ends
        self.pending[s] = self.last[fh] = self.pool.submit(self._write, self.last.get(fh), done, host, nb, pieces, fh)
        self.slot = (s + 1) % len(self.dev)

    def then(self, fh: BinaryIO, fn: Callable[[], None]) -> None:
        """Run fn() on a worker once every write to `fh` submitted so far is done (e.g. close the file)."""
        self.last[fh] = self.pool.submit(self._after, self.last.get(fh), fn)

    @staticmethod
    def _after(prev, fn) -> None:
        if prev is not None:
            prev.result()
        fn()

    def _write(self, prev, done, host: np.ndarray, nb: int, pieces, fh: BinaryIO) -> None:
        if prev is not None:
            prev.result()
        done.synchronize()
        if pieces is None:
            fh.write(memoryview(host[:nb]))
            return
        for arr, a, b in pieces:
            if b > a:
                fh.write(memoryview((host if arr is None else arr)[a:b]))

    def close(self) -> None:
        try:
            for f in [*self.pending, *self.last.values()]:
                if f is not None:
                    f.result()
        finally:
            self.pool.shutdown(wait=True)
            self.stream.synchronize()


class Engine:
    """One engine per (process, GPU)."""

    def __init__(self, device: Optional[int] = None):
        self.lib = _lib.load()  # ImportError if libkmg.so is missing
        if not torch.cuda.is_available():
            raise _lib.KmgError("no CUDA device visible: kman_b200 has no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else device)
        self._scratch: Dict[str, torch.Tensor] = {}
        self._small = torch.zeros(8, dtype=torch.int64, device=self.device)
        self._luts: Dict[Tuple[str, ab.NATYPES], Tuple[torch.Tensor, torch.Tensor]] = {}

    # ---- plumbing ---------------------------------------------------------------------------
    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def _buf(self, name: str, nbytes: int) -> torch.Tensor:
        """Named scratch buffer, grown geometrically and reused across calls."""
        t = self._scratch.get(name)
        if t is None or t.numel() < nbytes:
            self._scratch.pop(name, None)
            t = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=self.device)
            self._scratch[name] = t
        return t

    def _new(self, nbytes: int) -> torch.Tensor:
        return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=self.device)

    def _out(self, reuse: Optional[str], name: str, nbytes: int) -> torch.Tensor:
        """Output buffer: the engine scratch `reuse + name` when `reuse` is given (the benchmark loop), else fresh."""
        return self._buf(reuse + name, nbytes) if reuse else self._new(nbytes)

    def _status(self, ws: torch.Tensor) -> None:
        _lib.check(self.lib.kmg_ws_status(ws.data_ptr(), self._stream()))

    def lut_tensors(self, alphabet: str, natype: ab.NATYPES) -> Tuple[torch.Tensor, torch.Tensor]:
        key = (alphabet, natype)
        if key not in self._luts:
            lut, c16 = ab.lut_tables(alphabet, natype)
            self._luts[key] = (
                torch.from_numpy(lut.copy()).to(self.device),
                torch.from_numpy(c16.copy()).to(self.device),
            )
        return self._luts[key]

    # ---- upload -----------------------------------------------------------------------------
    @_on_device
    def upload(self, flat: FlatInput, alphabet: Optional[str] = None, natype: ab.NATYPES = ab.NATYPES.DNA,
               with_names: bool = True) -> DeviceInput:
        alphabet = alphabet or ab.default_alphabet()
        lut, c16 = self.lut_tensors(alphabet, natype)
        n = int(flat.bases.shape[0])
        bases = torch.empty(((n + 15) // 16 + 1) * 16, dtype=torch.uint8, device=self.device)
        if n:
            src = flat.bases if flat.bases.flags.writeable and flat.bases.flags.c_contiguous else np.array(flat.bases)
            bases[:n].copy_(torch.from_numpy(src), non_blocking=False)
        d = DeviceInput(bases, n, flat, alphabet, natype, lut, c16)
        if with_names:
            self._upload_names(d)
        return d

    @_on_device
    def load_fasta(self, path: str, alphabet: Optional[str] = None, natype: ab.NATYPES = ab.NATYPES.DNA,
                   with_names: bool = True) -> DeviceInput:
        """Read a FASTA file and flatten it ON THE GPU (kmg_fasta_flatten): the raw bytes go to
        the device once, line structure / header lines / blanks are resolved by three kernels.
        Files with TAB / VT / FF / control separators or non-ASCII bytes take the host loader,
        which implements the reference's rstrip() rule for them."""
        import gzip
        import os

        from kman_b200 import fasta

        if not os.path.isfile(path):
            raise AssertionError(f"input file not found: {path}")  # batcher.py:475-476
        opener = gzip.open if path.endswith(".gz") else open
        with opener(path, "rb") as fh:
            raw = fh.read()
        if len(raw) == 0:
            raise AssertionError("premature end of file or empty file")
        n_raw = len(raw)
        d_raw = torch.empty(((n_raw + 15) // 16 + 1) * 16, dtype=torch.uint8, device=self.device)
        import warnings

        with warnings.catch_warnings():  # (a read-only view of the bytes object: no second host copy)
            warnings.simplefilter("ignore", UserWarning)
            d_raw[:n_raw].copy_(torch.from_numpy(np.frombuffer(raw, np.uint8)))
        bases = torch.empty(((n_raw + 15) // 16 + 2) * 16, dtype=torch.uint8, device=self.device)
        max_rec = 1 << 16
        while True:
            rec_starts = torch.zeros(max_rec + 1, dtype=torch.int64, device=self.device)
            hdr_begin = torch.zeros(max_rec, dtype=torch.int64, device=self.device)
            ws_bytes = self.lib.kmg_fasta_workspace_bytes(n_raw)
            ws = self._buf("ws_fasta", ws_bytes)
            _lib.check(self.lib.kmg_fasta_flatten(d_raw.data_ptr(), n_raw, bases.data_ptr(), rec_starts.data_ptr(),
                                                  hdr_begin.data_ptr(), max_rec, self._small[5:].data_ptr(),
                                                  ws.data_ptr(), ws_bytes, self._stream()))
            n_out, n_rec, special = (int(x) for x in self._small[5:8].cpu().numpy().view(np.uint64))
            if special:
                return self.upload(fasta.parse_bytes(raw), alphabet, natype, with_names)
            if n_rec <= max_rec:
                break
            max_rec = n_rec
        if n_rec == 0:
            raise AssertionError("premature end of file or empty file")  # parsers.py:100-102
        hb = hdr_begin[:n_rec].cpu().numpy()
        titles = []
        for b in hb:
            b = int(b)
            e1, e2 = raw.find(b"\n", b), raw.find(b"\r", b)
            e = min(x for x in (e1, e2, n_raw) if x >= 0)
            titles.append(raw[b:e].decode("latin-1").rstrip())
        names = [t.split(" ")[0] for t in titles]
        flat = FlatInput(bases[:n_out].cpu().numpy(), rec_starts[: n_rec + 1].cpu().numpy().astype(np.uint64), names, titles)
        alphabet = alphabet or ab.default_alphabet()
        lut, c16 = self.lut_tensors(alphabet, natype)
        d = DeviceInput(bases, n_out, flat, alphabet, natype, lut, c16)
        if with_names:
            self._upload_names(d)
        return d

    def _upload_names(self, d: DeviceInput) -> None:
        flat = d.flat
        d.rec_starts = torch.from_numpy(flat.rec_starts.astype(np.int64)).to(self.device)
        nb = [nm.encode("latin-1") for nm in flat.names]
        offs = np.zeros(len(nb) + 1, np.int64)
        offs[1:] = np.cumsum([len(b) for b in nb])
        d.name_offs = torch.from_numpy(offs).to(self.device)
        d.names_buf = torch.from_numpy(np.frombuffer(b"".join(nb) + b"\0", np.uint8).copy()).to(self.device)

    @_on_device
    def count_windows(self, d: DeviceInput, k: int, rc: bool = False) -> Tuple[int, int]:
        """(narrow keys, wide-stream windows) of an input WITHOUT building a key: for k >= 12 the 4-mer
        histogram pre-pass of the bases knows both (kmg_extract_dest_counts with one destination);
        smaller k runs the extraction."""
        n_win = max(0, d.n_bases - k + 1)
        if n_win == 0:
            return 0, 0
        if k < 12:
            a = self.extract(d, k, rc, wide=False, val_bytes=0)
            return a.n, a.n_other
        counts = torch.zeros(2, dtype=torch.int64, device=self.device)
        ws_bytes = self.lib.kmg_dest_counts_workspace_bytes()
        ws = self._buf("ws_dest_counts", ws_bytes)
        _lib.check(self.lib.kmg_extract_dest_counts(d.bases.data_ptr(), d.n_bases, 0, n_win, k, int(rc), d.lut.data_ptr(), 1,
                                                    counts.data_ptr(), ws.data_ptr(), ws_bytes, self._stream()))
        n, n_other = (int(x) for x in counts.cpu())
        return n, n_other

    # ---- K1+K2 ------------------------------------------------------------------------------
    @_on_device
    def extract(self, d: DeviceInput, k: int, rc: bool = False, wide: bool = False, val_bytes: int = 0,
                win_begin: int = 0, win_end: Optional[int] = None, reuse: Optional[str] = None,
                want_hist: bool = False) -> KeyArray:
        """Keys (and payload) of the windows starting in [win_begin, win_end), emission order.

        `reuse`: name prefix of engine-owned scratch buffers to place the output in (the
        benchmark loop) instead of fresh allocations."""
        win_begin, win_end = window_range(d, k, win_begin, win_end)
        n_win = win_end - win_begin
        kb = key_bytes(k, wide)
        cap = max(n_win * keys_per_window(rc), 1)
        keys = self._out(reuse, "keys", cap * kb)
        keys_alt = self._out(reuse, "keys_alt", cap * kb)
        vals = self._out(reuse, "vals", cap * val_bytes) if val_bytes else None
        vals_alt = self._out(reuse, "vals_alt", cap * val_bytes) if val_bytes else None
        ws_bytes = self.lib.kmg_extract_workspace_bytes(n_win)
        ws = self._buf("ws_extract", ws_bytes)
        # fused digit histograms for the sort that follows (narrow stream only; they describe window offsets, not
        # canonical keys)
        hist = self._out(reuse, "hist", 16 * 256 * 8) if want_hist and not wide and k >= 4 and rc != CANONICAL else None
        _lib.check(
            self.lib.kmg_extract(
                d.bases.data_ptr(), d.n_bases, win_begin, win_end, k, int(rc), int(wide), d.lut.data_ptr(),
                d.comp16.data_ptr(), keys.data_ptr(), kb, _ptr(vals), val_bytes, d.pos_offset,
                self._small.data_ptr(), _ptr(hist), ws.data_ptr(), ws_bytes, self._stream(),
            )
        )
        self._status(ws)
        cnt = self._small[:2].cpu().numpy().view(np.uint64)
        return KeyArray(keys, keys_alt, vals, vals_alt, int(cnt[0]), kb, val_bytes, k, wide, n_other=int(cnt[1]),
                        hist=hist)

    # ---- K3 -----------------------------------------------------------------------------------
    @_on_device
    def sort(self, a: KeyArray, begin_bit: int = 0, end_bit: Optional[int] = None) -> KeyArray:
        end_bit = a.key_bits if end_bit is None else end_bit
        if a.key_bytes == 32:
            return self._sort256(a, end_bit)
        if a.n > 1 and end_bit > begin_bit:
            ws_bytes = self.lib.kmg_radix_sort_workspace_bytes(a.n, a.key_bytes, a.val_bytes, begin_bit, end_bit)
            ws = self._buf("ws_sort", ws_bytes)
            sel = C.c_int(0)
            hist = a.hist if (begin_bit == 0 and end_bit == a.key_bits) else None
            _lib.check(
                self.lib.kmg_radix_sort(
                    a.keys.data_ptr(), a.keys_alt.data_ptr(), _ptr(a.vals), _ptr(a.vals_alt), a.n, a.key_bytes,
                    a.val_bytes, begin_bit, end_bit, _ptr(hist), C.byref(sel), ws.data_ptr(), ws_bytes, self._stream(),
                )
            )
            a.hist = None
            self._last_sort_ws = ws
            if sel.value:
                a.keys, a.keys_alt = a.keys_alt, a.keys
                a.vals, a.vals_alt = a.vals_alt, a.vals
        a.is_sorted = True
        return a

    def _sort256(self, a: KeyArray, end_bit: int) -> KeyArray:
        """256-bit keys (wide stream, 33 <= k <= 64): kmg_sort256 sorts out of place into the alt buffers."""
        if a.n > 1 and end_bit > 0:
            ws_bytes = self.lib.kmg_sort256_workspace_bytes(a.n)
            ws = self._buf("ws_sort256", ws_bytes)
            _lib.check(self.lib.kmg_sort256(a.keys.data_ptr(), a.keys_alt.data_ptr(), _ptr(a.vals), _ptr(a.vals_alt), a.n,
                                            a.val_bytes, end_bit, ws.data_ptr(), ws_bytes, self._stream()))
            a.keys, a.keys_alt = a.keys_alt, a.keys
            a.vals, a.vals_alt = a.vals_alt, a.vals
        a.is_sorted = True
        return a

    @_on_device
    def sort_count(self, a: KeyArray, end_bit: Optional[int] = None, reuse: Optional[str] = None, min_count: int = 1,
                   max_count: Optional[int] = None) -> CountTable:
        """sort() + rle_count() in one native call (kmg_sort_count): when the hybrid finish applies,
        its local sort emits the (k-mer, count) table directly.  Consumes `a` (both key buffers).
        min_count / max_count: keep only the rows with min_count <= count <= max_count (kmg_sort_count_range;
        32-byte keys: kmg_filter_counts on the table)."""
        end_bit = a.key_bits if end_bit is None else end_bit
        assert a.val_bytes == 0
        rng = count_range(min_count, max_count)
        if a.key_bytes == 32:
            t = self.rle_count(self.sort(a, 0, end_bit), reuse=reuse)
            return t if rng is None else self.filter_counts(t, *rng)
        counts = self._out(reuse, "counts", a.n * 4)
        if a.n == 0:
            return CountTable(a.keys_alt, counts, 0, a.key_bytes, a.k, a.wide)
        ws_bytes = self.lib.kmg_sort_count_workspace_bytes(a.n, a.key_bytes, end_bit)
        ws = self._buf("ws_sort", ws_bytes)
        sel = C.c_int(0)
        hist = a.hist if end_bit == a.key_bits else None
        if rng is None:
            _lib.check(
                self.lib.kmg_sort_count(a.keys.data_ptr(), a.keys_alt.data_ptr(), a.n, a.key_bytes, end_bit, _ptr(hist),
                                        counts.data_ptr(), self._small[2:].data_ptr(), C.byref(sel), ws.data_ptr(),
                                        ws_bytes, self._stream())
            )
        else:
            _lib.check(
                self.lib.kmg_sort_count_range(a.keys.data_ptr(), a.keys_alt.data_ptr(), a.n, a.key_bytes, end_bit,
                                              _ptr(hist), rng[0], rng[1], counts.data_ptr(), self._small[2:].data_ptr(),
                                              C.byref(sel), ws.data_ptr(), ws_bytes, self._stream())
            )
        a.hist = None
        self._last_sort_ws = ws
        n_out = self._sort_result_rows(ws)
        return CountTable(a.keys_alt if sel.value else a.keys, counts, n_out, a.key_bytes, a.k, a.wide)

    def _sort_result_rows(self, ws: torch.Tensor) -> int:
        """Rows of the table kmg_sort_count / kmg_sort_uniq just produced.  When the hybrid finish ran,
        the call already synchronised and read the count and the status word back together
        (kmg_get_stat "n_out" / "ws_err"): no second round trip."""
        n_out, err = int(self.lib.kmg_get_stat(b"n_out")), int(self.lib.kmg_get_stat(b"ws_err"))
        if n_out >= 0 and err == 0:
            return n_out
        self._status(ws)
        return int(self._small[2:3].cpu().numpy().view(np.uint64)[0])

    # ---- K4 -----------------------------------------------------------------------------------
    @_on_device
    def rle_count(self, a: KeyArray, reuse: Optional[str] = None) -> CountTable:
        """Distinct keys + counts.  The distinct keys are written into `a.keys_alt`."""
        assert a.is_sorted
        counts = self._out(reuse, "counts", a.n * 4)
        if a.n == 0:
            return CountTable(a.keys_alt, counts, 0, a.key_bytes, a.k, a.wide)
        ws_bytes = self.lib.kmg_rle_workspace_bytes(a.n)
        ws = self._buf("ws_rle", ws_bytes)
        _lib.check(
            self.lib.kmg_rle_count(a.keys.data_ptr(), a.n, a.key_bytes, a.keys_alt.data_ptr(), counts.data_ptr(),
                                   self._small[2:].data_ptr(), ws.data_ptr(), ws_bytes, self._stream())
        )
        self._status(ws)
        n_out = int(self._small[2:3].cpu().numpy().view(np.uint64)[0])
        return CountTable(a.keys_alt, counts, n_out, a.key_bytes, a.k, a.wide)

    @_on_device
    def filter_counts(self, t: CountTable, min_count: int, max_count: int) -> CountTable:
        """The rows of `t` with min_count <= count <= max_count, in order, compacted in place (kmg_filter_counts)."""
        if t.n == 0:
            return t
        ws_bytes = self.lib.kmg_rle_workspace_bytes(t.n)
        ws = self._buf("ws_rle", ws_bytes)
        _lib.check(
            self.lib.kmg_filter_counts(t.keys.data_ptr(), t.counts.data_ptr(), t.n, t.key_bytes, min_count, max_count,
                                       t.keys.data_ptr(), t.counts.data_ptr(), self._small[2:].data_ptr(), ws.data_ptr(),
                                       ws_bytes, self._stream())
        )
        self._status(ws)
        n_out = int(self._small[2:3].cpu().numpy().view(np.uint64)[0])
        return CountTable(t.keys, t.counts, n_out, t.key_bytes, t.k, t.wide)

    @_on_device
    def sort_uniq(self, a: KeyArray, end_bit: Optional[int] = None) -> KeyArray:
        """sort() + singletons() in one native call (kmg_sort_uniq).  Repeated keys are dropped, so
        their order is irrelevant and the keys take the hybrid finish with the payload.  Consumes `a`."""
        end_bit = a.key_bits if end_bit is None else end_bit
        assert a.val_bytes in (4, 8)
        if a.key_bytes == 32:
            return self.singletons(self.sort(a, 0, end_bit))
        if a.n == 0:
            return KeyArray(a.keys_alt, None, a.vals_alt, None, 0, a.key_bytes, a.val_bytes, a.k, a.wide, is_sorted=True)
        ws_bytes = self.lib.kmg_sort_uniq_workspace_bytes(a.n, a.key_bytes, a.val_bytes, end_bit)
        ws = self._buf("ws_sort", ws_bytes)
        sel = C.c_int(0)
        hist = a.hist if end_bit == a.key_bits else None
        _lib.check(
            self.lib.kmg_sort_uniq(a.keys.data_ptr(), a.keys_alt.data_ptr(), a.vals.data_ptr(), a.vals_alt.data_ptr(), a.n,
                                   a.key_bytes, a.val_bytes, end_bit, _ptr(hist), self._small[2:].data_ptr(), C.byref(sel),
                                   ws.data_ptr(), ws_bytes, self._stream())
        )
        a.hist = None
        self._last_sort_ws = ws
        n_out = self._sort_result_rows(ws)
        k_, v_ = (a.keys_alt, a.vals_alt) if sel.value else (a.keys, a.vals)
        return KeyArray(k_, None, v_, None, n_out, a.key_bytes, a.val_bytes, a.k, a.wide, is_sorted=True)

    @_on_device
    def singletons(self, a: KeyArray) -> KeyArray:
        """Keys (+payload) that occur exactly once, ascending (written into the alt buffers)."""
        assert a.is_sorted
        if a.n == 0:
            return KeyArray(a.keys_alt, None, a.vals_alt, None, 0, a.key_bytes, a.val_bytes, a.k, a.wide, is_sorted=True)
        ws_bytes = self.lib.kmg_rle_workspace_bytes(a.n)
        ws = self._buf("ws_rle", ws_bytes)
        _lib.check(
            self.lib.kmg_select_singletons(a.keys.data_ptr(), _ptr(a.vals), a.n, a.key_bytes, a.val_bytes,
                                           a.keys_alt.data_ptr(), _ptr(a.vals_alt), self._small[2:].data_ptr(),
                                           ws.data_ptr(), ws_bytes, self._stream())
        )
        self._status(ws)
        n_out = int(self._small[2:3].cpu().numpy().view(np.uint64)[0])
        return KeyArray(a.keys_alt, None, a.vals_alt, None, n_out, a.key_bytes, a.val_bytes, a.k, a.wide, is_sorted=True)

    # ---- K5 -----------------------------------------------------------------------------------
    @_on_device
    def range_partition(self, a: KeyArray, n_parts: int) -> Tuple[KeyArray, np.ndarray]:
        """Stable split by the top key bits into n_parts regions (into the alt buffers)."""
        ws_bytes = self.lib.kmg_partition_workspace_bytes(max(a.n, 1), a.key_bytes, a.val_bytes)
        ws = self._buf("ws_sort", ws_bytes)
        pc = torch.zeros(n_parts, dtype=torch.int64, device=self.device)
        _lib.check(
            self.lib.kmg_range_partition(a.keys.data_ptr(), _ptr(a.vals), a.n, a.key_bytes, a.val_bytes, a.key_bits,
                                         n_parts, a.keys_alt.data_ptr(), _ptr(a.vals_alt), pc.data_ptr(),
                                         ws.data_ptr(), ws_bytes, self._stream())
        )
        if a.n:
            self._status(ws)
        a.keys, a.keys_alt = a.keys_alt, a.keys
        a.vals, a.vals_alt = a.vals_alt, a.vals
        return a, pc.cpu().numpy().astype(np.int64)

    # ---- K6 -----------------------------------------------------------------------------------
    @_on_device
    def format_counts(self, t: CountTable, rna: int = 0, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Device text "SEQ\\tCOUNT\\n" for one stream (uint8 tensor, exact length).  `out`: a buffer of at
        least t.n * (t.k + 12) bytes to write it into."""
        if t.n == 0:
            return torch.empty(0, dtype=torch.uint8, device=self.device)
        text = self._new(t.n * (t.k + 12)) if out is None else out
        ws_bytes = self.lib.kmg_format_workspace_bytes(t.n)
        ws = self._buf("ws_fmt", ws_bytes)
        _lib.check(
            self.lib.kmg_format_counts(t.keys.data_ptr(), t.counts.data_ptr(), t.n, t.key_bytes, t.k, int(t.wide), rna,
                                       text.data_ptr(), self._small[4:].data_ptr(), ws.data_ptr(), ws_bytes,
                                       self._stream())
        )
        self._status(ws)
        nbytes = int(self._small[4:5].cpu().numpy().view(np.uint64)[0])
        return text[:nbytes]

    @_on_device
    def format_uniq(self, s: KeyArray, d: DeviceInput, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Device text ">NAME:START-END:STRAND\\nSEQ\\n" for one stream.  `out`: a buffer of at least
        s.n * (s.k + 48 + longest name) bytes to write it into."""
        if s.n == 0:
            return torch.empty(0, dtype=torch.uint8, device=self.device)
        if d.rec_starts is None:
            self._upload_names(d)
        max_name = max((len(nm) for nm in d.flat.names), default=0)
        text = self._new(s.n * (s.k + 48 + max_name)) if out is None else out
        ws_bytes = self.lib.kmg_format_workspace_bytes(s.n)
        ws = self._buf("ws_fmt", ws_bytes)
        _lib.check(
            self.lib.kmg_format_uniq(s.keys.data_ptr(), s.vals.data_ptr(), s.n, s.key_bytes, s.val_bytes, s.k,
                                     int(s.wide), d.rna, d.rec_starts.data_ptr(), d.flat.n_rec, d.names_buf.data_ptr(),
                                     d.name_offs.data_ptr(), text.data_ptr(), self._small[4:].data_ptr(),
                                     ws.data_ptr(), ws_bytes, self._stream())
        )
        self._status(ws)
        nbytes = int(self._small[4:5].cpu().numpy().view(np.uint64)[0])
        return text[:nbytes]

    @_on_device
    def merge_ranks(self, narrow_keys: torch.Tensor, n_narrow: int, wide_keys: torch.Tensor, n_wide: int, k: int,
                    rna: int) -> Tuple[torch.Tensor, torch.Tensor]:
        rn = torch.zeros(max(n_narrow, 1), dtype=torch.int64, device=self.device)
        rw = torch.zeros(max(n_wide, 1), dtype=torch.int64, device=self.device)
        if k <= 32:
            _lib.check(
                self.lib.kmg_merge_ranks(narrow_keys.data_ptr(), n_narrow, 8, wide_keys.data_ptr(), n_wide, 16, k, rna,
                                         rn.data_ptr(), rw.data_ptr(), self._stream())
            )
        else:  # 16-byte narrow keys, 32-byte wide keys
            tmp = self._new(max(n_wide, 1) * 16)
            _lib.check(
                self.lib.kmg_merge_ranks_wide(narrow_keys.data_ptr(), n_narrow, wide_keys.data_ptr(), n_wide, k, rna,
                                              rn.data_ptr(), rw.data_ptr(), tmp.data_ptr(), self._stream())
            )
        return rn[:n_narrow], rw[:n_wide]

    # ---- whole path on one GPU ------------------------------------------------------------------
    def sorted_streams(self, d: DeviceInput, k: int, rc: bool, val_bytes: int) -> List[KeyArray]:
        """[narrow] or [narrow, wide]: extracted and sorted key arrays of the input."""
        narrow = self.sort(self.extract(d, k, rc, wide=False, val_bytes=val_bytes, want_hist=True))
        out = [narrow]
        if narrow.n_other:
            out.append(self.sort(self.extract(d, k, rc, wide=True, val_bytes=val_bytes)))
        return out

    def _pipeline_buffers(self, d: DeviceInput, k: int, rc: bool, val_bytes: int, reuse: Optional[str],
                          win_begin: int, win_end: Optional[int]):
        win_begin, win_end = window_range(d, k, win_begin, win_end)
        kb = key_bytes(k, False)
        cap = max((win_end - win_begin) * keys_per_window(rc), 1)
        keys, keys_alt = self._out(reuse, "keys", cap * kb), self._out(reuse, "keys_alt", cap * kb)
        vals = self._out(reuse, "vals", cap * val_bytes) if val_bytes else None
        vals_alt = self._out(reuse, "vals_alt", cap * val_bytes) if val_bytes else None
        ws_bytes = self.lib.kmg_pipeline_workspace_bytes(win_end - win_begin, k, int(rc), val_bytes)
        ws = self._buf("ws_pipeline", ws_bytes)
        return win_begin, win_end, kb, cap, keys, keys_alt, vals, vals_alt, ws, ws_bytes

    @_on_device
    def count_narrow(self, d: DeviceInput, k: int, rc: bool = False, reuse: Optional[str] = None, win_begin: int = 0,
                     win_end: Optional[int] = None, min_count: int = 1,
                     max_count: Optional[int] = None) -> Tuple[CountTable, int]:
        """(k-mer, count) table of the narrow stream in ONE native call (kmg_extract_sort_count: the
        extraction kernel is the sort's first prefix pass), and the number of windows that belong
        to the wide stream.  seq.py:284-328 + batch.py:156-168 + join.py:63-130,265-285.
        min_count / max_count: only the rows with min_count <= count <= max_count (kmg_extract_sort_count_range)."""
        rng = count_range(min_count, max_count)
        win_begin, win_end, kb, cap, keys, keys_alt, _, _, ws, ws_bytes = self._pipeline_buffers(
            d, k, rc, 0, reuse, win_begin, win_end)
        counts = self._out(reuse, "counts", cap * 4)
        res = (C.c_uint64 * 4)()
        if rng is None:
            _lib.check(self.lib.kmg_extract_sort_count(d.bases.data_ptr(), d.n_bases, win_begin, win_end, k, int(rc),
                                                       d.lut.data_ptr(), keys.data_ptr(), keys_alt.data_ptr(),
                                                       counts.data_ptr(), res, ws.data_ptr(), ws_bytes, self._stream()))
        else:
            _lib.check(self.lib.kmg_extract_sort_count_range(d.bases.data_ptr(), d.n_bases, win_begin, win_end, k, int(rc),
                                                             d.lut.data_ptr(), keys.data_ptr(), keys_alt.data_ptr(), rng[0],
                                                             rng[1], counts.data_ptr(), res, ws.data_ptr(), ws_bytes,
                                                             self._stream()))
        return CountTable(keys_alt if res[3] else keys, counts, int(res[0]), kb, k, False), int(res[2])

    @_on_device
    def uniq_narrow(self, d: DeviceInput, k: int, rc: bool = False, reuse: Optional[str] = None, win_begin: int = 0,
                    win_end: Optional[int] = None, val_bytes: Optional[int] = None) -> Tuple[KeyArray, int]:
        """Singleton keys with their (position << 1 | strand) payload of the narrow stream in ONE native
        call (kmg_extract_sort_uniq), and the number of wide-stream windows.  join.py:243-263."""
        vb = val_bytes or d.payload_bytes
        win_begin, win_end, kb, cap, keys, keys_alt, vals, vals_alt, ws, ws_bytes = self._pipeline_buffers(
            d, k, rc, vb, reuse, win_begin, win_end)
        res = (C.c_uint64 * 4)()
        _lib.check(self.lib.kmg_extract_sort_uniq(d.bases.data_ptr(), d.n_bases, win_begin, win_end, k, int(rc),
                                                  d.lut.data_ptr(), keys.data_ptr(), keys_alt.data_ptr(), vals.data_ptr(),
                                                  vals_alt.data_ptr(), vb, d.pos_offset, res, ws.data_ptr(), ws_bytes,
                                                  self._stream()))
        k_, v_ = (keys_alt, vals_alt) if res[3] else (keys, vals)
        return KeyArray(k_, None, v_, None, int(res[0]), kb, vb, k, False, is_sorted=True), int(res[2])

    def count(self, d: DeviceInput, k: int, rc: bool = False, min_count: int = 1,
              max_count: Optional[int] = None) -> List[CountTable]:
        """`kmer count` (SEQ_COUNT) on device: one CountTable per stream, restricted to the rows with
        min_count <= count <= max_count."""
        tab, n_other = self.count_narrow(d, k, rc, min_count=min_count, max_count=max_count)
        out = [tab]
        if n_other:
            out.append(self.sort_count(self.extract(d, k, rc, wide=True, val_bytes=0), min_count=min_count,
                                       max_count=max_count))
        return out

    def uniq(self, d: DeviceInput, k: int, rc: bool = False) -> List[KeyArray]:
        """`kmer uniq` on device: singleton keys with payload, one KeyArray per stream."""
        vb = d.payload_bytes
        sing, n_other = self.uniq_narrow(d, k, rc, val_bytes=vb)
        out = [sing]
        if n_other:
            out.append(self.sort_uniq(self.extract(d, k, rc, wide=True, val_bytes=vb)))
        return out

    # ---- key-range passes: output larger than the device ---------------------------------------------
    @_on_device
    def part_counts(self, d: DeviceInput, k: int, rc: bool, n_parts: int) -> Tuple[np.ndarray, np.ndarray]:
        """Keys per part of the narrow and of the wide stream (k >= 12): the narrow counts come from the
        4-mer histogram of the bases (kmg_extract_dest_counts); a count-only wide extraction
        (kmg_extract_wide_part_counts) runs only when the input has wide windows."""
        n_win = max(0, d.n_bases - k + 1)
        narrow, wide = np.zeros(n_parts, np.int64), np.zeros(n_parts, np.int64)
        if n_win == 0:
            return narrow, wide
        counts = torch.zeros(n_parts + 1, dtype=torch.int64, device=self.device)
        ws_bytes = self.lib.kmg_dest_counts_workspace_bytes()
        ws = self._buf("ws_dest_counts", ws_bytes)
        _lib.check(self.lib.kmg_extract_dest_counts(d.bases.data_ptr(), d.n_bases, 0, n_win, k, int(rc), d.lut.data_ptr(),
                                                    n_parts, counts.data_ptr(), ws.data_ptr(), ws_bytes, self._stream()))
        c = counts.cpu().numpy()
        narrow[:] = c[:n_parts]
        if c[n_parts]:
            _lib.check(self.lib.kmg_extract_wide_part_counts(d.bases.data_ptr(), d.n_bases, 0, n_win, k, int(rc),
                                                             d.lut.data_ptr(), d.comp16.data_ptr(), n_parts,
                                                             self._wide_parts(d.rna, n_parts).data_ptr(),
                                                             counts.data_ptr(), self._stream()))
            wide[:] = counts[:n_parts].cpu().numpy()
        return narrow, wide

    def _wide_parts(self, rna: int, n_parts: int) -> torch.Tensor:
        key = f"wide_parts_{rna}_{n_parts}"
        if key not in self._scratch:
            self._scratch[key] = torch.from_numpy(wide_part_table(rna, n_parts)).to(self.device)
        return self._scratch[key]

    @_on_device
    def extract_parts(self, d: DeviceInput, k: int, rc: bool, wide: bool, val_bytes: int, n_parts: int, part_lo: int,
                      part_hi: int, n_keys: int) -> KeyArray:
        """extract() restricted to the keys of parts [part_lo, part_hi) (kmg_extract_parts), into buffers of
        exactly `n_keys` keys (from part_counts)."""
        n_win = max(0, d.n_bases - k + 1)
        kb = key_bytes(k, wide)
        keys, keys_alt = self._new(n_keys * kb), self._new(n_keys * kb)
        vals = self._new(n_keys * val_bytes) if val_bytes else None
        vals_alt = self._new(n_keys * val_bytes) if val_bytes else None
        ws_bytes = self.lib.kmg_extract_workspace_bytes(n_win)
        ws = self._buf("ws_extract", ws_bytes)
        _lib.check(self.lib.kmg_extract_parts(
            d.bases.data_ptr(), d.n_bases, 0, n_win, k, int(rc), int(wide), d.lut.data_ptr(), d.comp16.data_ptr(), n_parts,
            part_lo, part_hi, self._wide_parts(d.rna, n_parts).data_ptr(), keys.data_ptr(), kb, _ptr(vals), val_bytes,
            d.pos_offset, self._small.data_ptr(), None, ws.data_ptr(), ws_bytes, self._stream()))
        self._status(ws)
        n = int(self._small[:1].cpu().numpy().view(np.uint64)[0])
        if n != n_keys:
            raise _lib.KmgError(f"parts [{part_lo}, {part_hi}) of {n_parts}: extracted {n} keys, counted {n_keys}")
        return KeyArray(keys, keys_alt, vals, vals_alt, n, kb, val_bytes, k, wide)

    def _line_bytes(self, d: DeviceInput, k: int, mode: str) -> int:
        """Text capacity per row that format_counts / format_uniq / format_vector require."""
        if mode == "vec":
            return 11
        return k + 12 if mode == "count" else k + 48 + max((len(nm) for nm in d.flat.names), default=0)

    def _one_pass_bytes(self, d: DeviceInput, k: int, rc: bool, mode: str, n_other: int, val_bytes: int,
                        text_bytes: int) -> int:
        """Device bytes of the whole-input path (count() / uniq()): window-sized buffers of the fused
        pipeline, then those of the wide stream while the narrow result is held."""
        lib = self.lib
        n_win = max(0, d.n_bases - k + 1)
        cap = max(n_win * keys_per_window(rc), 1)
        if mode == "vec":  # extract() with window-sized buffers, one stream at a time
            return pass_bytes(k, mode, cap, cap if n_other else 0, val_bytes, text_bytes, n_win)
        if mode == "histo":  # the fused pipeline, then the wide stream beside the (kept) pipeline workspace
            ws_pipe = lib.kmg_pipeline_histo_workspace_bytes(n_win, k, int(rc))
            need = 2 * cap * key_bytes(k, False) + ws_pipe + lib.kmg_extract_workspace_bytes(n_win)
            if n_other:
                need = max(need, ws_pipe + pass_bytes(k, mode, 0, n_other * keys_per_window(rc), 0, 0, n_win))
            return int(need)
        kb, kw = key_bytes(k, False), key_bytes(k, True)
        item = kb +(4 if mode == "count" else val_bytes)
        narrow = 2 * cap * item + lib.kmg_pipeline_workspace_bytes(n_win, k, int(rc), 0 if mode == "count" else val_bytes)
        if n_other:
            m = n_other * keys_per_window(rc)
            witem = kw + (4 if mode == "count" else val_bytes)
            wide = cap * item + 2 * cap * witem + pass_bytes(k, mode, 0, m, val_bytes, 0, n_win) + 8 * (cap + m)
            narrow = max(narrow, wide)
        return int(narrow + lib.kmg_extract_workspace_bytes(n_win) + text_bytes)

    def _resident_bytes(self, d: DeviceInput) -> int:
        return sum(int(t.numel()) * t.element_size() for t in (d.bases, d.rec_starts, d.names_buf, d.name_offs)
                   if t is not None)

    def device_budget(self, d: DeviceInput, budget_bytes: Optional[int] = None) -> int:
        """Device bytes a pass may use.  `budget_bytes` (or the KMG_DEVICE_BUDGET environment variable) is the
        whole job's budget, from which the resident bases, names and record starts are subtracted; by default
        it is the device's free memory (plus what torch's allocator caches) minus DEVICE_HEADROOM."""
        if budget_bytes is None and os.environ.get("KMG_DEVICE_BUDGET"):
            budget_bytes = int(os.environ["KMG_DEVICE_BUDGET"])
        if budget_bytes is not None:
            return int(budget_bytes) - self._resident_bytes(d)
        free, _ = torch.cuda.mem_get_info(self.device)
        cached = torch.cuda.memory_reserved(self.device) - torch.cuda.memory_allocated(self.device)
        return int(free + cached - DEVICE_HEADROOM)

    def _text_plan(self, d: DeviceInput, k: int, mode: str, chunk_rows: Optional[int]) -> Tuple[int, int]:
        """(rows per text chunk, device bytes of the text stage: two chunk buffers + the newline index; for
        "vec" two chunk buffers per gzip worker, chunks no longer than the longest record and by default no more
        buffer rows than bases)."""
        line = self._line_bytes(d, k, mode)
        if mode == "vec":
            workers = self._vec_workers(d)
            longest = int(np.diff(d.flat.rec_starts.astype(np.int64)).max(initial=1))
            rows = max(1, min(chunk_rows or min(VEC_CHUNK_ROWS, -(-d.n_bases // (2 * workers))), longest))
            return rows, 2 * workers * rows * line + self.lib.kmg_format_workspace_bytes(rows)
        rows = max(1, chunk_rows or TEXT_CHUNK_BYTES // line)
        return rows, 2 * rows * line + rows * line + rows * (2 if mode == "uniq" else 1) * 8

    @_on_device
    def plan_passes(self, d: DeviceInput, k: int, rc: bool, mode: str, budget_bytes: Optional[int] = None,
                    chunk_rows: Optional[int] = None, text: bool = True) -> PassPlan:
        """Split `kmer count` (mode "count") / `kmer uniq` ("uniq") / `kmer count -m VEC_COUNT*` ("vec") / `kmer histo`
        ("histo", never a text stage) into
        key-range passes that fit the device budget (device_budget; for "vec" minus the resident vector pair,
        8 * (n_bases + 1) bytes).  Everything fits: one pass on the whole-input path.  Otherwise contiguous
        parts of PASS_PARTS are grouped (plan_parts; needs k >= 12, ValueError if not or if one part alone
        does not fit).  text=False: no text stage (Engine.abundance copies the vectors out instead)."""
        if mode not in ("count", "uniq", "vec", "histo"):
            raise AssertionError(f"unknown mode {mode!r}")
        budget = self.device_budget(d, budget_bytes)
        if mode == "vec":
            budget -= 8 * (d.n_bases + 1)
        vb = d.payload_bytes
        text_bytes = self._text_plan(d, k, mode, chunk_rows)[1] if text and mode != "histo" else 0
        n, n_other = self.count_windows(d, k, rc)
        one = self._one_pass_bytes(d, k, rc, mode, n_other, vb, text_bytes)
        n_win = max(0, d.n_bases - k + 1)
        return make_plan(k, budget, one, (n, n_other * keys_per_window(rc)), lambda: self.part_counts(d, k, rc, PASS_PARTS),
                         lambda a, b: pass_bytes(k, mode, a, b, vb, text_bytes, n_win))

    def write_count(self, d: DeviceInput, k: int, rc: bool, fh: BinaryIO, budget_bytes: Optional[int] = None,
                    chunk_rows: Optional[int] = None, min_count: int = 1, max_count: Optional[int] = None) -> PassPlan:
        """Write the bytes of count_text() to the binary file object `fh`, pass by pass and chunk by chunk, so
        device memory is bounded by the budget and host memory by the text chunk.  Returns the plan.
        min_count / max_count: only the lines whose count is in [min_count, max_count] (the count plan)."""
        return self._write_passes(d, k, rc, fh, "count", budget_bytes, chunk_rows, count_range(min_count, max_count))

    def write_uniq(self, d: DeviceInput, k: int, rc: bool, fh: BinaryIO, budget_bytes: Optional[int] = None,
                   chunk_rows: Optional[int] = None) -> PassPlan:
        """Write the bytes of uniq_text() to `fh` (see write_count)."""
        return self._write_passes(d, k, rc, fh, "uniq", budget_bytes, chunk_rows)

    def write_batch(self, d: DeviceInput, k: int, rc: bool, fh: BinaryIO, chunk_rows: Optional[int] = None) -> None:
        """Write the text of the reference's batch files (batch.py:281-296: every k-mer as
        ">ref:start-end:strand\\nSEQ\\n", stably sorted by sequence, batch.py:156-168) to `fh` as one sorted
        batch; how the reference splits records over files is not part of its contract (SURVEY.md f-3).  The
        payload sorts are stable, so equal sequences keep their emission order.  rc = CANONICAL: AssertionError."""
        per_strand(rc)
        self._write_text(d, k, "uniq", fh, [self.sorted_streams(d, k, rc, d.payload_bytes)], chunk_rows)

    def count_text(self, d: DeviceInput, k: int, rc: bool = False, min_count: int = 1,
                   max_count: Optional[int] = None) -> bytes:
        """Bytes of the reference's `kmer count` output file (join.py:284), from the whole-input path; with a
        range, only the lines whose count is in [min_count, max_count]."""
        fh = io.BytesIO()
        self._write_text(d, k, "count", fh, [self.count(d, k, rc, min_count, max_count)])
        return fh.getvalue()

    def uniq_text(self, d: DeviceInput, k: int, rc: bool = False) -> bytes:
        """Bytes of the reference's `kmer uniq` output file (join.py:262), from the whole-input path."""
        fh = io.BytesIO()
        self._write_text(d, k, "uniq", fh, [self.uniq(d, k, rc)])
        return fh.getvalue()

    @_on_device
    def _write_passes(self, d: DeviceInput, k: int, rc: bool, fh: BinaryIO, mode: str, budget_bytes: Optional[int],
                      chunk_rows: Optional[int], rng: Optional[Tuple[int, int]] = None) -> PassPlan:
        if d.rec_starts is None and mode == "uniq":  # resident before the budget is taken
            self._upload_names(d)
        plan = self.plan_passes(d, k, rc, mode, budget_bytes, chunk_rows)
        plan.pass_ms = self._write_text(d, k, mode, fh, self.pass_tables(d, k, rc, mode, plan, rng), chunk_rows)
        return plan

    @_on_device
    def _write_text(self, d: DeviceInput, k: int, mode: str, fh: BinaryIO, passes: Iterable[list],
                    chunk_rows: Optional[int] = None) -> List[float]:
        """Write the text of every table list of `passes` ([narrow] or [narrow, wide] sorted tables, formatted
        as `mode` "count" or "uniq" lines) to `fh`, in chunks of `chunk_rows` narrow rows (default: 256 MB of
        text) through one _ChunkSink.  Returns each list's time between CUDA events, its production included."""
        rows, _ = self._text_plan(d, k, mode, chunk_rows)
        sink = _ChunkSink(self, fh, rows * self._line_bytes(d, k, mode))
        passes, pass_ms = iter(passes), []
        try:
            while True:
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record()
                tabs = next(passes, None)
                if tabs is None:
                    break
                self._emit_chunks(sink, d, k, mode, tabs, rows)
                del tabs  # a pass's buffers are freed before the next pass allocates its own
                t1.record()
                t1.synchronize()
                pass_ms.append(t0.elapsed_time(t1))
        finally:
            sink.close()
        return pass_ms

    def pass_tables(self, d: DeviceInput, k: int, rc: bool, mode: str, plan: PassPlan,
                    rng: Optional[Tuple[int, int]] = None):
        """Yield, pass by pass, the sorted tables of `plan`: [narrow] or [narrow, wide] CountTables (count) /
        singleton KeyArrays (uniq).  Concatenated in pass order they are the tables of count() / uniq().
        rng (count): (min_count, max_count) of the rows kept, None for all."""
        vb = d.payload_bytes
        lo_c, hi_c = rng if rng is not None else (1, None)
        for lo, hi in plan.parts:
            if plan.n_parts == 1:
                yield self.count(d, k, rc, lo_c, hi_c) if mode == "count" else self.uniq(d, k, rc)
                continue
            tabs = []
            for wide, n_keys in ((False, int(plan.narrow[lo:hi].sum())), (True, int(plan.wide[lo:hi].sum()))):
                if wide and not n_keys:
                    break
                a = self.extract_parts(d, k, rc, wide, 0 if mode == "count" else vb, plan.n_parts, lo, hi, n_keys)
                tabs.append(self.sort_count(a, min_count=lo_c, max_count=hi_c) if mode == "count" else self.sort_uniq(a))
                del a
            yield tabs
            del tabs

    def _emit_chunks(self, sink: _ChunkSink, d: DeviceInput, k: int, mode: str, tabs: list, rows: int) -> None:
        """Text of one pass (narrow table + optional wide table) in chunks of `rows` narrow rows; the wide
        lines go into the chunk whose rows they sort among (merge_ranks)."""
        per = 1 if mode == "count" else 2  # lines per row
        nar = tabs[0]
        n = nar.n
        rw = np.zeros(0, np.int64)
        wid = tabs[1] if len(tabs) > 1 and tabs[1].n else None
        if wid is not None:
            if n:
                rn, rw_d = self.merge_ranks(nar.keys, n, wid.keys, wid.n, k, d.rna)
                del rn
                rw = rw_d.cpu().numpy()
            else:
                rw = np.zeros(wid.n, np.int64)

        def fmt(t, lo: int, cnt: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
            if mode == "count":
                part = CountTable(t.keys[lo * t.key_bytes:], t.counts[lo * 4:], cnt, t.key_bytes, k, t.wide)
                return self.format_counts(part, d.rna, out)
            part = KeyArray(t.keys[lo * t.key_bytes:], None, t.vals[lo * t.val_bytes:], None, cnt, t.key_bytes,
                            t.val_bytes, k, t.wide, is_sorted=True)
            return self.format_uniq(part, d, out)

        starts = list(range(0, n, rows)) or [0]
        for ci, lo in enumerate(starts):
            hi = min(lo + rows, n)
            last = ci == len(starts) - 1
            jlo = int(np.searchsorted(rw, lo, "left"))
            jhi = len(rw) if last else int(np.searchsorted(rw, hi, "left"))
            buf = sink.buffer()
            text = fmt(nar, lo, hi - lo, buf)
            if jhi == jlo:
                sink.submit(text, None)
                continue
            # wide lines of this chunk: host text + line boundaries; byte offsets of the narrow rows they precede
            tw = fmt(wid, jlo, jhi - jlo).cpu().numpy()
            w_ends = np.concatenate(([0], np.flatnonzero(tw == 10)[per - 1::per] + 1))
            q = rw[jlo:jhi] - lo  # insert before narrow row q of the chunk
            inner = np.unique(q[(q > 0) & (q < hi - lo)])
            offs = {0: 0, hi - lo: int(text.numel())}
            if inner.size:
                nl = torch.nonzero(text == 10).flatten()
                at = torch.from_numpy(inner * per - 1).to(self.device)
                for qq, e in zip(inner.tolist(), (nl[at] + 1).cpu().numpy().tolist()):
                    offs[qq] = int(e)
                del nl
            pieces, prev, j = [], 0, 0
            while j < len(q):
                j2 = j
                while j2 < len(q) and q[j2] == q[j]:
                    j2 += 1
                o = offs[int(q[j])]
                pieces.append((None, prev, o))
                pieces.append((tw, int(w_ends[j]), int(w_ends[j2])))
                prev, j = o, j2
            pieces.append((None, prev, int(text.numel())))
            sink.submit(text, pieces)

    # ---- abundance vectors: kmer count -m VEC_COUNT / VEC_COUNT_MASKED ----------------------------------
    @_on_device
    def abundance(self, d: DeviceInput, k: int, rc: bool = False, masked: bool = False,
                  budget_bytes: Optional[int] = None) -> Tuple[np.ndarray, np.ndarray]:
        """VEC_COUNT / VEC_COUNT_MASKED (join.py:287-335): per flat position the number of occurrences of the
        k-mer that starts there ('+' vector) / of its reverse complement ('-' vector); masked: occurrences
        in other records only.  Computed by the pass loop of write_vectors (_fill_vectors) under
        plan_passes(mode="vec").  Returns host uint32 arrays over the flat buffer.  rc = CANONICAL: AssertionError."""
        per_strand(rc)
        if d.rec_starts is None:
            self._upload_names(d)
        out, _ = self._fill_vectors(d, k, rc, masked, self.plan_passes(d, k, rc, "vec", budget_bytes, text=False))
        host = out.cpu().numpy().view(np.uint32)
        return host[: d.n_bases + 1], host[d.n_bases + 1:]

    def _fill_vectors(self, d: DeviceInput, k: int, rc: bool, masked: bool, plan: PassPlan) -> Tuple[torch.Tensor, List[float]]:
        """The device vector pair (int32 holding uint32, '+' over flat [0, n_bases], '-' after it) and the time of
        each pass.  Every pass extracts the keys of its parts with their payload, one stream at a time, sorts
        them stably (payloads ascend inside a run: position order in, stable sort) and scatters every element's
        group size (kmg_abundance_scatter).  Equal k-mers share a part, so each group is whole inside one pass
        and the scatter writes final values; the one-pass plan extracts without a part filter."""
        n = d.n_bases
        out = torch.zeros(2 * (n + 1), dtype=torch.int32, device=self.device)
        plus, minus = out[: n + 1], out[n + 1:]
        err = torch.zeros(1, dtype=torch.int32, device=self.device)
        vb = d.payload_bytes
        pass_ms = []
        for lo, hi in plan.parts:
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            for wide, per_part in ((False, plan.narrow), (True, plan.wide)):
                n_keys = int(per_part[lo:hi].sum())
                if plan.n_parts == 1 and (n_keys or not wide):
                    a = self.extract(d, k, rc, wide=wide, val_bytes=vb, want_hist=not wide)
                elif plan.n_parts > 1 and n_keys:
                    a = self.extract_parts(d, k, rc, wide, vb, plan.n_parts, lo, hi, n_keys)
                else:
                    continue
                a = self.sort(a)
                if a.n:
                    _lib.check(self.lib.kmg_abundance_scatter(
                        a.keys.data_ptr(), a.vals.data_ptr(), a.n, a.key_bytes, a.val_bytes, d.rec_starts.data_ptr(),
                        d.flat.n_rec, int(masked), d.pos_offset, plus.data_ptr(), minus.data_ptr(), err.data_ptr(),
                        self._stream()))
                del a  # the narrow buffers are freed before the wide stream is extracted
            t1.record()
            t1.synchronize()
            pass_ms.append(t0.elapsed_time(t1))
        if int(err.item()):
            raise ValueError("a k-mer occurs more than 2^32-1 times: count does not fit uint32")
        return out, pass_ms

    @_on_device
    def vector_extents(self, d: DeviceInput, plus: torch.Tensor, minus: torch.Tensor) -> np.ndarray:
        """int64 [n_rec, 2]: length of every record's '+' / '-' vector, its last non-zero entry + 1 or 0
        (kmg_vector_extents): one small copy instead of the vectors."""
        n_rec = d.flat.n_rec
        if n_rec == 0:
            return np.zeros((0, 2), np.int64)
        out = torch.empty(2 * n_rec, dtype=torch.int64, device=self.device)
        _lib.check(self.lib.kmg_vector_extents(plus.data_ptr(), minus.data_ptr(), d.n_bases, d.rec_starts.data_ptr(), n_rec,
                                               out.data_ptr(), self._stream()))
        return out.cpu().numpy().reshape(n_rec, 2)

    @_on_device
    def format_vector(self, counts: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Device text "COUNT\\n" per entry of `counts` (a 32-bit vector slice, read as uint32), exact length.
        `out`: a buffer of at least 11 * n bytes to write it into."""
        n = int(counts.numel())
        if n == 0:
            return torch.empty(0, dtype=torch.uint8, device=self.device)
        text = self._new(11 * n) if out is None else out
        ws_bytes = self.lib.kmg_format_workspace_bytes(n)
        ws = self._buf("ws_fmt", ws_bytes)
        _lib.check(self.lib.kmg_format_vector(counts.data_ptr(), n, text.data_ptr(), self._small[4:].data_ptr(),
                                              ws.data_ptr(), ws_bytes, self._stream()))
        self._status(ws)
        nbytes = int(self._small[4:5].cpu().numpy().view(np.uint64)[0])
        return text[:nbytes]

    def _vec_workers(self, d: DeviceInput) -> int:
        return max(1, min(VEC_GZIP_THREADS, 2 * d.flat.n_rec))

    @_on_device
    def write_vectors(self, d: DeviceInput, k: int, rc: bool, masked: bool, dirpath: str,
                      budget_bytes: Optional[int] = None, chunk_rows: Optional[int] = None) -> PassPlan:
        """`kmer count -m VEC_COUNT` (masked: VEC_COUNT_MASKED): one `REF___STRAND.gz` per non-empty vector in
        `dirpath` (extension stripped, abundance.vector_paths), the files abundance.write_vectors writes for
        device_vectors().  The vector pair stays on the device: the passes of plan_passes(mode="vec") fill it,
        kmg_vector_extents trims it, and each vector leaves as device text in chunks of `chunk_rows` entries
        through pinned buffers.  Files are gzip-compressed (one stream each, level 9 as gzip.open) on a pool of
        host threads while the GPU formats the next chunks: host memory is O(threads x chunk).  Returns the plan
        with pass_ms and text_ms filled in.  rc = CANONICAL: AssertionError (the vectors are per strand)."""
        per_strand(rc)
        import gzip
        from collections import deque

        from kman_b200 import abundance

        names = d.flat.names
        abundance.check_unique_names(names)
        if d.rec_starts is None:
            self._upload_names(d)
        plan = self.plan_passes(d, k, rc, "vec", budget_bytes, chunk_rows)
        vec, plan.pass_ms = self._fill_vectors(d, k, rc, masked, plan)
        n = d.n_bases
        strands = (vec[: n + 1], vec[n + 1:])
        lengths = self.vector_extents(d, *strands)
        jobs = [(r, s, int(lengths[r, s])) for r in range(len(names)) for s in (0, 1) if lengths[r, s]]
        paths = abundance.vector_paths(dirpath, [(names[r], "+-"[s]) for r, s, _ in jobs])
        if not jobs:
            return plan
        rows, _ = self._text_plan(d, k, "vec", chunk_rows)
        workers = min(self._vec_workers(d), len(jobs))
        header = np.frombuffer(b"# k=%d\n" % k, np.uint8)
        starts = d.flat.rec_starts.astype(np.int64)
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        todo, active, opened = deque(zip(jobs, paths)), [], []
        sink = _ChunkSink(self, None, rows * 11, slots=2 * workers, workers=workers)
        try:
            while todo or active:
                while todo and len(active) < workers:  # one file per worker, chunks submitted round robin
                    (r, s, length), path = todo.popleft()
                    opened.append(gzip.open(path, "wb"))
                    active.append([opened[-1], strands[s][int(starts[r]):int(starts[r]) + length], 0])
                for lane in list(active):
                    fh, v, off = lane
                    cnt = min(rows, int(v.numel()) - off)
                    text = self.format_vector(v[off:off + cnt], sink.buffer())
                    sink.submit(text, [(header, 0, header.size), (None, 0, int(text.numel()))] if off == 0 else None, fh)
                    lane[2] = off + cnt
                    if lane[2] == v.numel():
                        sink.then(fh, fh.close)
                        active.remove(lane)
            t1.record()
        finally:
            sink.close()
            for fh in opened:
                fh.close()
        t1.synchronize()
        plan.text_ms = t0.elapsed_time(t1)
        return plan

    # ---- multiplicity spectrum: kmer histo ---------------------------------------------------------------
    @_on_device
    def histo_narrow(self, d: DeviceInput, k: int, rc: bool, out: Tuple[int, int, int], reuse: Optional[str] = None) -> int:
        """Add the narrow stream's multiplicity histogram to `out` = (d_hist, d_big, d_n_big) device addresses in ONE
        native call (kmg_extract_sort_histo: count_narrow()'s front end, no table); returns the number of windows
        that belong to the wide stream."""
        win_begin, win_end = window_range(d, k)
        kb = key_bytes(k, False)
        cap = max((win_end - win_begin) * keys_per_window(rc), 1)
        keys, keys_alt = self._out(reuse, "keys", cap * kb), self._out(reuse, "keys_alt", cap * kb)
        ws_bytes = self.lib.kmg_pipeline_histo_workspace_bytes(win_end - win_begin, k, int(rc))
        ws = self._buf("ws_pipeline", ws_bytes)
        res = (C.c_uint64 * 4)()
        _lib.check(self.lib.kmg_extract_sort_histo(d.bases.data_ptr(), d.n_bases, win_begin, win_end, k, int(rc),
                                                   d.lut.data_ptr(), keys.data_ptr(), keys_alt.data_ptr(), *out, res,
                                                   ws.data_ptr(), ws_bytes, self._stream()))
        return int(res[2])

    @_on_device
    def sort_histo(self, a: KeyArray, out: Tuple[int, int, int]) -> None:
        """Add the multiplicity histogram of the keys of `a` to `out` (see histo_narrow).  8- and 16-byte keys:
        kmg_sort_histo (consumes both key buffers); 32-byte wide keys: kmg_sort256 + kmg_rle_count +
        kmg_count_histogram."""
        assert a.val_bytes == 0
        if a.n == 0:
            return
        if a.key_bytes == 32:
            t = self.rle_count(self.sort(a))
            _lib.check(self.lib.kmg_count_histogram(t.counts.data_ptr(), t.n, *out, self._stream()))
            return
        ws_bytes = self.lib.kmg_sort_histo_workspace_bytes(a.n, a.key_bytes, a.key_bits)
        ws = self._buf("ws_sort", ws_bytes)
        _lib.check(self.lib.kmg_sort_histo(a.keys.data_ptr(), a.keys_alt.data_ptr(), a.n, a.key_bytes, a.key_bits,
                                           _ptr(a.hist), *out, ws.data_ptr(), ws_bytes, self._stream()))
        a.hist = None
        self._status(ws)

    def _histogram(self, d: DeviceInput, k: int, rc: bool, budget_bytes: Optional[int]) -> Tuple[np.ndarray, np.ndarray, PassPlan]:
        window_range(d, k)  # (the k checks, before any work)
        plan = self.plan_passes(d, k, rc, "histo", budget_bytes, text=False)
        total = int(plan.narrow.sum() + plan.wide.sum())
        nbins = _lib.KMG_HISTO_BINS
        # one device buffer, read back once: bins [nbins] | list length | list of multiplicities >= nbins
        acc = torch.zeros(8 * (nbins + 1) + 4 * (total // nbins + 1), dtype=torch.uint8, device=self.device)
        out = (acc.data_ptr(), acc.data_ptr() + 8 * (nbins + 1), acc.data_ptr() + 8 * nbins)
        for lo, hi in plan.parts:
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            if plan.n_parts == 1:
                if self.histo_narrow(d, k, rc, out):
                    self.sort_histo(self.extract(d, k, rc, wide=True, val_bytes=0), out)
            else:
                for wide, per_part in ((False, plan.narrow), (True, plan.wide)):
                    n_keys = int(per_part[lo:hi].sum())
                    if n_keys:
                        self.sort_histo(self.extract_parts(d, k, rc, wide, 0, plan.n_parts, lo, hi, n_keys), out)
            t1.record()
            t1.synchronize()
            plan.pass_ms.append(t0.elapsed_time(t1))
        raw = acc.cpu().numpy()
        bins = raw[: 8 * (nbins + 1)].view(np.uint64)
        big = raw[8 * (nbins + 1):].view(np.uint32)[: int(bins[nbins])]
        mult = np.flatnonzero(bins[:nbins]).astype(np.uint64)
        n_kmers = bins[:nbins][mult.astype(np.int64)]
        if big.size:
            bm, bc = np.unique(big, return_counts=True)
            mult = np.concatenate([mult, bm.astype(np.uint64)])
            n_kmers = np.concatenate([n_kmers, bc.astype(np.uint64)])
        return mult, n_kmers.astype(np.uint64), plan

    @_on_device
    def histogram(self, d: DeviceInput, k: int, rc: bool = False,
                  budget_bytes: Optional[int] = None) -> Tuple[np.ndarray, np.ndarray]:
        """`kmer histo`: the multiplicity spectrum of the (k-mer, count) table count() would build, without the
        table.  Returns uint64 arrays (mult, n_kmers): every multiplicity that occurs, ascending, and the number
        of distinct k-mers seen exactly that often.  Narrow and wide stream, and the key-range passes of
        plan_passes(mode="histo") when the input does not fit `budget_bytes`, add into one device histogram."""
        mult, n_kmers, _ = self._histogram(d, k, rc, budget_bytes)
        return mult, n_kmers

    def write_histogram(self, d: DeviceInput, k: int, rc: bool, fh: BinaryIO,
                        budget_bytes: Optional[int] = None) -> PassPlan:
        """Write histogram() to the binary file `fh`, one "M\tN\n" line per multiplicity M (nothing for an empty
        result).  Returns the plan with pass_ms filled in."""
        mult, n_kmers, plan = self._histogram(d, k, rc, budget_bytes)
        fh.write("".join("%d\t%d\n" % mn for mn in zip(mult.tolist(), n_kmers.tolist())).encode("ascii"))
        return plan


_engines: Dict[int, Engine] = {}


def get_engine(device: Optional[int] = None) -> Engine:
    """Process-wide engine for a device (created on first use)."""
    if not torch.cuda.is_available():
        _lib.load()
        raise _lib.KmgError("no CUDA device visible: kman_b200 has no CPU fallback")
    idx = torch.cuda.current_device() if device is None else device
    if idx not in _engines:
        _engines[idx] = Engine(idx)
    return _engines[idx]
