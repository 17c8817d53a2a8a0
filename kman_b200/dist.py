"""Multi-GPU path: one process per GPU, torch.distributed for the plumbing.

There is nothing like this in the reference (it merges batch files on one host,
kmermaid/join.py:63-93).  The two partitioning rules are:

  * INPUT: the flat base buffer is cut into `world` contiguous chunks of window starts; a
    rank's chunk of bases carries k-1 extra bases so that every window lies in exactly one
    chunk -- the reference's own chunking rule, Sequence.batcher (kmermaid/seq.py:361-383,
    known answer tests/test_seq.py:136-138).
  * KEYS: range partition by the top key bits, part = ((key >> (bits-16)) * world) >> 16
    (libkmg's kmg_range_partition), so rank r ends up with key range r: equal k-mers meet on
    one GPU (counts are final, no second reduction) and the rank-order concatenation of the
    per-rank sorted outputs is globally sorted.

The only collective on the data path is ONE all-to-all of the partitioned keys (and payload
in uniq mode), preceded by an all-gather of the world x world count matrix.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Tuple

import os

import numpy as np
import torch
import torch.distributed as dist


# ---- pure host logic (unit-tested on CPU) ------------------------------------------------------
def chunk_windows(n_bases: int, k: int, world: int) -> List[Tuple[int, int]]:
    """Split the window starts [0, n_bases-k+1) into `world` contiguous ranges [b, e).

    Rank r needs bases [b, e + k - 1): consecutive chunks overlap by k-1 bases, exactly like
    Sequence.batcher's `start += batchSize - k + 1` (seq.py:379-383)."""
    n_win = max(0, n_bases - k + 1)
    per = (n_win + world - 1) // world if world else 0
    out = []
    for r in range(world):
        b = min(r * per, n_win)
        e = min(b + per, n_win)
        out.append((b, e))
    return out


def chunk_bases(n_bases: int, k: int, world: int) -> List[Tuple[int, int]]:
    """Base ranges [b, e) each rank must hold (window range + k-1 overlap)."""
    return [(b, min(n_bases, e + k - 1) if e > b else b) for b, e in chunk_windows(n_bases, k, world)]


def part_of_keys(keys_hi16: np.ndarray, world: int) -> np.ndarray:
    """numpy mirror of libkmg's RangeDigit on the top 16 key bits (used by the CPU tests)."""
    return (keys_hi16.astype(np.uint64) * np.uint64(world)) >> np.uint64(16)


def sort_bits_after_partition(key_bits: int, world: int) -> int:
    """Bits the local sort still has to cover.  When `world` is a power of two, the top
    log2(world) bits are constant inside a rank after the range partition."""
    if world & (world - 1) == 0:
        return max(0, key_bits - (world.bit_length() - 1))
    return key_bits



# ---- collectives ---------------------------------------------------------------------------------
# The product backend is NCCL (one process per GPU; collectives are stream-ordered, so an all-reduce
# doubles as a device-side fence).  A gloo group is accepted for the TEST topology "two ranks sharing
# ONE GPU" (tests/test_gpu_dist.py: NCCL refuses two ranks per device, CUDA IPC does not): the tensor is
# staged through the host, which also makes every collective a full host-level barrier.
def _staged(group) -> bool:
    return dist.get_backend(group) == "gloo"


def _all_reduce(t: torch.Tensor, op=None, group=None) -> None:
    op = dist.ReduceOp.SUM if op is None else op
    if t.is_cuda and _staged(group):
        h = t.cpu()
        dist.all_reduce(h, op=op, group=group)
        t.copy_(h)
    else:
        dist.all_reduce(t, op=op, group=group)


def _all_gather_into_tensor(out: torch.Tensor, t: torch.Tensor, group=None) -> None:
    if t.is_cuda and _staged(group):
        world = dist.get_world_size(group)
        parts = [torch.empty(t.shape, dtype=t.dtype) for _ in range(world)]
        dist.all_gather(parts, t.cpu(), group=group)
        out.copy_(torch.cat([p.reshape(-1) for p in parts]).reshape(out.shape))
    else:
        dist.all_gather_into_tensor(out, t, group=group)


def _all_to_all_single(recv: torch.Tensor, send: torch.Tensor, output_split_sizes, input_split_sizes, group=None) -> None:
    if send.is_cuda and _staged(group):
        h = torch.empty(recv.shape, dtype=recv.dtype)
        dist.all_to_all_single(h, send.cpu(), output_split_sizes=output_split_sizes,
                               input_split_sizes=input_split_sizes, group=group)
        recv.copy_(h)
    else:
        dist.all_to_all_single(recv, send, output_split_sizes=output_split_sizes, input_split_sizes=input_split_sizes,
                               group=group)


# ---- exchange ------------------------------------------------------------------------------------
def gather_count_matrix(send_counts: np.ndarray, device: torch.device, group=None) -> np.ndarray:
    """All-gather of every rank's per-destination counts -> (world, world) int64 matrix
    M[src, dst]."""
    world = dist.get_world_size(group)
    mine = torch.from_numpy(np.ascontiguousarray(send_counts, dtype=np.int64)).to(device)
    allc = torch.empty(world * world, dtype=torch.int64, device=device)
    _all_gather_into_tensor(allc, mine, group=group)
    return allc.cpu().numpy().reshape(world, world)


def exchange(send: torch.Tensor, send_counts: np.ndarray, elems_per_item: int = 1, group=None,
             matrix: Optional[np.ndarray] = None) -> Tuple[torch.Tensor, np.ndarray]:
    """One all-to-all(v).  `send` holds the items grouped by destination rank (int64 view,
    `elems_per_item` int64 per item); returns (recv tensor, per-source item counts)."""
    rank = dist.get_rank(group)
    if matrix is None:
        matrix = gather_count_matrix(send_counts, send.device, group)
    recv_counts = matrix[:, rank].copy()
    recv = torch.empty(int(recv_counts.sum()) * elems_per_item, dtype=send.dtype, device=send.device)
    _all_to_all_single(
        recv,
        send[: int(np.sum(send_counts)) * elems_per_item],
        output_split_sizes=[int(c) * elems_per_item for c in recv_counts],
        input_split_sizes=[int(c) * elems_per_item for c in send_counts],
        group=group,
    )
    return recv, recv_counts


@dataclass
class RankShard:
    """What one rank holds of a distributed input."""

    device_input: object  # engine.DeviceInput of the rank's chunk (+ k-1 overlap)
    win_begin: int  # local window range inside the chunk (always 0 .. n)
    win_end: int
    n_windows_global: int


class _PeerUnavailable(RuntimeError):
    """CUDA IPC peer mapping failed on at least one rank: every rank falls back to NCCL together."""


class _DevMem:
    """A raw device allocation exposed to torch through __cuda_array_interface__ (no copy)."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


class PeerBuffers:
    """Receive buffers of all ranks, mapped into this process with CUDA IPC.

    Every rank allocates its receive buffer through libkmg (kmg_ipc_alloc), the 64-byte handles
    are all-gathered, and each rank maps its peers' buffers (kmg_ipc_open).  `ptr_table` is the
    device array of per-destination base pointers.  Every buffer starts with a HEADER whose first
    word is the destination's shared cursor (kmg_extract_scatter_shared); the keys / payloads
    start at `data` / `data_table`.

    The constructor never raises between collectives: a rank whose allocation or mapping fails still
    takes part in the handle all-gather (with None) and ends up with `ok = False`; the caller
    all-reduces `ok` and every rank then releases what it holds WITHOUT further collectives
    (`release_local`)."""

    HEADER = 256

    def __init__(self, engine, nbytes: int, group=None):
        import ctypes as C

        from kman_b200 import _lib

        self.eng, self.lib, self.group = engine, engine.lib, group
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.nbytes = int(nbytes)  # payload bytes (without the header)
        self.ok, self.error = True, ""
        self.local_ptr, self.local, self.peer_ptrs = None, None, []
        handle = (C.c_uint8 * 64)()
        try:
            ptr = C.c_void_p()
            _lib.check(self.lib.kmg_ipc_alloc(self.nbytes + self.HEADER, C.byref(ptr), handle))
            self.local_ptr = ptr.value
        except Exception as exc:  # CUDA IPC unavailable (container policy, out of memory, ...)
            self.ok, self.error = False, repr(exc)
        handles = [None] * self.world
        dist.all_gather_object(handles, bytes(handle) if self.ok else None, group=group)
        if self.ok and any(h is None for h in handles):
            self.ok, self.error = False, "a peer could not allocate its receive buffer"
        if self.ok:
            try:
                for r, h in enumerate(handles):
                    if r == self.rank:
                        self.peer_ptrs.append(self.local_ptr)
                        continue
                    q = C.c_void_p()
                    hb = (C.c_uint8 * 64).from_buffer_copy(h)
                    _lib.check(self.lib.kmg_ipc_open(hb, C.byref(q)))
                    self.peer_ptrs.append(q.value)
            except Exception as exc:
                self.ok, self.error = False, repr(exc)
        if not self.ok:
            return
        self.local = torch.as_tensor(_DevMem(self.local_ptr, self.nbytes + self.HEADER), device=engine.device)
        self.data = self.local[self.HEADER:]
        self.cursor = self.local[:8].view(torch.int64)
        self.ptr_table = torch.tensor(self.peer_ptrs, dtype=torch.int64, device=engine.device)
        self.data_table = self.ptr_table + self.HEADER

    def owns(self, t: Optional[torch.Tensor]) -> bool:
        """Does `t` live inside this rank's receive buffer?"""
        if t is None or self.local_ptr is None:
            return False
        return self.local_ptr <= t.data_ptr() < self.local_ptr + self.nbytes + self.HEADER

    def release_local(self):
        """Unmap the peers and free the own buffer; no collective (safe when only some ranks fail)."""
        torch.cuda.synchronize()
        for r, q in enumerate(self.peer_ptrs):
            if r != self.rank and q is not None:
                self.lib.kmg_ipc_close(q)
        self.peer_ptrs = []
        self.local = None
        if self.local_ptr is not None:
            self.lib.kmg_ipc_free(self.local_ptr)
            self.local_ptr = None

    def close(self):
        """Collective release: nobody may still be storing into a buffer that is about to be freed."""
        torch.cuda.synchronize()
        dist.barrier(group=self.group)
        self.release_local()


class DistributedCounter:
    """`kmer count` / `kmer uniq` across the GPUs of one box.

    Two exchange paths: `p2p=True` (default when CUDA IPC works) fuses extraction, range partition
    and the transfer into ONE kernel that stores keys into the owners' receive buffers over NVLink;
    `p2p=False` is the plain path: extract -> range partition pass -> NCCL all-to-all.

    Results (CountTable / KeyArray) live in torch-owned memory: a table that the sort left inside the
    peer-mapped receive buffer is copied out before it is returned, so it stays valid while peers
    store the next step's keys.  With `reuse` scratch (the benchmark loop) a result is valid until
    the next call on this counter."""

    def __init__(self, engine, group=None, p2p: Optional[bool] = None):
        self.eng = engine
        self.group = group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.p2p = (os.environ.get("KMG_DIST_P2P", "1") != "0") if p2p is None else p2p
        self._peer_keys: Optional[PeerBuffers] = None
        self._peer_vals: Optional[PeerBuffers] = None
        # single-launch exchange with shared cursors: measured faster up to 4 GPUs (N=2 +14 %, N=4 +4.5 %);
        # at 8 the 8 x 8 sources x destinations contend for the cursor words and the exact exchange
        # wins (-4 %).  KMG_DIST_SHARED=0/1 overrides.
        env = os.environ.get("KMG_DIST_SHARED")
        self.shared = (self.world <= 4) if env is None else env != "0"
        self._cap_elems = 0  # elements the receive buffers are provisioned for; identical on every rank
        self._timing = {} if os.environ.get("KMG_DIST_TIMING") == "1" else None
        self._t_last = None
        self._info_host = torch.zeros(8, dtype=torch.int64).pin_memory() if torch.cuda.is_available() else None

    def _mark(self, name: str) -> None:
        """KMG_DIST_TIMING=1: wall-clock per stage (synchronising; a development aid, see
        tools/dist_stage_bench.py)."""
        if self._timing is None:
            return
        import time

        torch.cuda.synchronize()
        now = time.perf_counter()
        if self._t_last is not None:
            self._timing[name] = self._timing.get(name, 0.0) + (now - self._t_last)
        self._t_last = now

    # ---- fused extraction + partition + peer stores ---------------------------------------------
    def _ensure_peer(self, which: str, nbytes: int) -> PeerBuffers:
        """(Re)allocate the mapped receive buffers.  `nbytes` derives from values every rank agrees on
        (all-gathered counts / all-reduced maxima), so all ranks take the same decision here and
        issue the same collectives, whether or not the mapping succeeds on every one of them."""
        cur = getattr(self, which)
        if cur is not None and cur.nbytes >= nbytes:
            return cur
        if cur is not None:
            cur.close()
            setattr(self, which, None)
        cur = PeerBuffers(self.eng, int(nbytes * 1.1) + 4096, self.group)
        flag = torch.tensor([1 if cur.ok else 0], dtype=torch.int64, device=self.eng.device)
        _all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)
        if int(flag.item()) == 0:
            err = cur.error or "a peer could not map the receive buffers"
            cur.release_local()  # no collective: ranks that failed early hold nothing to fence
            raise _PeerUnavailable(err)
        setattr(self, which, cur)
        return cur

    def _dest_counts(self, d, k: int, rc: bool, kb: int) -> torch.Tensor:
        """Per-destination key counts of this rank's windows (+ wide-stream windows in [G])."""
        from kman_b200 import _lib

        eng, lib, G = self.eng, self.eng.lib, self.world
        n_win = max(0, d.n_bases - k + 1)
        counts = torch.zeros(G + 1, dtype=torch.int64, device=eng.device)
        if k >= 12 and G & (G - 1) == 0:
            # from the 4-mer histogram of the bases: no second key-building pass
            ws_bytes = lib.kmg_dest_counts_workspace_bytes()
            ws = eng._buf("ws_dest_counts", ws_bytes)
            _lib.check(lib.kmg_extract_dest_counts(d.bases.data_ptr(), d.n_bases, 0, n_win, k, int(rc), d.lut.data_ptr(), G,
                                                   counts.data_ptr(), ws.data_ptr(), ws_bytes, eng._stream()))
        else:
            _lib.check(lib.kmg_extract_scatter(d.bases.data_ptr(), d.n_bases, 0, n_win, k, int(rc), d.lut.data_ptr(), G, None,
                                               None, kb, 0, d.pos_offset, None, counts.data_ptr(), 1, eng._stream()))
        return counts

    def _extract_exchange_p2p(self, d, k: int, rc: bool, with_vals: bool):
        """Exact regions: per-destination counts (from the 4-mer histogram), ONE all-gather of the
        G x G matrix, region offsets computed on the device, then one kernel extracts the keys and
        stores them into the owning GPUs' receive buffers.  In steady state (buffers provisioned) the
        host does not look at the matrix before the scatter launch: the kernel itself refuses to store
        past the buffers' capacity, and ONE read-back after the fence brings the received count, the
        overflow flag and the wide-window total."""
        from kman_b200 import _lib
        from kman_b200.engine import KeyArray

        eng, lib, G = self.eng, self.eng.lib, self.world
        kb = 8 if k <= 32 else 16
        vb = 8 if with_vals else 0
        n_win = max(0, d.n_bases - k + 1)
        self._mark("(outside)")
        counts = self._dest_counts(d, k, rc, kb)
        self._mark("per-destination counts")
        allc = torch.empty(G * (G + 1), dtype=torch.int64, device=eng.device)
        _all_gather_into_tensor(allc, counts, group=self.group)
        M = allc.view(G, G + 1)
        # my region inside destination dst starts after the regions of the sources before me
        cursors = M[: self.rank, :G].sum(dim=0) if self.rank else torch.zeros(G, dtype=torch.int64, device=eng.device)
        per_dst = M[:, :G].sum(dim=0)
        info = torch.stack([per_dst[self.rank], per_dst.max(), M[:, G].sum()])
        self._mark("all-gather of the count matrix + device-side offsets")
        for attempt in range(2):
            have = self._peer_keys is not None and (not with_vals or self._peer_vals is not None)
            if not have or attempt == 1:
                # (first use, or the guarded launch overflowed: size the buffers from the matrix)
                n_recv, recv_max, n_wide = (int(x) for x in info.cpu())
                self._cap_elems = max(self._cap_elems, int(recv_max * 1.1) + 65536)
            cap = self._cap_elems
            pk = self._ensure_peer("_peer_keys", cap * kb)
            pv = self._ensure_peer("_peer_vals", cap * vb) if with_vals else None
            cap_fit = min(pk.nbytes // kb, pv.nbytes // vb) if pv else pk.nbytes // kb
            status = torch.zeros(2, dtype=torch.int32, device=eng.device)
            cur = cursors.clone()
            # No fence is needed before the stores: the all-gather above completed, so every rank had
            # entered it, and each rank enters it only after (in stream order) it stopped reading its
            # receive buffer of the previous step.
            _lib.check(lib.kmg_extract_scatter_checked(d.bases.data_ptr(), d.n_bases, 0, n_win, k, int(rc), d.lut.data_ptr(),
                                                       G, pk.data_table.data_ptr(), pv.data_table.data_ptr() if pv else None,
                                                       kb, vb, d.pos_offset, cur.data_ptr(), cap_fit, status.data_ptr(),
                                                       eng._stream()))
            self._mark("extract + scatter kernel")
            # device-side fence (no host sync): every rank's peer stores, stream-ordered before its
            # contribution, have landed when the all-reduce completes; it also carries the overflow flag
            _all_reduce(status, op=dist.ReduceOp.MAX, group=self.group)
            self._info_host[:5].copy_(torch.cat([info, status.to(torch.int64)]), non_blocking=True)
            torch.cuda.current_stream(eng.device).synchronize()
            n_recv, recv_max, n_wide, overflow = (int(self._info_host[i]) for i in (0, 1, 2, 3))
            self._mark("fence + read-back")
            if not overflow:
                break
        assert not overflow, "receive buffers sized from the exact count matrix overflowed"
        self._cap_elems = max(self._cap_elems, int(recv_max * 1.1) + 65536)
        alt = eng._buf("p2p_keys_alt", max(n_recv, 1) * kb)
        valt = eng._buf("p2p_vals_alt", max(n_recv, 1) * vb) if with_vals else None
        return KeyArray(pk.data, alt, pv.data if pv else None, valt, n_recv, kb, vb, k, False), n_wide

    def _extract_exchange_shared(self, d, k: int, rc: bool, with_vals: bool):
        """Single-launch exchange: no count launch, no count matrix.  Every destination owns one
        cursor (first word of its receive buffer) that all sources advance with system-scope
        atomics; the buffers are provisioned for 1.25 x the largest per-rank key count seen so far
        (keys that spread evenly over the key ranges).  Returns None when a buffer overflowed (skewed
        keys, or an input larger than any before): the caller then runs the exact exchange, which
        also re-provisions the buffers.

        Every rank issues the same collectives in the same order whatever its own chunk size is: the
        capacity only ever changes through all-reduced values (the MAX of the per-rank key counts
        rides on the second fence, which every step runs anyway)."""
        from kman_b200 import _lib
        from kman_b200.engine import KeyArray

        eng, lib, G = self.eng, self.eng.lib, self.world
        kb = 8 if k <= 32 else 16
        vb = 8 if with_vals else 0
        n_win = max(0, d.n_bases - k + 1)
        n_mine = n_win * (2 if rc else 1)
        scale = float(os.environ.get("KMG_DIST_CAP_SCALE", "1.25"))  # (tests force overflows with a small one)
        self._mark("(outside)")
        if self._cap_elems == 0:  # first exchange of this counter -- on every rank
            t = torch.tensor([n_mine], dtype=torch.int64, device=eng.device)
            _all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
            self._cap_elems = int(int(t.item()) * scale) + 4096
        cap = self._cap_elems
        pk = self._ensure_peer("_peer_keys", cap * kb)
        pv = self._ensure_peer("_peer_vals", cap * vb) if with_vals else None
        cap_fit = min(pk.nbytes // kb, pv.nbytes // vb) if pv else pk.nbytes // kb
        status = torch.zeros(3, dtype=torch.int64, device=eng.device)  # overflow, wide windows seen, keys of this rank
        status32 = torch.zeros(2, dtype=torch.int32, device=eng.device)
        pk.cursor.zero_()
        # device-side barrier (no host sync): every cursor is zero, nobody still reads the last step's keys
        fence = torch.zeros(1, dtype=torch.int32, device=eng.device)
        _all_reduce(fence, group=self.group)
        self._mark("fence 1")
        _lib.check(lib.kmg_extract_scatter_shared(d.bases.data_ptr(), d.n_bases, 0, n_win, k, int(rc), d.lut.data_ptr(), G,
                                                  pk.data_table.data_ptr(), pv.data_table.data_ptr() if pv else None, kb,
                                                  vb, d.pos_offset, pk.ptr_table.data_ptr(), cap_fit, status32.data_ptr(),
                                                  eng._stream()))
        self._mark("extract + scatter kernel")
        # fence + agreement: every rank's peer stores (stream-ordered before its contribution) have landed
        status[:2] = status32
        status[2] = n_mine
        _all_reduce(status, op=dist.ReduceOp.MAX, group=self.group)
        self._info_host[:4].copy_(torch.cat([status, pk.cursor]), non_blocking=True)
        torch.cuda.current_stream(eng.device).synchronize()
        overflow, wide_seen, n_max, n_recv = (int(self._info_host[i]) for i in range(4))
        self._mark("fence 2 + read-back")
        # the same value on every rank: inputs that grew are provisioned for from the next step on
        self._cap_elems = max(self._cap_elems, int(n_max * scale) + 4096)
        if overflow:
            return None
        alt = eng._buf("p2p_keys_alt", max(n_recv, 1) * kb)
        valt = eng._buf("p2p_vals_alt", max(n_recv, 1) * vb) if with_vals else None
        return KeyArray(pk.data, alt, pv.data if pv else None, valt, n_recv, kb, vb, k, False), wide_seen

    def _exchange(self, d, k: int, rc: bool, with_vals: bool):
        """Fused extraction + exchange over peer memory: single launch when it fits, exact otherwise.
        Returns (received KeyArray, wide-stream indicator: > 0 if ANY rank saw wide windows)."""
        r = self._extract_exchange_shared(d, k, rc, with_vals) if self.shared else None
        if r is None:
            r = self._extract_exchange_p2p(d, k, rc, with_vals)
        return r

    def shard(self, flat, k: int, alphabet: Optional[str] = None, natype=None):
        """Upload this rank's chunk of a host-resident flat input (k-1 overlap)."""
        from kman_b200 import alphabet as ab
        from kman_b200.fasta import FlatInput

        natype = natype or ab.NATYPES.DNA
        n_bases = int(flat.bases.shape[0])
        b, e = chunk_bases(n_bases, k, self.world)[self.rank]
        sub = FlatInput(flat.bases[b:e], flat.rec_starts, flat.names, flat.titles)
        d = self.eng.upload(sub, alphabet, natype, with_names=False)
        d.pos_offset = b
        return d

    def _partition_exchange(self, a, with_vals: bool):
        """range partition -> count matrix -> all-to-all; returns the received KeyArray."""
        from kman_b200.engine import KeyArray

        a, pc = self.eng.range_partition(a, self.world)
        per = a.key_bytes // 8
        send = a.keys[: max(a.n, 1) * a.key_bytes].view(torch.int64)
        matrix = gather_count_matrix(pc, a.keys.device, self.group)
        recv, recv_counts = exchange(send, pc, per, self.group, matrix)
        n = int(recv_counts.sum())
        rvals = None
        if with_vals:
            vper = 1
            v64 = a.vals[: max(a.n, 1) * a.val_bytes]
            if a.val_bytes == 4:
                # widen the payload for the exchange so one int64 all-to-all suffices
                v64 = v64.view(torch.int32).to(torch.int64).contiguous().view(torch.uint8)
            rv, _ = exchange(v64.view(torch.int64), pc, vper, self.group, matrix)
            rvals = rv.view(torch.uint8)
        kbuf = recv.view(torch.uint8)
        alt = torch.empty(max(kbuf.numel(), 16), dtype=torch.uint8, device=kbuf.device)
        valt = torch.empty(max(rvals.numel(), 16), dtype=torch.uint8, device=kbuf.device) if with_vals else None
        if kbuf.numel() == 0:
            kbuf = torch.empty(16, dtype=torch.uint8, device=alt.device)
        if with_vals and rvals.numel() == 0:
            rvals = torch.empty(16, dtype=torch.uint8, device=alt.device)
        return KeyArray(kbuf, alt, rvals, valt, n, a.key_bytes, 8 if with_vals else 0, a.k, a.wide)

    def _own(self, t: Optional[torch.Tensor], nbytes: int) -> Optional[torch.Tensor]:
        """A result tensor the sort left inside a peer-mapped receive buffer is copied into torch-owned
        memory (peers overwrite the buffer in the next exchange; it may even be freed and re-mapped)."""
        if t is None:
            return None
        for pb in (self._peer_keys, self._peer_vals):
            if pb is not None and pb.owns(t):
                return t[: max(nbytes, 16)].clone()
        return t

    def _narrow(self, d, k: int, rc: bool, with_vals: bool):
        """(received narrow keys of this rank's key range, does ANY rank hold wide-stream windows)"""
        if self.p2p and k >= 8:
            try:
                return self._exchange(d, k, rc, with_vals)
            except _PeerUnavailable as exc:
                self._fall_back(exc)
        a = self.eng.extract(d, k, rc, wide=False, val_bytes=8 if with_vals else 0)
        n_other = torch.tensor([a.n_other], dtype=torch.int64, device=a.keys.device)
        _all_reduce(n_other, group=self.group)
        return self._partition_exchange(a, with_vals), int(n_other.item())

    def _wide(self, d, k: int, rc: bool, with_vals: bool):
        """The wide (non-ACGT alphabet symbols) stream across ranks: windows are rare, so the plain
        path does it -- local extraction, range partition on the 4-bit keys, all-to-all.
        Collective: every rank calls it once any rank saw a wide window."""
        a = self.eng.extract(d, k, rc, wide=True, val_bytes=8 if with_vals else 0)
        if a.key_bytes == 32:
            return self._wide256_exchange(a, with_vals)
        return self._partition_exchange(a, with_vals)

    def _wide256_exchange(self, a, with_vals: bool):
        """33 <= k <= 64: 256-bit wide keys.  Sorted locally first, a rank's share of every key range is a
        contiguous slice; the slices travel with one all-to-all and the receiver sorts its G sorted runs
        again (kmg_sort256 both times).  Same range rule as the narrow stream: part = (top 16 key bits * G) >> 16."""
        from kman_b200.engine import KeyArray

        eng, G = self.eng, self.world
        a = eng.sort(a)
        dev = a.keys.device
        limbs = a.keys[: max(a.n, 1) * 32].view(torch.int64).view(-1, 4)[: a.n]
        sh = a.key_bits - 16  # >= 116: the top 16 bits sit in limb sh // 64 and possibly the next one
        li, off = sh // 64, sh % 64
        top = (limbs[:, li] >> off) & ((1 << (64 - off)) - 1 if off else -1)
        if off > 48:
            top = top | (limbs[:, li + 1] << (64 - off))
        part = ((top & 0xFFFF) * G) >> 16
        pc = torch.bincount(part, minlength=G).cpu().numpy().astype(np.int64) if a.n else np.zeros(G, np.int64)
        matrix = gather_count_matrix(pc, dev, self.group)
        send = a.keys[: max(a.n, 1) * 32].view(torch.int64)
        recv, recv_counts = exchange(send, pc, 4, self.group, matrix)
        n = int(recv_counts.sum())
        rvals = None
        if with_vals:
            rv, _ = exchange(a.vals[: max(a.n, 1) * 8].view(torch.int64), pc, 1, self.group, matrix)
            rvals = rv.view(torch.uint8)
        kbuf = recv.view(torch.uint8)
        if kbuf.numel() == 0:
            kbuf = torch.empty(32, dtype=torch.uint8, device=dev)
        if with_vals and rvals.numel() == 0:
            rvals = torch.empty(16, dtype=torch.uint8, device=dev)
        alt = torch.empty(max(kbuf.numel(), 32), dtype=torch.uint8, device=dev)
        valt = torch.empty(max(rvals.numel(), 16), dtype=torch.uint8, device=dev) if with_vals else None
        return KeyArray(kbuf, alt, rvals, valt, n, 32, 8 if with_vals else 0, a.k, True)

    def count_streams(self, d, k: int, rc: bool = False, reuse: Optional[str] = "p2p_"):
        """This rank's slice (key range `rank`) of the global count table: [narrow] or [narrow, wide]
        CountTables; rank-order concatenation per stream is globally sorted, counts are final.  rc = CANONICAL:
        AssertionError (the exchange has no canonical keys)."""
        from kman_b200.engine import per_strand

        per_strand(rc)
        r, any_wide = self._narrow(d, k, rc, with_vals=False)
        tab = self.eng.sort_count(r, sort_bits_after_partition(r.key_bits, self.world), reuse=reuse)
        tab.keys = self._own(tab.keys, tab.n * tab.key_bytes)
        self._mark("sort + count")
        out = [tab]
        if any_wide:
            w = self._wide(d, k, rc, with_vals=False)
            out.append(self.eng.sort_count(w, sort_bits_after_partition(w.key_bits, self.world)))
        return out

    def count(self, d, k: int, rc: bool = False):
        """Narrow-stream slice of the count table (see count_streams for inputs with N / IUPAC symbols:
        with the ACGT-only alphabet every valid window is narrow)."""
        return self.count_streams(d, k, rc)[0]

    def uniq_streams(self, d, k: int, rc: bool = False):
        """This rank's slice of the global singleton list (keys + (pos<<1|strand) payload) per stream.  rc = CANONICAL:
        AssertionError."""
        from kman_b200.engine import per_strand

        per_strand(rc)
        r, any_wide = self._narrow(d, k, rc, with_vals=True)
        s = self.eng.sort_uniq(r, sort_bits_after_partition(r.key_bits, self.world))
        s.keys, s.vals = self._own(s.keys, s.n * s.key_bytes), self._own(s.vals, s.n * s.val_bytes)
        out = [s]
        if any_wide:
            w = self._wide(d, k, rc, with_vals=True)
            out.append(self.eng.sort_uniq(w, sort_bits_after_partition(w.key_bits, self.world)))
        return out

    def uniq(self, d, k: int, rc: bool = False):
        return self.uniq_streams(d, k, rc)[0]

    def _fall_back(self, exc) -> None:
        """Every rank raised together (the failure flag is all-reduced): use the NCCL all-to-all path."""
        import warnings

        self.p2p = False
        if self.rank == 0:
            warnings.warn(f"CUDA IPC peer buffers unavailable ({exc}); using the NCCL all-to-all exchange")

    def close(self):
        for which in ("_peer_keys", "_peer_vals"):
            cur = getattr(self, which)
            if cur is not None:
                cur.close()
                setattr(self, which, None)
