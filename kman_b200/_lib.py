"""ctypes binding of libkmg.so (include/kmg.h).  Fails loudly when the library is missing:
there is no CPU fallback anywhere in this package."""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libkmg.so")

KMG_OK = 0
KMG_ERR_ARG, KMG_ERR_CUDA, KMG_ERR_WS, KMG_ERR_RANGE, KMG_ERR_STATE = -1, -2, -3, -4, -5
KMG_HISTO_BINS = 4096  # include/kmg.h
KMG_CANONICAL = 2  # include/kmg.h: `rc` of the canonical strand rule

u8p = C.POINTER(C.c_uint8)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)
vp = C.c_void_p
u64 = C.c_uint64
u32 = C.c_uint32
sz = C.c_size_t
i32 = C.c_int

# name -> (restype, argtypes); mirrors include/kmg.h one to one
SIGNATURES = {
    "kmg_version": (i32, []),
    "kmg_last_error": (C.c_char_p, []),
    "kmg_device_count": (i32, []),
    "kmg_build_lut": (i32, [C.c_char_p, C.c_char_p, u8p, u8p]),
    "kmg_ws_status": (i32, [vp, vp]),
    "kmg_extract_workspace_bytes": (sz, [u64]),
    "kmg_extract": (i32, [vp, u64, u64, u64, i32, i32, i32, vp, vp, vp, i32, vp, i32, u64, vp, vp, vp, sz, vp]),
    "kmg_wide_part_table": (i32, [i32, i32, u8p]),
    "kmg_extract_parts": (i32, [vp, u64, u64, u64, i32, i32, i32, vp, vp, i32, i32, i32, vp, vp, i32, vp, i32, u64, vp,
                                vp, vp, sz, vp]),
    "kmg_extract_wide_part_counts": (i32, [vp, u64, u64, u64, i32, i32, vp, vp, i32, vp, vp, vp]),
    "kmg_radix_sort_workspace_bytes": (sz, [u64, i32, i32, i32, i32]),
    "kmg_radix_sort": (i32, [vp, vp, vp, vp, u64, i32, i32, i32, i32, vp, C.POINTER(i32), vp, sz, vp]),
    "kmg_rle_workspace_bytes": (sz, [u64]),
    "kmg_rle_count": (i32, [vp, u64, i32, vp, vp, vp, vp, sz, vp]),
    "kmg_sort_uniq_workspace_bytes": (sz, [u64, i32, i32, i32]),
    "kmg_sort_uniq": (i32, [vp, vp, vp, vp, u64, i32, i32, i32, vp, vp, C.POINTER(C.c_int), vp, sz, vp]),
    "kmg_sort_count_workspace_bytes": (sz, [u64, i32, i32]),
    "kmg_sort_count": (i32, [vp, vp, u64, i32, i32, vp, vp, vp, C.POINTER(C.c_int), vp, sz, vp]),
    "kmg_pipeline_workspace_bytes": (sz, [u64, i32, i32, i32]),
    "kmg_extract_sort_count": (i32, [vp, u64, u64, u64, i32, i32, vp, vp, vp, vp, u64p, vp, sz, vp]),
    "kmg_sort_count_range": (i32, [vp, vp, u64, i32, i32, vp, u32, u32, vp, vp, C.POINTER(C.c_int), vp, sz, vp]),
    "kmg_extract_sort_count_range": (i32, [vp, u64, u64, u64, i32, i32, vp, vp, vp, u32, u32, vp, u64p, vp, sz, vp]),
    "kmg_filter_counts": (i32, [vp, vp, u64, i32, u32, u32, vp, vp, vp, vp, sz, vp]),
    "kmg_extract_sort_uniq": (i32, [vp, u64, u64, u64, i32, i32, vp, vp, vp, vp, vp, i32, u64, u64p, vp, sz, vp]),
    "kmg_sort_histo_workspace_bytes": (sz, [u64, i32, i32]),
    "kmg_sort_histo": (i32, [vp, vp, u64, i32, i32, vp, vp, vp, vp, vp, sz, vp]),
    "kmg_count_histogram": (i32, [vp, u64, vp, vp, vp, vp]),
    "kmg_pipeline_histo_workspace_bytes": (sz, [u64, i32, i32]),
    "kmg_extract_sort_histo": (i32, [vp, u64, u64, u64, i32, i32, vp, vp, vp, vp, vp, vp, u64p, vp, sz, vp]),
    "kmg_abundance_scatter": (i32, [vp, vp, u64, i32, i32, vp, C.c_uint32, i32, u64, vp, vp, vp, vp]),
    "kmg_vector_extents": (i32, [vp, vp, u64, vp, C.c_uint32, vp, vp]),
    "kmg_format_vector": (i32, [vp, u64, vp, vp, vp, sz, vp]),
    "kmg_sort256_workspace_bytes": (sz, [u64]),
    "kmg_sort256": (i32, [vp, vp, vp, vp, u64, i32, i32, vp, sz, vp]),
    "kmg_merge_ranks_wide": (i32, [vp, u64, vp, u64, i32, i32, vp, vp, vp, vp]),
    "kmg_select_singletons": (i32, [vp, vp, u64, i32, i32, vp, vp, vp, vp, sz, vp]),
    "kmg_partition_workspace_bytes": (sz, [u64, i32, i32]),
    "kmg_range_partition": (i32, [vp, vp, u64, i32, i32, i32, i32, vp, vp, vp, vp, sz, vp]),
    "kmg_extract_scatter": (i32, [vp, u64, u64, u64, i32, i32, vp, i32, vp, vp, i32, i32, u64, vp, vp, i32, vp]),
    "kmg_extract_scatter_checked": (i32, [vp, u64, u64, u64, i32, i32, vp, i32, vp, vp, i32, i32, u64, vp, u64, vp, vp]),
    "kmg_dest_counts_workspace_bytes": (sz, []),
    "kmg_extract_dest_counts": (i32, [vp, u64, u64, u64, i32, i32, vp, i32, vp, vp, sz, vp]),
    "kmg_extract_scatter_shared": (i32, [vp, u64, u64, u64, i32, i32, vp, i32, vp, vp, i32, i32, u64, vp, u64, vp, vp]),
    "kmg_ipc_alloc": (i32, [sz, C.POINTER(vp), u8p]),
    "kmg_ipc_open": (i32, [u8p, C.POINTER(vp)]),
    "kmg_ipc_close": (i32, [vp]),
    "kmg_ipc_free": (i32, [vp]),
    "kmg_fasta_workspace_bytes": (sz, [u64]),
    "kmg_fasta_flatten": (i32, [vp, u64, vp, vp, vp, u64, vp, vp, sz, vp]),
    "kmg_format_workspace_bytes": (sz, [u64]),
    "kmg_format_counts": (i32, [vp, vp, u64, i32, i32, i32, i32, vp, vp, vp, sz, vp]),
    "kmg_format_uniq": (i32, [vp, vp, u64, i32, i32, i32, i32, i32, vp, C.c_uint32, vp, vp, vp, vp, vp, sz, vp]),
    "kmg_merge_ranks": (i32, [vp, u64, i32, vp, u64, i32, i32, i32, vp, vp, vp]),
    "kmg_ctx_create": (i32, [i32, C.POINTER(vp)]),
    "kmg_ctx_destroy": (None, [vp]),
    "kmg_count_host": (i32, [vp, vp, u64, i32, i32, vp, vp, vp, u64, u64p]),
    "kmg_uniq_host": (i32, [vp, vp, u64, i32, i32, vp, vp, vp, u64, u64p]),
    "kmg_set_option": (i32, [C.c_char_p, C.c_int64]),
    "kmg_get_stat": (C.c_int64, [C.c_char_p]),
}

_lock = threading.Lock()
_lib = None


class KmgError(RuntimeError):
    """A libkmg call failed (CUDA error, workspace, device-side check)."""


def load() -> C.CDLL:
    """Load libkmg.so (once).  Raises ImportError with build instructions if it is absent."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.isfile(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: the CUDA extension is not built. Run "
                "`python -c 'import __graft_entry__ as g; g.build()'` (or `make -C kman_b200/csrc`). "
                "kman_b200 has no CPU fallback."
            )
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the library lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib


def check(rc: int) -> None:
    """Translate a libkmg return code into the reference's error conventions: argument
    errors are AssertionError (batcher.py:475-478, batch.py:240-243), the rest RuntimeError."""
    if rc == KMG_OK:
        return
    msg = load().kmg_last_error().decode("utf-8", "replace")
    if rc == KMG_ERR_ARG:
        raise AssertionError(msg)
    if rc == KMG_ERR_RANGE:
        raise ValueError(msg)
    raise KmgError(f"libkmg error {rc}: {msg}")
