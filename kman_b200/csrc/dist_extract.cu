// Fused extraction + range partition + peer-memory exchange for the multi-GPU path.
//
// There is no counterpart in the reference (it merges batch files on one host,
// kmermaid/join.py:63-93).  The extraction itself is the K1+K2 front end of extract_tile.cuh
// (kmermaid/seq.py:284-328, rc :245-282); what differs is where the keys go: every key is
// written straight into the receive buffer of the GPU that owns its key range
//     part = ((key >> (2k-16)) * n_parts) >> 16
// through peer-mapped pointers (CUDA IPC over NVLink), so the range partition pass, its
// histogram and the NCCL all-to-all of the staged keys all disappear and the transfer
// overlaps the extraction tile by tile.  A first launch in COUNT_ONLY mode sizes the regions
// (reads the bases only); region placement is then  offset[src][dst] = sum of the earlier
// sources' counts, exchanged as a G x G matrix.
//
// The order of the keys inside a destination region is not deterministic (tiles reserve their
// slots with an atomic cursor); the full radix sort that follows makes the result deterministic.
#include <type_traits>

#include "extract_tile.cuh"

namespace kmg {

constexpr int DX_BLOCK = 256;
constexpr int DX_MAX_PARTS = 64;

struct ScatterParams {
    const uint8_t* bases;
    uint64_t n_bases;
    uint64_t win_begin, win_end;
    uint64_t first_tile;
    int k;
    int n_parts;
    const uint8_t* lut;
    void* const* dest_keys;        // device array [n_parts]: base of this source's view of every receive buffer
    void* const* dest_vals;        // device array [n_parts] or null
    unsigned long long* cursors;   // [n_parts] next free element in each destination (this source's region)
    unsigned long long* counts;    // COUNT_ONLY: [n_parts] keys per destination, [n_parts] = wide windows
    uint64_t pos_offset;
    // shared-cursor mode (kmg_extract_scatter_shared): ONE cursor per destination, living in the
    // destination's memory and advanced by every source with system-scope atomics over NVLink
    unsigned long long* const* cursor_ptrs;  // device array [n_parts] or null
    unsigned long long capacity;             // elements every receive buffer holds
    uint32_t* status;                        // [0] = 1: a reservation passed `capacity`; [1] = 1: wide windows seen
};
constexpr unsigned long long DX_NO_STORE = ~0ull;

template <typename KeyT>
__device__ __forceinline__ uint32_t part_of(const KeyT& key, int key_bits, uint32_t n_parts) {
    return (key_digit(key, key_bits - 16, 0xFFFFu) * n_parts) >> 16;
}

// rank of this lane's key among the tile's keys with the same destination (any order across
// warps is fine): lanes with equal `part` are found with ceil(log2 n_parts) ballots and their
// lowest lane reserves the group's slots with one shared-memory atomic
__device__ __forceinline__ uint32_t part_rank(uint32_t part, bool active, int part_bits, uint32_t* s_cnt) {
    uint32_t m = __ballot_sync(0xffffffffu, active);
    for (int b = 0; b < part_bits; ++b) {
        const uint32_t bal = __ballot_sync(0xffffffffu, (part >> b) & 1u);
        m &= bal ^ (((part >> b) & 1u) - 1u);
    }
    if (!active) m = 0;
    const uint32_t lower = __popc(m & lanemask_lt());
    uint32_t base = 0;
    if (active && lower == 0) base = atomicAdd(&s_cnt[part], __popc(m));
    base = __shfl_sync(0xffffffffu, base, m ? __ffs(m) - 1 : 0);
    return base + lower;
}

template <typename KeyT, int PPT, bool RC, int VAL_BYTES, bool COUNT_ONLY>
__global__ void __launch_bounds__(DX_BLOCK) extract_scatter_kernel(const ScatterParams p) {
    constexpr int TILE = DX_BLOCK * PPT;
    constexpr int WORDS = TILE / 16 + EX_HALO_WORDS;
    constexpr int OUT_PER_WIN = RC ? 2 : 1;
    using ValT = typename std::conditional<VAL_BYTES == 4, uint32_t, uint64_t>::type;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    KeyT* s_keys = reinterpret_cast<KeyT*>(smem_raw);
    ValT* s_vals = reinterpret_cast<ValT*>(smem_raw + sizeof(KeyT) * TILE * OUT_PER_WIN);
    __shared__ uint32_t s_codes[WORDS];
    __shared__ uint16_t s_bad[WORDS];
    __shared__ uint16_t s_inv[WORDS];
    __shared__ uint8_t s_lut[256];
    __shared__ uint32_t s_cnt[DX_MAX_PARTS], s_off[DX_MAX_PARTS + 1];
    __shared__ unsigned long long s_base[DX_MAX_PARTS];
    __shared__ uint32_t s_wide;

    const int t = threadIdx.x;
    const uint32_t tile = blockIdx.x;
    if (t < DX_MAX_PARTS) s_cnt[t] = 0;
    if (t == 0) s_wide = 0;
    s_lut[t] = p.lut[t];
    __syncthreads();
    const uint64_t tile_pos = (p.first_tile + tile) * (uint64_t)TILE;

    encode_tile_words<DX_BLOCK, WORDS>(p.bases, p.n_bases, t, tile_pos, s_lut, s_codes, s_bad, s_inv);
    __syncthreads();

    // ---- K2: rolling windows ---------------------------------------------------------------------
    const int k = p.k;
    const int key_bits = 2 * k;
    const int joff = (t * PPT) & 15;
    const auto [X0, X1, X2, B0, B1, I0, I1] = load_tile_words(s_codes, s_bad, s_inv, (t * PPT) >> 4);
    int part_bits = 0;
    while ((1 << part_bits) < p.n_parts) ++part_bits;

    // Window validity as narrow_window_flags (extract_tile.cuh) decides it, but taken one window at a time
    // next to that window's ranks: computed for all PPT windows up front, the same rule costs this kernel
    // up to 10 registers (rc) and an 8-byte spill (u128 keys, 8-byte payload).
    // fast path: no base that is bad for the narrow stream among the PPT+k-1 bases my windows span
    bool span_clean;
    {
        const uint64_t W0 = joff == 0 ? B0 : ((B0 << joff) | (B1 >> (64 - joff)));
        const int span = PPT + k - 1;
        if (span <= 64) span_clean = (W0 >> (64 - span)) == 0;
        else span_clean = W0 == 0 && ((B1 << joff) >> (128 - span)) == 0;
    }
    uint32_t vf = 0, nwide = 0;
    // slot of every emitted key inside its destination group of the tile: (part << 20) | rank
    uint32_t where[PPT * OUT_PER_WIN];
    KeyT keys[PPT];
#pragma unroll
    for (int j = 0; j < PPT; ++j) {
        // (every lane ranks every window: part_rank's ballots are warp-collective)
        const int je = joff + j;
        const uint64_t pos = tile_pos + (uint64_t)t * PPT + j;
        const bool in_range = pos >= p.win_begin && pos < p.win_end;
        bool valid = in_range;
        if (!span_clean) {
            const uint64_t bm = (je == 0 ? B0 : ((B0 << je) | (B1 >> (64 - je)))) >> (64 - k);
            const uint64_t im = (je == 0 ? I0 : ((I0 << je) | (I1 >> (64 - je)))) >> (64 - k);
            valid = in_range && bm == 0;
            if (in_range && im == 0 && bm != 0) ++nwide;
        }
        if (valid) vf |= 1u << j;
        const KeyT key = build_key<KeyT>(X0, X1, X2, joff + j, k);
        keys[j] = key;
        const uint32_t part = valid ? part_of(key, key_bits, (uint32_t)p.n_parts) : 0u;
        const uint32_t rank = part_rank(part, valid, part_bits, s_cnt);
        where[j * OUT_PER_WIN] = (part << 20) | rank;
        if constexpr (RC) {
            const KeyT rk = rc_key(key, k);
            const uint32_t part2 = valid ? part_of(rk, key_bits, (uint32_t)p.n_parts) : 0u;
            const uint32_t rank2 = part_rank(part2, valid, part_bits, s_cnt);
            where[j * 2 + 1] = (part2 << 20) | rank2;
        }
    }
    if (nwide) atomicAdd(&s_wide, nwide);
    __syncthreads();

    if constexpr (COUNT_ONLY) {
        if (t < p.n_parts && s_cnt[t]) atomicAdd(&p.counts[t], (unsigned long long)s_cnt[t]);
        if (t == 0 && s_wide) atomicAdd(&p.counts[p.n_parts], (unsigned long long)s_wide);
        return;
    } else {
        // reserve the tile's slots in every destination region; group offsets in the staging buffer
        if (t < p.n_parts && s_cnt[t]) {
            if (p.cursor_ptrs) {
                const unsigned long long b = atomicAdd_system(p.cursor_ptrs[t], (unsigned long long)s_cnt[t]);
                if (b + s_cnt[t] > p.capacity) {  // the caller re-runs the exchange with exact region sizes
                    atomicExch(&p.status[0], 1u);
                    s_base[t] = DX_NO_STORE;
                } else {
                    s_base[t] = b;
                }
            } else {
                const unsigned long long b = atomicAdd(&p.cursors[t], (unsigned long long)s_cnt[t]);
                // (kmg_extract_scatter_checked: the caller launched before it knew whether the receive
                // buffers still fit; nothing is stored past their end)
                if (p.capacity && b + s_cnt[t] > p.capacity) {
                    atomicExch(&p.status[0], 1u);
                    s_base[t] = DX_NO_STORE;
                } else {
                    s_base[t] = b;
                }
            }
        }
        if (t == 0 && s_wide && p.status) atomicExch(&p.status[1], 1u);
        if (t == 0) {
            uint32_t run = 0;
            for (int d = 0; d < p.n_parts; ++d) {
                s_off[d] = run;
                run += s_cnt[d];
            }
            s_off[p.n_parts] = run;
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < PPT; ++j) {
            if (!((vf >> j) & 1u)) continue;
            const uint64_t pos = tile_pos + (uint64_t)t * PPT + j + p.pos_offset;
            const uint32_t w0 = where[j * OUT_PER_WIN];
            const uint32_t i0 = s_off[w0 >> 20] + (w0 & 0xFFFFFu);
            s_keys[i0] = keys[j];
            if constexpr (VAL_BYTES != 0) s_vals[i0] = make_val<ValT>(pos, 0);
            if constexpr (RC) {
                const uint32_t w1 = where[j * 2 + 1];
                const uint32_t i1 = s_off[w1 >> 20] + (w1 & 0xFFFFFu);
                s_keys[i1] = rc_key(keys[j], k);
                if constexpr (VAL_BYTES != 0) s_vals[i1] = make_val<ValT>(pos, 1);
            }
        }
        __syncthreads();
        // peer stores: every destination group is a contiguous run -> coalesced NVLink writes, and 128-byte
        // aligned ones: a run starts anywhere in its destination, so the threads are assigned from the
        // 128-byte line the run starts in (the first lanes of the first round sit idle) and every warp store
        // covers whole lines instead of straddling them
        constexpr uint32_t LINE = 128 / sizeof(KeyT);
        for (int d = 0; d < p.n_parts; ++d) {
            const unsigned long long b = s_base[d];
            if (b == DX_NO_STORE) continue;
            const uint32_t cnt = s_off[d + 1] - s_off[d];
            const uint32_t shift = (uint32_t)((reinterpret_cast<uintptr_t>(p.dest_keys[d]) / sizeof(KeyT) + b) & (LINE - 1));
            KeyT* dk = reinterpret_cast<KeyT*>(p.dest_keys[d]) + b;
            for (uint32_t j = t; j < cnt + shift; j += DX_BLOCK) {
                if (j < shift) continue;
                const uint32_t o = j - shift;
                dk[o] = s_keys[s_off[d] + o];
                if constexpr (VAL_BYTES != 0) (reinterpret_cast<ValT*>(p.dest_vals[d]) + b)[o] = s_vals[s_off[d] + o];
            }
        }
    }
}

template <typename KeyT, int PPT, bool RC, int VB, bool CO>
static int launch_scatter(const ScatterParams& p, uint32_t n_tiles, cudaStream_t st) {
    constexpr int TILE = DX_BLOCK * PPT;
    const size_t smem = CO ? 16 : (sizeof(KeyT) + (VB == 4 ? 4 : (VB == 8 ? 8 : 0))) * (size_t)TILE * (RC ? 2 : 1);
    auto kern = extract_scatter_kernel<KeyT, PPT, RC, VB, CO>;
    KMG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<n_tiles, DX_BLOCK, smem, st>>>(p);
    KMG_LAUNCH_CHECK();
    return KMG_OK;
}

template <typename KeyT, int PPT, bool CO>
static int dispatch_scatter(const ScatterParams& p, uint32_t n_tiles, int rc, int vb, cudaStream_t st) {
    if (CO) vb = 0;
    if (rc) {
        if (vb == 0) return launch_scatter<KeyT, PPT, true, 0, CO>(p, n_tiles, st);
        if (vb == 4) return launch_scatter<KeyT, PPT, true, 4, CO>(p, n_tiles, st);
        return launch_scatter<KeyT, PPT, true, 8, CO>(p, n_tiles, st);
    }
    if (vb == 0) return launch_scatter<KeyT, PPT, false, 0, CO>(p, n_tiles, st);
    if (vb == 4) return launch_scatter<KeyT, PPT, false, 4, CO>(p, n_tiles, st);
    return launch_scatter<KeyT, PPT, false, 8, CO>(p, n_tiles, st);
}

}  // namespace kmg

using namespace kmg;

static int scatter_impl(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k, int rc,
                        const uint8_t* d_lut256, int n_parts, void* const* d_dest_keys, void* const* d_dest_vals,
                        int key_bytes, int val_bytes, uint64_t pos_offset, uint64_t* d_cursors, uint64_t* d_counts,
                        int count_only, uint64_t* const* d_cursor_ptrs, uint64_t capacity, uint32_t* d_status,
                        void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    KMG_REQUIRE(rc != KMG_CANONICAL, KMG_ERR_ARG, "the multi-GPU exchange has no canonical keys (rc must be 0 or 1)");
    KMG_REQUIRE(k >= 8, KMG_ERR_RANGE, "the multi-GPU range partition needs k >= 8 (16 key bits), got %d", k);
    KMG_REQUIRE(k <= 64, KMG_ERR_RANGE, "k=%d: this build supports k <= 64", k);
    KMG_REQUIRE(n_parts >= 1 && n_parts <= DX_MAX_PARTS, KMG_ERR_ARG, "n_parts must be in [1,%d]", DX_MAX_PARTS);
    KMG_REQUIRE(win_begin <= win_end, KMG_ERR_ARG, "win_begin > win_end");
    KMG_REQUIRE(val_bytes == 0 || val_bytes == 4 || val_bytes == 8, KMG_ERR_ARG, "val_bytes must be 0, 4 or 8");
    if (val_bytes == 4)
        KMG_REQUIRE(((pos_offset + n_bases) << 1) < (1ull << 32), KMG_ERR_RANGE, "val_bytes=4 needs < 2^31 positions");
    KMG_REQUIRE(key_bytes == (k <= 32 ? 8 : 16), KMG_ERR_ARG, "key_bytes must be %d for k=%d", k <= 32 ? 8 : 16, k);
    KMG_REQUIRE(((uintptr_t)d_bases & 15) == 0, KMG_ERR_ARG, "d_bases must be 16-byte aligned");
    KMG_REQUIRE(d_lut256, KMG_ERR_ARG, "null pointer argument");
    if (count_only) {
        KMG_REQUIRE(d_counts, KMG_ERR_ARG, "d_counts is null");
        KMG_CUDA(cudaMemsetAsync(d_counts, 0, sizeof(uint64_t) * (n_parts + 1), st));
    } else {
        KMG_REQUIRE(d_dest_keys && (d_cursors || d_cursor_ptrs), KMG_ERR_ARG, "null pointer argument");
        KMG_REQUIRE((val_bytes == 0) == (d_dest_vals == nullptr), KMG_ERR_ARG, "d_dest_vals / val_bytes mismatch");
    }
    if (win_end == win_begin) return KMG_OK;
    const uint64_t tile = (uint64_t)DX_BLOCK * (key_bytes == 8 ? 16 : 8);
    const uint64_t first_tile = win_begin / tile;
    const uint64_t n_tiles = (win_end + tile - 1) / tile - first_tile;
    KMG_REQUIRE(n_tiles < (1ull << 31), KMG_ERR_RANGE, "too many tiles");
    ScatterParams p;
    p.bases = d_bases;
    p.n_bases = n_bases;
    p.win_begin = win_begin;
    p.win_end = win_end;
    p.first_tile = first_tile;
    p.k = k;
    p.n_parts = n_parts;
    p.lut = d_lut256;
    p.dest_keys = d_dest_keys;
    p.dest_vals = d_dest_vals;
    p.cursors = reinterpret_cast<unsigned long long*>(d_cursors);
    p.counts = reinterpret_cast<unsigned long long*>(d_counts);
    p.pos_offset = pos_offset;
    p.cursor_ptrs = reinterpret_cast<unsigned long long* const*>(d_cursor_ptrs);
    p.capacity = capacity;
    p.status = d_status;
    if (count_only) {
        if (key_bytes == 8) return dispatch_scatter<uint64_t, 16, true>(p, (uint32_t)n_tiles, rc, 0, st);
        return dispatch_scatter<u128, 8, true>(p, (uint32_t)n_tiles, rc, 0, st);
    }
    if (key_bytes == 8) return dispatch_scatter<uint64_t, 16, false>(p, (uint32_t)n_tiles, rc, val_bytes, st);
    return dispatch_scatter<u128, 8, false>(p, (uint32_t)n_tiles, rc, val_bytes, st);
}

extern "C" int kmg_extract_scatter(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k,
                                   int rc, const uint8_t* d_lut256, int n_parts, void* const* d_dest_keys,
                                   void* const* d_dest_vals, int key_bytes, int val_bytes, uint64_t pos_offset,
                                   uint64_t* d_cursors, uint64_t* d_counts, int count_only, void* stream) {
    return scatter_impl(d_bases, n_bases, win_begin, win_end, k, rc, d_lut256, n_parts, d_dest_keys, d_dest_vals, key_bytes,
                        val_bytes, pos_offset, d_cursors, d_counts, count_only, nullptr, 0, nullptr, stream);
}

extern "C" int kmg_extract_scatter_checked(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end,
                                           int k, int rc, const uint8_t* d_lut256, int n_parts, void* const* d_dest_keys,
                                           void* const* d_dest_vals, int key_bytes, int val_bytes, uint64_t pos_offset,
                                           uint64_t* d_cursors, uint64_t capacity, uint32_t* d_status, void* stream) {
    KMG_REQUIRE(d_cursors && d_status && capacity > 0, KMG_ERR_ARG, "null pointer argument");
    return scatter_impl(d_bases, n_bases, win_begin, win_end, k, rc, d_lut256, n_parts, d_dest_keys, d_dest_vals, key_bytes,
                        val_bytes, pos_offset, d_cursors, nullptr, 0, nullptr, capacity, d_status, stream);
}

extern "C" int kmg_extract_scatter_shared(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end,
                                          int k, int rc, const uint8_t* d_lut256, int n_parts, void* const* d_dest_keys,
                                          void* const* d_dest_vals, int key_bytes, int val_bytes, uint64_t pos_offset,
                                          uint64_t* const* d_cursor_ptrs, uint64_t capacity, uint32_t* d_status,
                                          void* stream) {
    KMG_REQUIRE(d_cursor_ptrs && d_status && capacity > 0, KMG_ERR_ARG, "null pointer argument");
    return scatter_impl(d_bases, n_bases, win_begin, win_end, k, rc, d_lut256, n_parts, d_dest_keys, d_dest_vals, key_bytes,
                        val_bytes, pos_offset, nullptr, nullptr, 0, d_cursor_ptrs, capacity, d_status, stream);
}

// ---- peer memory through CUDA IPC -----------------------------------------------------------------
extern "C" int kmg_ipc_alloc(size_t bytes, void** d_ptr_out, uint8_t* h_handle64) {
    KMG_REQUIRE(d_ptr_out && h_handle64 && bytes > 0, KMG_ERR_ARG, "bad argument");
    void* ptr = nullptr;
    KMG_CUDA(cudaMalloc(&ptr, bytes));
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, ptr);
    if (e != cudaSuccess) {
        cudaFree(ptr);
        set_error("cudaIpcGetMemHandle: %s", cudaGetErrorString(e));
        return KMG_ERR_CUDA;
    }
    static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
    memcpy(h_handle64, &h, 64);
    *d_ptr_out = ptr;
    return KMG_OK;
}

extern "C" int kmg_ipc_open(const uint8_t* h_handle64, void** d_ptr_out) {
    KMG_REQUIRE(d_ptr_out && h_handle64, KMG_ERR_ARG, "bad argument");
    cudaIpcMemHandle_t h;
    memcpy(&h, h_handle64, 64);
    KMG_CUDA(cudaIpcOpenMemHandle(d_ptr_out, h, cudaIpcMemLazyEnablePeerAccess));
    return KMG_OK;
}

extern "C" int kmg_ipc_close(void* d_ptr) {
    KMG_CUDA(cudaIpcCloseMemHandle(d_ptr));
    return KMG_OK;
}

extern "C" int kmg_ipc_free(void* d_ptr) {
    KMG_CUDA(cudaFree(d_ptr));
    return KMG_OK;
}
