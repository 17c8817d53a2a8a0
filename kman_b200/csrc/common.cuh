// Shared device/host helpers for libkmg (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <type_traits>

#include "../../include/kmg.h"

namespace kmg {

// ---- error plumbing ---------------------------------------------------------------------
void set_error(const char* fmt, ...);
void bump_launches(int n = 1);

#define KMG_CUDA(call)                                                                          \
    do {                                                                                        \
        cudaError_t e__ = (call);                                                               \
        if (e__ != cudaSuccess) {                                                               \
            kmg::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            return KMG_ERR_CUDA;                                                                \
        }                                                                                       \
    } while (0)

#define KMG_REQUIRE(cond, code, ...)    \
    do {                                \
        if (!(cond)) {                  \
            kmg::set_error(__VA_ARGS__); \
            return (code);              \
        }                               \
    } while (0)

#define KMG_LAUNCH_CHECK()                                                                \
    do {                                                                                  \
        cudaError_t e__ = cudaGetLastError();                                             \
        if (e__ != cudaSuccess) {                                                         \
            kmg::set_error("%s:%d: launch failed: %s", __FILE__, __LINE__, cudaGetErrorString(e__)); \
            return KMG_ERR_CUDA;                                                          \
        }                                                                                 \
        kmg::bump_launches();                                                             \
    } while (0)

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---- radix pass plan (shared by the sort and by the extract kernel's fused histograms) -------------
constexpr int MAX_PASSES = 16;
constexpr int SORT_RADIX_BITS = 8;
constexpr int SORT_RADIX = 1 << SORT_RADIX_BITS;

struct PassPlan {
    int num_passes;
    int shift[MAX_PASSES];
    int bits[MAX_PASSES];
};

// Full 8-bit digits from `begin_bit` upwards; the top pass takes what is left.  Packed keys hold
// 2 bits per base, so with begin_bit = 0 every digit is a whole number of bases -- which is what
// lets kmg_extract derive all digit histograms from ONE 4-mer histogram (extract.cu).
static inline PassPlan make_plan(int begin_bit, int end_bit) {
    PassPlan plan;
    memset(&plan, 0, sizeof(plan));
    const int bits = end_bit - begin_bit;
    const int np = (bits + SORT_RADIX_BITS - 1) / SORT_RADIX_BITS;
    plan.num_passes = np;
    for (int i = 0; i < np; ++i) {
        plan.shift[i] = begin_bit + i * SORT_RADIX_BITS;
        plan.bits[i] = i + 1 < np ? SORT_RADIX_BITS : bits - i * SORT_RADIX_BITS;
    }
    return plan;
}

// ---- cross-file plumbing of the fused pipeline (pipeline.cu) -----------------------------------------
// the rows a count table keeps (kmg_sort_count_range): min_count <= count <= max_count; the full range is
// the plain count table
struct CountRange {
    uint32_t min_count = 1, max_count = 0xFFFFFFFFu;
    bool full() const { return min_count == 1 && max_count == 0xFFFFFFFFu; }
};
// fused run-length count / singleton request of a hybrid sort: `done` = the local sort produced the
// result itself (counts == null: singletons with payload, kmg_sort_uniq)
struct CountOut {
    uint32_t* counts;
    unsigned long long* n_out;
    bool done;
    CountRange range = {};
};
// multiplicity histogram (kmg_sort_histo): hist[m] = distinct keys seen m times for m < KMG_HISTO_BINS;
// larger multiplicities are appended to big[] (*n_big entries, in no order); *err becomes 2 for a
// multiplicity beyond uint32
struct HistoOut {
    unsigned long long* hist;
    uint32_t* big;
    unsigned long long* n_big;
    uint32_t* err;
};
// histogram request of a hybrid sort: `done` = the finish (fused local sort + re-sorted ranges) produced
// all of it; otherwise the caller histograms the sorted keys after resetting `out`
struct HistoReq {
    HistoOut out;
    bool done;
};
// keys already grouped by the prefix: with bucket_starts == null by the lowest prefix byte only (the keys
// are in d_keys; pb = 24), else by all 16 prefix bits (pb = 16; the keys are in d_keys_alt when in_alt)
// -- plus the histograms of the three top key bytes
struct PrePartitioned {
    int pb;                         // prefix width, 16 or 24
    const unsigned long long* top;  // device [3][256]: bits [2k-24,2k-16), [2k-16,2k-8), [2k-8,2k)
    const unsigned long long* bucket_starts = nullptr;  // device [65537]: first key of every 16-bit bucket, then n
    bool in_alt = false;
};
// extract.cu
size_t top_hist_workspace_bytes();
int extract_top_hist(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k, int rc,
                     const uint8_t* d_lut256, uint64_t* d_counts, unsigned long long* d_top, unsigned long long* d_plan,
                     void* d_ws, size_t ws_bytes, cudaStream_t st);
// histogram of the canonical keys' top byte (d_top_row[256]) and d_counts = valid narrow windows, wide-stream
// windows, both zeroed by the call (12 <= k <= 64)
int extract_canonical_top(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k,
                          const uint8_t* d_lut256, unsigned long long* d_top_row, unsigned long long* d_counts,
                          cudaStream_t st);
// Pre-pass of the fused pipeline (histogram of the top 16 key bits over the valid narrow windows).
// `zeroed` = spill [65536] | top [3][256] | plan [4], zeroed by the call; plan = keys, largest top-byte
// count, valid narrow windows, wide-stream windows.
constexpr size_t P16_ZEROED_WORDS = 65536 + 3 * 256 + 4;
static inline unsigned long long* p16_top(unsigned long long* zeroed) { return zeroed + 65536; }
static inline unsigned long long* p16_plan(unsigned long long* zeroed) { return zeroed + 65536 + 3 * 256; }
// one tile of region_partition: tile.n keys from tile.first on, all in top-byte region tile.region (n = 0: none)
struct RpTile {
    unsigned long long first;
    uint32_t n, region;
};
// keys of one region_partition tile; the tile list of n keys has at most n / tile_keys + 257 entries
uint32_t region_tile_keys(int key_bytes, int val_bytes);
struct Prefix16Out {
    unsigned long long* zeroed;         // [P16_ZEROED_WORDS]
    unsigned long long* region_starts;  // [256] exclusive scan of the top-byte row
    unsigned long long* starts;         // [65537] first key of every 16-bit bucket, then the number of keys
    unsigned long long* cursors;        // [65536] copy of starts[0 .. 65536) (region_partition's cursors)
    uint32_t* rows;                     // prefix16_rows_bytes(): the per-CTA counts
    RpTile* tiles;                      // region_partition's tile list
    uint32_t tile_keys;                 // region_tile_keys() of the keys to come
};
size_t prefix16_rows_bytes();
int extract_prefix16_hist(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k, int rc,
                          const uint8_t* d_lut256, const Prefix16Out& o, cudaStream_t st);
// keys (+ payload) grouped by their top byte -> grouped by their top 16 bits (cursors: Prefix16Out::cursors,
// tiles: Prefix16Out::tiles)
int region_partition(const void* d_keys_in, void* d_keys_out, const void* d_vals_in, void* d_vals_out, uint64_t n,
                     int key_bytes, int val_bytes, const RpTile* d_tiles, unsigned long long* d_cursors, int digit_shift,
                     cudaStream_t st);
int extract_digit_scatter(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k, int rc,
                          const uint8_t* d_lut256, void* d_keys_out, int key_bytes, void* d_vals_out, int val_bytes,
                          uint64_t pos_offset, unsigned long long* d_cursors, int digit_shift, cudaStream_t st);
// radix_sort.cu
bool hybrid_sort_applies(uint64_t n, int key_bytes, int val_bytes, int end_bit, bool pairs_ok);
int hybrid_choose_pb(uint64_t n, unsigned long long max_top_byte_count, int key_bytes, int val_bytes);
int sort_count_core(void* d_keys, void* d_keys_alt, uint64_t n, int key_bytes, int end_bit, const uint64_t* d_hist_in,
                    uint32_t* d_counts_out, uint64_t* d_n_out, int* h_selector_out, void* d_ws, size_t ws_bytes, void* stream,
                    const PrePartitioned* pre, CountRange range = {});
// order-preserving compaction of a count table to the rows in range (kmg_filter_counts); may run in place
int filter_counts(const void* d_keys, const uint32_t* d_counts, uint64_t n, int key_bytes, CountRange range, void* d_keys_out,
                  uint32_t* d_counts_out, uint64_t* d_n_out, void* d_ws, size_t ws_bytes, cudaStream_t st);
int sort_uniq_core(void* d_keys, void* d_keys_alt, void* d_vals, void* d_vals_alt, uint64_t n, int key_bytes, int val_bytes,
                   int end_bit, const uint64_t* d_hist_in, uint64_t* d_n_out, int* h_selector_out, void* d_ws,
                   size_t ws_bytes, void* stream, const PrePartitioned* pre);
int sort_histo_core(void* d_keys, void* d_keys_alt, uint64_t n, int key_bytes, int end_bit, const uint64_t* d_hist_in,
                    const HistoOut& out, void* d_ws, size_t ws_bytes, cudaStream_t st, const PrePartitioned* pre);
void exclusive_scan_256(const unsigned long long* d_hist_row, unsigned long long* d_out, cudaStream_t st);
extern thread_local int64_t g_stat_last_n_out, g_stat_last_err;
// kmg_set_option("time_passes", 1): event pairs around a launch (kind 0 onesweep pass, 1 local sort,
// 2 histogram pre-pass, 3 fused extraction pass)
void timing_begin(cudaStream_t st);
void timing_end(cudaStream_t st, int kind);

// keys an extraction emits per valid window under the strand rule `rc` (kmg.h): two with the reverse
// complement beside every key, one forward-only or canonical
__host__ __device__ constexpr int keys_per_window(int rc) { return rc == KMG_CANONICAL ? 1 : (rc ? 2 : 1); }

// ---- 128-bit key ------------------------------------------------------------------------
struct __align__(16) u128 {
    uint64_t lo, hi;
};

__host__ __device__ __forceinline__ bool operator==(const u128& a, const u128& b) { return a.lo == b.lo && a.hi == b.hi; }
__host__ __device__ __forceinline__ bool operator!=(const u128& a, const u128& b) { return !(a == b); }
__host__ __device__ __forceinline__ bool operator<(const u128& a, const u128& b) {
    return a.hi < b.hi || (a.hi == b.hi && a.lo < b.lo);
}

// ---- 256-bit key: the wide (4-bit code) stream at 33 <= k <= 64 ---------------------------------------
struct __align__(16) u256 {
    u128 lo, hi;
};
__host__ __device__ __forceinline__ bool operator==(const u256& a, const u256& b) { return a.lo == b.lo && a.hi == b.hi; }
__host__ __device__ __forceinline__ bool operator!=(const u256& a, const u256& b) { return !(a == b); }
__host__ __device__ __forceinline__ bool operator<(const u256& a, const u256& b) {
    return a.hi < b.hi || (a.hi == b.hi && a.lo < b.lo);
}

// digit = (key >> shift) & mask ; shift < 8*sizeof(key), digit width <= 16
__device__ __forceinline__ uint32_t key_digit(uint64_t k, int shift, uint32_t mask) {
    return (uint32_t)(k >> shift) & mask;
}
__device__ __forceinline__ uint32_t key_digit(const u128& k, int shift, uint32_t mask) {
    uint64_t v;
    if (shift >= 64) {
        v = k.hi >> (shift - 64);
    } else if (shift == 0) {
        v = k.lo;
    } else {
        v = (k.lo >> shift) | (k.hi << (64 - shift));
    }
    return (uint32_t)v & mask;
}
// (digits of a 256-bit key never straddle its 128-bit halves where this is used: 4-bit symbols)
__device__ __forceinline__ uint32_t key_digit(const u256& k, int shift, uint32_t mask) {
    return shift >= 128 ? key_digit(k.hi, shift - 128, mask) : key_digit(k.lo, shift, mask);
}
__device__ __forceinline__ uint64_t key_all_ones(uint64_t) { return ~0ull; }
__device__ __forceinline__ u128 key_all_ones(u128) { return u128{~0ull, ~0ull}; }

// ---- memory-ordering primitives for decoupled look-back -----------------------------------
__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_u32(uint32_t* p, uint32_t v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_relaxed_u32(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_u32(uint32_t* p, uint32_t v) {
    asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint64_t ld_acquire_u64(const uint64_t* p) {
    uint64_t v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_u64(uint64_t* p, uint64_t v) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint64_t ld_relaxed_u64(const uint64_t* p) {
    uint64_t v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_u64(uint64_t* p, uint64_t v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// A spin that can never hang the GPU: after SPIN_LIMIT polls the kernel raises a device
// error flag and returns garbage; the host turns the flag into KMG_ERR_STATE.
constexpr uint32_t SPIN_LIMIT = 1u << 24;

// ---- 64-bit single-word tile prefix (flag in the top 2 bits, 62-bit value) ----------------
// Used by extract (compaction), select_singletons and format (byte offsets).
constexpr uint64_t TP_FLAG_AGG = 1ull << 62;
constexpr uint64_t TP_FLAG_INCL = 2ull << 62;
constexpr uint64_t TP_VALUE_MASK = (1ull << 62) - 1;

// ---- three-level tile prefix for single-value scans ----------------------------------------------
// Tiles form groups of SC_GROUP consecutive tiles, groups form super-groups of SC_SUPER groups.
// A tile's exclusive prefix is
//   (inclusive prefix of the previous SUPER-GROUP)                       sinc[s-1]   1 word
// + (sums of the earlier groups of its own super-group)                  gsum[..]    <= SC_SUPER-1 words
// + (aggregates of the earlier tiles of its own group)                   agg[..]     <= SC_GROUP-1 words
// Aggregates and group sums depend on nothing but their own tiles, so the only dependency CHAIN is
// sinc[s-1] -> sinc[s]: one link per SC_GROUP * SC_SUPER = 4096 tiles.  (With the chain at group
// level -- one L2 round trip per 128 tiles -- the 190 links of a 24 k-tile launch took as long as the
// whole kernel: 38 % of extract's stall samples sat behind it; a chained or decoupled look-back
// over single tiles is worse still, see profiles/r01_ncu_summary.md.)
// Layout: state[0 .. n_tiles) aggregates | gsum[n_tiles / SC_GROUP + 1] | sinc[...]; zero-initialised;
// tile ids handed out in launch order (atomic ticket).  The flag travels in the word (bit 63).
constexpr uint32_t SC_GROUP = 128;
constexpr uint32_t SC_SUPER = 32;
constexpr uint64_t SC_FLAG = 1ull << 63;
constexpr uint64_t SC_VALUE_MASK = SC_FLAG - 1;

__host__ __device__ __forceinline__ uint64_t sc_groups(uint64_t n_tiles) { return n_tiles / SC_GROUP + 1; }
// words the state array needs for n_tiles tiles
static inline size_t sc_state_words(uint64_t n_tiles) {
    return n_tiles + sc_groups(n_tiles) + sc_groups(n_tiles) / SC_SUPER + 2;
}

__device__ __forceinline__ uint64_t sc_wait(const uint64_t* p, uint64_t w, uint32_t& spins, uint32_t* err_flag) {
    while (!(w & SC_FLAG)) {
        if (++spins > SPIN_LIMIT) {
            atomicExch(err_flag, 1u);
            return SC_FLAG;
        }
        w = ld_relaxed_u64(p);
    }
    return w;
}

// Publish the tile's aggregate (one thread).  Do this as EARLY as the aggregate is known and
// resolve as LATE as possible: the slack is what keeps tiles from waiting for each other.
__device__ __forceinline__ void tile_prefix_publish(uint64_t* state, uint32_t tile, uint64_t aggregate) {
    st_relaxed_u64(&state[tile], SC_FLAG | aggregate);
}

// Called by ALL 32 lanes of ONE warp of the tile, after tile_prefix_publish(); every lane receives
// the exclusive prefix (sum of the aggregates of all earlier tiles).
__device__ __forceinline__ uint64_t tile_prefix_resolve_warp(uint64_t* state, uint32_t n_tiles, uint32_t tile,
                                                             uint64_t aggregate, uint32_t* err_flag) {
    static_assert(SC_SUPER <= 32, "one group sum per lane");
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t g = tile / SC_GROUP, r = tile % SC_GROUP;
    const uint32_t s = g / SC_SUPER, q = g % SC_SUPER;
    uint64_t* gsum = state + n_tiles;
    uint64_t* sinc = gsum + sc_groups(n_tiles);
    uint32_t spins = 0;
    // all loads first, waits afterwards
    uint64_t sv = SC_FLAG, gv = SC_FLAG;
    if (lane == 0 && s > 0) sv = ld_relaxed_u64(&sinc[s - 1]);
    if (lane < q) gv = ld_relaxed_u64(&gsum[g - 1 - lane]);
    uint64_t w[SC_GROUP / 32];
#pragma unroll
    for (int k = 0; k < (int)(SC_GROUP / 32); ++k) {
        const uint32_t j = lane + 1 + 32 * k;
        w[k] = j <= r ? ld_relaxed_u64(&state[tile - j]) : SC_FLAG;
    }
    uint64_t own = 0;  // earlier tiles of the own group
#pragma unroll
    for (int k = 0; k < (int)(SC_GROUP / 32); ++k) {
        const uint32_t j = lane + 1 + 32 * k;
        if (j <= r) w[k] = sc_wait(&state[tile - j], w[k], spins, err_flag);
        own += w[k] & SC_VALUE_MASK;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) own += __shfl_xor_sync(0xffffffffu, own, o);
    // the group's last tile publishes the group sum -- before it waits for anything outside the group
    if (r == SC_GROUP - 1 && lane == 0) st_relaxed_u64(&gsum[g], SC_FLAG | (own + aggregate));
    if (lane < q) gv = sc_wait(&gsum[g - 1 - lane], gv, spins, err_flag);
    if (lane == 0 && s > 0) sv = sc_wait(&sinc[s - 1], sv, spins, err_flag);
    uint64_t outer = (gv & SC_VALUE_MASK) + (sv & SC_VALUE_MASK);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) outer += __shfl_xor_sync(0xffffffffu, outer, o);
    const uint64_t excl = outer + own;
    // ... and the super-group's last tile the chained inclusive prefix
    if (r == SC_GROUP - 1 && q == SC_SUPER - 1 && lane == 0) st_relaxed_u64(&sinc[s], SC_FLAG | (excl + aggregate));
    return excl;
}

// publish + resolve back to back (kernels without useful work to put in between)
__device__ __forceinline__ uint64_t tile_prefix_exclusive_warp(uint64_t* state, uint32_t n_tiles, uint32_t tile,
                                                               uint64_t aggregate, uint32_t* err_flag) {
    if ((threadIdx.x & 31) == 0) tile_prefix_publish(state, tile, aggregate);
    return tile_prefix_resolve_warp(state, n_tiles, tile, aggregate, err_flag);
}

// ---- workspace header ---------------------------------------------------------------------
// Every stage workspace starts with this 256-byte header, zeroed by the host entry point
// before the launch; kmg_ws_status() reads `err` back.
struct WsHeader {
    uint32_t ticket;  // dynamic tile id dispenser
    uint32_t err;     // != 0: a look-back spin hit SPIN_LIMIT (cannot happen on a healthy device)
    uint32_t pad[62];
};
static_assert(sizeof(WsHeader) == 256, "WsHeader must be 256 bytes");

// shared-memory staging index with one padding slot every 16 (8-byte items) / 8 (16-byte)
template <int ITEM_BYTES>
__host__ __device__ __forceinline__ uint32_t pad_idx(uint32_t i) {
    return ITEM_BYTES >= 16 ? i + (i >> 3) : i + (i >> 4);
}

// ---- TMA bulk copy (cp.async.bulk, SASS UBLKCP) + mbarrier ----------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// global -> shared bulk copy through the TMA engine; dst/src 16-byte aligned, bytes a multiple of 16
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// hint: pull a range into L2 ahead of its consumer (no shared memory involved)
__device__ __forceinline__ void tma_prefetch_l2(const void* gmem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gmem_src), "r"(bytes) : "memory");
}

// ---- warp helpers ---------------------------------------------------------------------
__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ uint32_t lanemask_lt() {
    uint32_t m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

template <typename T>
__device__ __forceinline__ T warp_incl_scan(T v) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        T t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane_id() >= (uint32_t)o) v += t;
    }
    return v;
}

// Block-wide exclusive scan of one value per thread; returns exclusive prefix and total.
// `smem` needs (BLOCK/32 + 1) entries of T.  Contains two __syncthreads().
template <int BLOCK, typename T>
__device__ __forceinline__ T block_excl_scan(T v, T* smem, T& total) {
    constexpr int WARPS = BLOCK / 32;
    T incl = warp_incl_scan(v);
    const uint32_t w = threadIdx.x >> 5;
    if (lane_id() == 31) smem[w] = incl;
    __syncthreads();
    if (w == 0) {
        T x = (lane_id() < WARPS) ? smem[lane_id()] : T(0);
        T xi = warp_incl_scan(x);
        if (lane_id() < WARPS) smem[lane_id()] = xi - x;
        if (lane_id() == WARPS - 1) smem[WARPS] = xi;
    }
    __syncthreads();
    total = smem[WARPS];
    return smem[w] + incl - v;
}

}  // namespace kmg
