// K3: HBM-resident stable LSD radix sort ("onesweep": one read + one write of the keys per
// digit pass, chained-scan look-back between tiles instead of a separate scan pass), and
// K5: the range partition used before the multi-GPU exchange (the same kernel with a
// different digit function).
//
// Replaces Batch.sorted (kmermaid/batch.py:156-168: stable sort by sequence string) and the
// ordering work of the n-way heap merge (kmermaid/join.py:63-93).  For equal-length
// upper-case strings the packed integer order equals the string order, and stability keeps
// equal k-mers in emission (position) order exactly like Timsort + heapq.merge do.
//
// Per pass and tile:
//   1. coalesced warp-striped load of ITEMS keys per thread
//   2. per-warp digit ranking with ballot matching into per-warp shared-memory histograms
//   3. block prefix over warps and digits -> tile-local sorted position of every key
//   4. one thread per digit publishes the tile's digit count and looks back over earlier
//      tiles (32-bit word: 2 flag bits + 30-bit count) -> global base of the digit run
//   5. keys (then payload) are reordered through shared memory so that every digit run is
//      written with consecutive threads -> coalesced stores of run-length ~TILE/RADIX keys
#include <cmath>
#include <type_traits>

#include "common.cuh"

namespace kmg {

// ---- digit functions --------------------------------------------------------------------
struct ShiftDigit {
    int shift;
    uint32_t mask;
    template <typename KeyT>
    __device__ __forceinline__ uint32_t operator()(const KeyT& k) const {
        return key_digit(k, shift, mask);
    }
};
// part = ((key >> (key_bits-16)) * n_parts) >> 16
struct RangeDigit {
    int shift;  // key_bits - 16
    uint32_t n_parts;
    template <typename KeyT>
    __device__ __forceinline__ uint32_t operator()(const KeyT& k) const {
        return (key_digit(k, shift, 0xFFFFu) * n_parts) >> 16;
    }
};

// ---- histogram of every pass in one read sweep ---------------------------------------------
template <typename KeyT, int RADIX_BITS>
__global__ void __launch_bounds__(512) radix_hist_kernel(const KeyT* __restrict__ keys, uint64_t n, PassPlan plan,
                                                         unsigned long long* __restrict__ hist) {
    constexpr int RADIX = 1 << RADIX_BITS;
    extern __shared__ uint32_t s_hist[];  // [num_passes][RADIX]
    const int np = plan.num_passes;
    for (int i = threadIdx.x; i < np * RADIX; i += blockDim.x) s_hist[i] = 0;
    __syncthreads();
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const KeyT key = keys[i];
        for (int p = 0; p < np; ++p) {
            const uint32_t d = key_digit(key, plan.shift[p], (1u << plan.bits[p]) - 1u);
            atomicAdd(&s_hist[p * RADIX + d], 1u);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < np * RADIX; i += blockDim.x) {
        const uint32_t c = s_hist[i];
        if (c) atomicAdd(&hist[i], (unsigned long long)c);
    }
}

template <typename KeyT, typename DigitOp>
__global__ void __launch_bounds__(512) digit_hist_kernel(const KeyT* __restrict__ keys, uint64_t n, DigitOp op,
                                                         int radix, unsigned long long* __restrict__ hist) {
    extern __shared__ uint32_t s_hist[];
    for (int i = threadIdx.x; i < radix; i += blockDim.x) s_hist[i] = 0;
    __syncthreads();
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        atomicAdd(&s_hist[op(keys[i])], 1u);
    __syncthreads();
    for (int i = threadIdx.x; i < radix; i += blockDim.x) {
        const uint32_t c = s_hist[i];
        if (c) atomicAdd(&hist[i], (unsigned long long)c);
    }
}

// exclusive scan of each pass' histogram: one warp per pass.  bins[p][d] = sum(hist[p][<d]).
// `counts_out` (optional) receives a copy of the raw histogram of pass 0 (partition sizes).
__global__ void radix_scan_kernel(const unsigned long long* __restrict__ hist, uint64_t* __restrict__ bins,
                                  int radix, int bins_stride, uint64_t* counts_out) {
    const int p = blockIdx.x;
    const unsigned long long* h = hist + (size_t)p * radix;
    uint64_t* b = bins + (size_t)p * bins_stride;
    uint64_t run = 0;
    for (int base = 0; base < radix; base += 32) {
        const int d = base + threadIdx.x;
        const uint64_t c = d < radix ? h[d] : 0;
        if (counts_out && p == 0 && d < radix) counts_out[d] = c;
        const uint64_t incl = warp_incl_scan(c);
        if (d < radix) b[d] = run + incl - c;
        run += __shfl_sync(0xffffffffu, incl, 31);
    }
}

// ---- the onesweep pass ----------------------------------------------------------------------
constexpr uint32_t LB_VALUE_MASK = (1u << 30) - 1;

struct OnesweepParams {
    const void* keys_in;
    void* keys_out;
    const void* vals_in;
    void* vals_out;
    uint32_t n;  // keys in this part (< 2^30)
    const uint64_t* bins_in;  // [RADIX] global base of each digit run for this part
    uint64_t* bins_out;       // [RADIX] base for the next part (may be null)
    uint32_t* lb_agg;         // [tiles][RADIX]   tag | digit count of the tile
    uint32_t* lb_ginc;        // [groups][RADIX]  tag | digit count of all tiles up to the END of the group
    uint32_t* ticket;
    uint32_t* err;
    uint32_t tag;  // (epoch 1..3) << 30: words carrying another tag are "not written yet", so the
                   // arrays need no re-zeroing between the passes of one sort
};

template <int VAL_BYTES>
struct ValType {
    using type = uint64_t;
};
template <>
struct ValType<4> {
    using type = uint32_t;
};

// Two-level look-back.  Tiles form groups of LB_GROUP consecutive tiles.  A tile's exclusive
// prefix = (inclusive prefix of the previous GROUP) + (counts of the earlier tiles of its own
// group).  Tile counts are published early in every tile's life and depend on nothing, so the
// only dependency chain runs over the groups' last tiles, which resolve their prefix EARLY
// (right after publishing their counts): one link per LB_GROUP tiles instead of one per tile.
// Every word carries the launch's 2-bit tag; a word with another tag has not been written yet.
// (group sizes 16 to 48 and prefetch distances 96 to 400 measured within 5 %: profiles/r01_stage_sweep_v15.log)
constexpr uint32_t LB_GROUP = 32;
constexpr int LB_BATCH = 16;           // loads a thread keeps in flight
constexpr uint32_t PREFETCH_TILES = 192;  // L2 prefetch distance in tiles

__device__ __forceinline__ uint32_t lookback_two_level(const uint32_t* __restrict__ lb_agg,
                                                       const uint32_t* __restrict__ lb_ginc, uint32_t tile,
                                                       int d, int radix, uint32_t tag,
                                                       uint32_t* err) {
    const uint32_t g = tile / LB_GROUP, r = tile % LB_GROUP;
    uint32_t excl = 0, spins = 0;
    const uint32_t* gsrc = lb_ginc + (size_t)(g ? g - 1 : 0) * radix + d;
    uint32_t gw = g ? ld_relaxed_u32(gsrc) : tag;  // issued first: it is the one that may lag
    const uint32_t* row = lb_agg + (size_t)tile * radix + d;
    for (uint32_t j0 = 1; j0 <= r; j0 += LB_BATCH) {
        uint32_t w[LB_BATCH];
#pragma unroll
        for (int q = 0; q < LB_BATCH; ++q) w[q] = (j0 + q <= r) ? ld_relaxed_u32(row - (size_t)(j0 + q) * radix) : tag;
#pragma unroll
        for (int q = 0; q < LB_BATCH; ++q) {
            while ((w[q] & ~LB_VALUE_MASK) != tag) {
                if (++spins > SPIN_LIMIT) {
                    atomicExch(err, 1u);
                    w[q] = tag;
                    break;
                }
                w[q] = ld_relaxed_u32(row - (size_t)(j0 + q) * radix);
            }
            excl += w[q] & LB_VALUE_MASK;
        }
    }
    while ((gw & ~LB_VALUE_MASK) != tag) {
        if (++spins > SPIN_LIMIT) {
            atomicExch(err, 1u);
            gw = tag;
            break;
        }
        gw = ld_relaxed_u32(gsrc);
    }
    return excl + (gw & LB_VALUE_MASK);
}

constexpr int OS_BLOCK = 256;  // threads of an onesweep CTA

// How a warp finds the lanes that hold the same digit (phase 3).  The stable ranking alternates per
// item between 8 ballots (ALU) and a shared-memory table of lane masks (LSU).  UNSTABLE: the rank among
// equal digits is the value the histogram atomic returned -- no matching at all.  Only for a pass whose
// order inside a digit does not matter: the first prefix pass of the hybrid finish (the local sort
// orders everything below the prefix).
template <typename KeyT, int VAL_BYTES, int IPT, bool UNSTABLE, typename DigitOp, bool FULL>
__device__ __forceinline__ void onesweep_tile(const OnesweepParams& p, const DigitOp& digit_of, unsigned char* smem_raw,
                                              uint32_t* s_scan, uint64_t* s_bar, const uint32_t tile,
                                              const uint32_t n_valid) {
    constexpr int RADIX_BITS = SORT_RADIX_BITS;
    constexpr int RADIX = SORT_RADIX;
    constexpr int BLOCK = OS_BLOCK;
    constexpr int WARPS = BLOCK / 32;
    constexpr int TILE = BLOCK * IPT;
    // (a partial tile pads with digit RADIX-1 slots that must rank AFTER the real keys: stable path,
    // ballots only -- the unstable kernel has no lane-mask table)
    constexpr bool ATOMIC_RANK = UNSTABLE && FULL;
    static_assert(RADIX <= BLOCK, "one thread per digit in the prefix / look-back phases");
    using ValT = typename ValType<VAL_BYTES>::type;
    constexpr int ITEM_BYTES = sizeof(KeyT) > sizeof(ValT) ? sizeof(KeyT) : sizeof(ValT);

    KeyT* s_keys = reinterpret_cast<KeyT*>(smem_raw);
    ValT* s_vals = reinterpret_cast<ValT*>(smem_raw);
    uint32_t* s_whist = reinterpret_cast<uint32_t*>(smem_raw + (size_t)ITEM_BYTES * TILE);  // [WARPS][RADIX]
    uint32_t* s_tbl = s_whist + WARPS * RADIX;                                               // [WARPS][RADIX] (stable)
    uint64_t* s_goff = reinterpret_cast<uint64_t*>(s_tbl + (UNSTABLE ? 0 : WARPS * RADIX));  // [RADIX]

    const int t = threadIdx.x;
    const uint32_t lane = t & 31, warp = t >> 5;
    const uint32_t n_tiles = gridDim.x;
    const uint32_t tile_base = tile * (uint32_t)TILE;
    uint32_t* my_hist = s_whist + warp * RADIX;
    const uint32_t tag = p.tag;

    // ---- 1. load (warp-striped, coalesced) + per-warp digit histogram ------------------------
    const KeyT* keys_in = reinterpret_cast<const KeyT*>(p.keys_in) + tile_base;
    KeyT keys[IPT];
    const uint32_t wbase = warp * 32 * IPT + lane;
    if constexpr (FULL) {
        // TMA-staged tile: the bulk copies into the (still idle) staging buffer were issued by
        // thread 0 at kernel entry (onesweep_kernel); wait for them, then pick the keys up
        // warp-striped from shared memory (conflict-free)
        mbar_wait(s_bar, 0);
#pragma unroll
        for (int i = 0; i < IPT; ++i) keys[i] = s_keys[wbase + i * 32];
        // (the barriers of phases 1-3 separate these reads from the scatter into the same buffer)
    } else {
#pragma unroll
        for (int i = 0; i < IPT; ++i) {
            const uint32_t idx = wbase + i * 32;
            keys[i] = idx < n_valid ? keys_in[idx] : key_all_ones(KeyT{});
        }
    }
    uint32_t dg[IPT];
#pragma unroll
    for (int i = 0; i < IPT; ++i) {
        const uint32_t idx = wbase + i * 32;
        // slots past the end of a partial tile rank into the last digit, after every real key
        dg[i] = (FULL || idx < n_valid) ? digit_of(keys[i]) : (uint32_t)(RADIX - 1);
        if constexpr (ATOMIC_RANK) dg[i] |= atomicAdd(&my_hist[dg[i]], 1u) << RADIX_BITS;  // digit | rank in the warp
        else atomicAdd(&my_hist[dg[i]], 1u);
    }
    __syncthreads();

    // ---- 2. prefix over warps and digits; publish the tile's digit counts EARLY ----------------
    const uint32_t padding = (uint32_t)TILE - n_valid;
    const int d = t;  // digit owned by this thread in phases 2 and 4 (if < RADIX)
    uint32_t cnt = 0;
    if (d < RADIX) {
        uint32_t run = 0;
#pragma unroll
        for (int w = 0; w < WARPS; ++w) {
            const uint32_t c = s_whist[w * RADIX + d];
            s_whist[w * RADIX + d] = run;
            run += c;
        }
        cnt = run;
        uint32_t c = run;
        if (!FULL && d == RADIX - 1) c -= padding;
        st_relaxed_u32(p.lb_agg + (size_t)tile * RADIX + d, tag | c);
    }
    uint32_t total;
    const uint32_t bin_excl = block_excl_scan<BLOCK, uint32_t>(cnt, s_scan, total);
    const bool group_end = tile % LB_GROUP == LB_GROUP - 1;
    uint32_t excl = 0;
    if (d < RADIX) {
        // fold the digit's tile-local base into every warp's running offset
#pragma unroll
        for (int w = 0; w < WARPS; ++w) s_whist[w * RADIX + d] += bin_excl;
        if (group_end) {  // the chain link: resolve and publish the group's inclusive prefix now
            uint32_t c = cnt;
            if (!FULL && d == RADIX - 1) c -= padding;
            excl = lookback_two_level(p.lb_agg, p.lb_ginc, tile, d, RADIX, tag, p.err);
            st_relaxed_u32(p.lb_ginc + (size_t)(tile / LB_GROUP) * RADIX + d, tag | (excl + c));
        }
    }
    __syncthreads();

    // ---- 3. rank inside the warp; my_hist[] already holds final tile-local offsets, so
    //         slot = offset + rank among the same-digit lanes.  The lanes holding the same digit
    //         are found either with 8 ballots (ALU) or through a shared-memory table of lane
    //         masks (one atomicOr + one load per key, LSU); alternating both keeps either pipe
    //         off its limit (profiles/r01_ncu_summary.md). ----------------------------------------
    uint32_t slot[IPT];
    const uint32_t lt = lanemask_lt();
    const uint32_t my_bit = 1u << lane;
#pragma unroll
    for (int i = 0; i < IPT; ++i) {
        if constexpr (ATOMIC_RANK) {
            slot[i] = my_hist[dg[i] & (RADIX - 1)] + (dg[i] >> RADIX_BITS);
            continue;
        }
        const uint32_t dd = dg[i];
        uint32_t m, cur;
        if (!UNSTABLE && (i & 1)) {
            uint32_t* tbl = s_tbl + warp * RADIX;
            atomicOr(&tbl[dd], my_bit);
            __syncwarp();
            m = tbl[dd];
            cur = my_hist[dd];
            __syncwarp();
            if ((m & lt) == 0) {  // lowest lane of the group
                tbl[dd] = 0;
                my_hist[dd] = cur + __popc(m);
            }
        } else {
            m = 0xffffffffu;
#pragma unroll
            for (int b = 0; b < RADIX_BITS; ++b) {
                const uint32_t bal = __ballot_sync(0xffffffffu, (dd >> b) & 1u);
                m &= bal ^ (((dd >> b) & 1u) - 1u);  // bal where my bit is 1, ~bal where it is 0
            }
            __syncwarp();  // the previous item's leader update is visible
            cur = my_hist[dd];
            __syncwarp();  // everyone has read before the leader overwrites
            if ((m & lt) == 0) my_hist[dd] = cur + __popc(m);
        }
        slot[i] = cur + __popc(m & lt);
    }

    // ---- 4. stage the keys in shared memory; every digit's thread resolves its global base ---------
#pragma unroll
    for (int i = 0; i < IPT; ++i) s_keys[slot[i]] = keys[i];
    if (d < RADIX) {
        uint32_t c = cnt;
        if (!FULL && d == RADIX - 1) c -= padding;
        if (!group_end && tile != 0) excl = lookback_two_level(p.lb_agg, p.lb_ginc, tile, d, RADIX, tag, p.err);
        const uint64_t gbase = p.bins_in[d];
        // destination of local sorted slot s holding digit d:  s_goff[d] + s
        s_goff[d] = gbase + excl - bin_excl;
        if (p.bins_out && tile == n_tiles - 1) p.bins_out[d] = gbase + excl + c;
    }
    __syncthreads();

    // ---- 5. coalesced run writes -----------------------------------------------------------------
    KeyT* keys_out = reinterpret_cast<KeyT*>(p.keys_out);
#pragma unroll
    for (int i = 0; i < IPT; ++i) {
        const uint32_t s = t + i * BLOCK;
        if (FULL || s < n_valid) {
            const KeyT key = s_keys[s];
            const uint32_t dd = digit_of(key);
            dg[i] = dd;
            keys_out[s_goff[dd] + s] = key;
        }
    }
    if constexpr (VAL_BYTES != 0) {
        const ValT* vals_in = reinterpret_cast<const ValT*>(p.vals_in) + tile_base;
        ValT vals[IPT];
#pragma unroll
        for (int i = 0; i < IPT; ++i) {
            const uint32_t idx = wbase + i * 32;
            vals[i] = (FULL || idx < n_valid) ? vals_in[idx] : ValT(0);
        }
        __syncthreads();  // all key reads from the staging buffer are done
#pragma unroll
        for (int i = 0; i < IPT; ++i) s_vals[slot[i]] = vals[i];
        __syncthreads();
        ValT* vals_out = reinterpret_cast<ValT*>(p.vals_out);
#pragma unroll
        for (int i = 0; i < IPT; ++i) {
            const uint32_t s = t + i * BLOCK;
            if (FULL || s < n_valid) vals_out[s_goff[dg[i]] + s] = s_vals[s];
        }
    }
}

// resident CTAs per SM the register allocation aims for
constexpr int min_ctas(int ipt) { return ipt <= 16 ? 3 : 2; }

template <typename KeyT, int VAL_BYTES, int IPT, bool UNSTABLE, typename DigitOp>
__global__ void __launch_bounds__(OS_BLOCK, min_ctas(IPT)) onesweep_kernel(const OnesweepParams p, const DigitOp digit_of) {
    constexpr int RADIX = SORT_RADIX;
    constexpr int BLOCK = OS_BLOCK;
    constexpr int WARPS = BLOCK / 32;
    constexpr int TILE = BLOCK * IPT;
    constexpr int NTBL = UNSTABLE ? 0 : 1;
    using ValT = typename ValType<VAL_BYTES>::type;
    constexpr int ITEM_BYTES = sizeof(KeyT) > sizeof(ValT) ? sizeof(KeyT) : sizeof(ValT);
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint32_t* s_whist = reinterpret_cast<uint32_t*>(smem_raw + (size_t)ITEM_BYTES * TILE);
    __shared__ uint32_t s_scan[WARPS + 1];
    __shared__ uint32_t s_tile;

    __shared__ __align__(8) uint64_t s_bar;
    const int t = threadIdx.x;
    if (t == 0) {
        s_tile = atomicAdd(p.ticket, 1u);
        mbar_init(&s_bar, 1);
        // full tile: start the TMA bulk load of the keys right away, it overlaps the set-up below
        const uint32_t my_tile = s_tile;
        if ((uint64_t)(my_tile + 1) * TILE <= p.n) {
            constexpr uint32_t BYTES = (uint32_t)TILE * sizeof(KeyT);
            constexpr uint32_t CHUNK = 16384;
            mbar_expect_tx(&s_bar, BYTES);
            const char* src = reinterpret_cast<const char*>(p.keys_in) + (size_t)my_tile * BYTES;
            for (uint32_t o = 0; o < BYTES; o += CHUNK)
                tma_load_1d(smem_raw + o, src + o, BYTES - o < CHUNK ? BYTES - o : CHUNK, &s_bar);
            // pull the tile a later CTA will work on into L2 (DRAM has headroom, latency does not)
            const uint64_t ahead = (uint64_t)my_tile + PREFETCH_TILES;
            if ((ahead + 1) * TILE <= p.n) {
                const char* nxt = reinterpret_cast<const char*>(p.keys_in) + (size_t)ahead * BYTES;
                for (uint32_t o = 0; o < BYTES; o += CHUNK) tma_prefetch_l2(nxt + o, BYTES - o < CHUNK ? BYTES - o : CHUNK);
            }
        }
    }
    {   // warp histograms + match tables, 16 bytes per store
        uint4* z = reinterpret_cast<uint4*>(s_whist);
        for (int i = t; i < (1 + NTBL) * WARPS * RADIX / 4; i += BLOCK) z[i] = make_uint4(0, 0, 0, 0);
    }
    __syncthreads();
    const uint32_t tile = s_tile;
    if (t == 0 && tile == gridDim.x - 1) *p.ticket = 0;  // every ticket of this launch is taken
    const uint32_t n_valid = min((uint32_t)TILE, p.n - tile * (uint32_t)TILE);
    if (n_valid == (uint32_t)TILE)
        onesweep_tile<KeyT, VAL_BYTES, IPT, UNSTABLE, DigitOp, true>(p, digit_of, smem_raw, s_scan, &s_bar, tile, n_valid);
    else
        onesweep_tile<KeyT, VAL_BYTES, IPT, UNSTABLE, DigitOp, false>(p, digit_of, smem_raw, s_scan, &s_bar, tile, n_valid);
}

#include "local_sort.cuh"
#include "local_sort_fine.cuh"

template <typename KeyT, int VB, int IPT, bool UNSTABLE>
static size_t onesweep_smem() {
    using ValT = typename ValType<VB>::type;
    const size_t item = sizeof(KeyT) > (VB ? sizeof(ValT) : 0) ? sizeof(KeyT) : sizeof(ValT);
    return item * OS_BLOCK * IPT + (size_t)(UNSTABLE ? 1 : 2) * (OS_BLOCK / 32) * SORT_RADIX * 4 + (size_t)SORT_RADIX * 8;
}

template <typename KeyT, int VB, int IPT, bool UNSTABLE, typename DigitOp>
static int launch_onesweep(const OnesweepParams& p, const DigitOp& op, cudaStream_t st) {
    auto kern = onesweep_kernel<KeyT, VB, IPT, UNSTABLE, DigitOp>;
    const size_t smem = onesweep_smem<KeyT, VB, IPT, UNSTABLE>();
    KMG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const uint32_t tiles = (p.n + OS_BLOCK * IPT - 1) / (OS_BLOCK * IPT);
    kern<<<tiles, OS_BLOCK, smem, st>>>(p, op);
    KMG_LAUNCH_CHECK();
    return KMG_OK;
}

// 8-byte keys: 24 keys per thread (best measured on B200)
template <typename KeyT, int VB>
static int dispatch_tile(bool unstable, const OnesweepParams& p, const ShiftDigit& op, cudaStream_t st) {
    return unstable ? launch_onesweep<KeyT, VB, 24, true>(p, op, st) : launch_onesweep<KeyT, VB, 24, false>(p, op, st);
}
// the partition pass runs once per exchange: one configuration is enough
template <typename KeyT, int VB>
static int dispatch_tile(bool, const OnesweepParams& p, const RangeDigit& op, cudaStream_t st) {
    return launch_onesweep<KeyT, VB, 16, false>(p, op, st);
}

template <typename DigitOp>
static int dispatch_onesweep(bool unstable, int key_bytes, int val_bytes, const OnesweepParams& p, const DigitOp& op,
                             cudaStream_t st) {
    if (key_bytes == 8) {
        if (val_bytes == 0) return dispatch_tile<uint64_t, 0>(unstable, p, op, st);
        if (val_bytes == 4) return dispatch_tile<uint64_t, 4>(unstable, p, op, st);
        return dispatch_tile<uint64_t, 8>(unstable, p, op, st);
    }
    // 16-byte keys: half the items per thread, stable ranking
    if (val_bytes == 0) return launch_onesweep<u128, 0, 8, false>(p, op, st);
    if (val_bytes == 4) return launch_onesweep<u128, 4, 8, false>(p, op, st);
    return launch_onesweep<u128, 8, 8, false>(p, op, st);
}

int g_time_passes = 0;  // kmg_set_option("time_passes", 1): bracket every pass launch with events
thread_local int64_t g_stat_sort_passes = 0;
thread_local int64_t g_stat_hybrid_irregular = -1;

// live per-launch timing of the dominant kernel (bench.py's roofline): event pairs recorded
// on the caller's stream around each onesweep launch, read back by kmg_get_stat().
constexpr int MAX_TIMED = 64;
thread_local cudaEvent_t g_ev[2 * MAX_TIMED];
thread_local int g_ev_made = 0, g_ev_used = 0;
thread_local int g_ev_kind[MAX_TIMED];          // 0: prefix pass (onesweep / region partition), 1: local sort, 2: histogram pre-pass, 3: fused extraction pass
thread_local double g_pass_ms_total[4] = {0, 0, 0, 0};
thread_local int64_t g_pass_count_total[4] = {0, 0, 0, 0};

void timing_collect();
void timing_begin(cudaStream_t st) {
    if (g_time_passes && g_ev_used >= MAX_TIMED) timing_collect();
    if (!g_time_passes || g_ev_used >= MAX_TIMED) return;
    while (g_ev_made < 2 * MAX_TIMED) cudaEventCreate(&g_ev[g_ev_made++]);
    cudaEventRecord(g_ev[2 * g_ev_used], st);
}
void timing_end(cudaStream_t st, int kind) {
    if (!g_time_passes || g_ev_used >= MAX_TIMED) return;
    cudaEventRecord(g_ev[2 * g_ev_used + 1], st);
    g_ev_kind[g_ev_used] = kind;
    ++g_ev_used;
}
// folds the recorded pairs into the running totals (synchronises on the last event)
void timing_collect() {
    for (int i = 0; i < g_ev_used; ++i) {
        float ms = 0;
        if (cudaEventSynchronize(g_ev[2 * i + 1]) == cudaSuccess &&
            cudaEventElapsedTime(&ms, g_ev[2 * i], g_ev[2 * i + 1]) == cudaSuccess) {
            g_pass_ms_total[g_ev_kind[i]] += ms;
            ++g_pass_count_total[g_ev_kind[i]];
        }
    }
    g_ev_used = 0;
}
double timing_total_ms(int kind) { return g_pass_ms_total[kind]; }
int64_t timing_count(int kind) { return g_pass_count_total[kind]; }
void timing_reset() {
    g_ev_used = 0;
    for (int i = 0; i < 4; ++i) {
        g_pass_ms_total[i] = 0;
        g_pass_count_total[i] = 0;
    }
}

// keys per look-back part: 30-bit counts, multiple of every tile size (lcm of tiles | 2^k*3)
constexpr uint64_t PART_MAX = ((1ull << 30) - 1) / (4096ull * 3 * 3 * 5) * (4096ull * 3 * 3 * 5);

struct SortWs {
    WsHeader* hdr;
    unsigned long long* hist;  // [MAX_PASSES][RADIX]
    uint64_t* bins;            // [MAX_PASSES][2][RADIX]
    uint32_t* lookback;        // [tiles_per_part][RADIX] tile counts, then [groups][RADIX] group prefixes
    size_t lb_words;           // words of the tile-count array
    // hybrid finish (see local_sort_kernel); all null / 0 when the sort cannot take it
    bool hybrid;
    uint64_t* hyb_bounds;      // [n / LS_T_MIN + 2] tile bounds
    uint32_t* hyb_flag;        // [n / LS_T_MIN + 2] irregular tiles
    uint64_t* hyb_off;         // [n / LS_T_MIN + 2] their offsets in the gather buffer
    uint64_t* hyb_state;       // tile prefix state of the fused count (sc_state_words(n / LS_T_MIN + 2))
    size_t zero_bytes;         // everything up to here is zeroed at the start of a sort
    uint64_t irr_cap;          // keys the gather buffers hold
    void* irr_buf[2];          // gather buffer + its ping-pong partner (irr_cap keys each)
    void* irr_vbuf[2];         // the same for the payload (payload sorts)
    void* irr_ws;              // workspace of the sort of the gathered keys
    size_t irr_ws_bytes;
    size_t total;
};

int g_hybrid = 1;     // kmg_set_option("hybrid", 0/1)
int g_local_tile = 7936;  // kmg_set_option("local_tile", positions): target tile width of the local sort
int g_count_fused = 1;  // kmg_set_option("count_fused", 0/1): let the hybrid finish emit the count table itself
int g_hybrid_pb = 0;  // kmg_set_option("hybrid_pb", 0 | 16 | 24): force the prefix width (0 = by n and skew)
constexpr uint64_t HYBRID_MIN_N = 1ull << 20;
constexpr uint64_t HYBRID_MAX_N = 1ull << 33;  // 32-bit tile ids at the smallest tile width

// Key-only sorts (8- or 16-byte keys) over bits [0, end_bit), end_bit >= 32, of 2^20 .. 2^33 keys.
static bool hybrid_applies(uint64_t n, int key_bytes, int val_bytes, int begin_bit, int end_bit, bool pairs_ok = false);

static SortWs carve_sort_ws(void* ws, uint64_t n, int key_bytes, bool hybrid, int val_bytes = 0) {
    SortWs w;
    memset(&w, 0, sizeof(w));
    char* p = (char*)ws;
    w.hdr = (WsHeader*)p;
    p += sizeof(WsHeader);
    w.hist = (unsigned long long*)p;
    p += sizeof(uint64_t) * MAX_PASSES * SORT_RADIX;
    w.bins = (uint64_t*)p;
    p += sizeof(uint64_t) * MAX_PASSES * 2 * SORT_RADIX;
    w.lookback = (uint32_t*)p;
    const uint64_t part = n < PART_MAX ? n : PART_MAX;
    const uint64_t min_tile = key_bytes == 16 ? 2048 : 4096;  // smallest tile of any configuration
    const uint64_t tiles = (part + min_tile - 1) / min_tile + 1;
    w.lb_words = align_up(tiles * SORT_RADIX * sizeof(uint32_t), 256) / sizeof(uint32_t);
    p += w.lb_words * sizeof(uint32_t) + align_up((tiles / LB_GROUP + 2) * SORT_RADIX * sizeof(uint32_t), 256);
    w.hybrid = hybrid;
    if (hybrid) {
        const uint64_t lt = n / LS_T_MIN + 2;
        w.hyb_flag = (uint32_t*)p;
        p += align_up(lt * sizeof(uint32_t), 256);
        w.hyb_state = (uint64_t*)p;
        p += align_up(sc_state_words(lt) * sizeof(uint64_t), 256);
    }
    w.zero_bytes = p - (char*)ws;
    if (hybrid) {
        const uint64_t lt = n / LS_T_MIN + 2;
        w.hyb_bounds = (uint64_t*)p;
        p += align_up(lt * sizeof(uint64_t), 256);
        w.hyb_off = (uint64_t*)p;
        p += align_up(lt * sizeof(uint64_t), 256);
        // irregular tiles are re-sorted through a side buffer of n / 8 keys (beyond that the whole
        // sort falls back to the plain passes)
        w.irr_cap = std::max<uint64_t>(n / 8, 1ull << 16);
        for (int i = 0; i < 2; ++i) {
            w.irr_buf[i] = p;
            p += align_up(w.irr_cap * (size_t)key_bytes, 256);
        }
        for (int i = 0; i < 2 && val_bytes; ++i) {
            w.irr_vbuf[i] = p;
            p += align_up(w.irr_cap * (size_t)val_bytes, 256);
        }
        w.irr_ws = p;
        w.irr_ws_bytes = carve_sort_ws(nullptr, w.irr_cap, key_bytes, false).total;
        p += align_up(w.irr_ws_bytes, 256);
    }
    w.total = p - (char*)ws;
    return w;
}

// Payload sorts take it only when the caller does not need equal keys in input order (`pairs_ok`:
// kmg_sort_uniq).
static bool hybrid_applies(uint64_t n, int key_bytes, int val_bytes, int begin_bit, int end_bit, bool pairs_ok) {
    if (val_bytes != 0 && !pairs_ok) return false;
    return g_hybrid && begin_bit == 0 && end_bit >= 32 && n >= HYBRID_MIN_N && n <= HYBRID_MAX_N;
}

thread_local int64_t g_stat_hybrid_path = 0;  // 0 plain passes, 1 hybrid, 2 hybrid + re-sorted ranges, 3 fell back
thread_local int64_t g_stat_hybrid_big_runs = -1;
// what the last hybrid sort of this thread already read back when it synchronised (-1: nothing):
// callers that would otherwise read the status word / the result count again can skip their own sync
thread_local int64_t g_stat_last_n_out = -1;
thread_local int64_t g_stat_last_err = -1;

// header words of a sort workspace used by the hybrid finish (all inside WsHeader::pad, zeroed with it)
//   pad[0..1] irregular tiles   pad[2..3] runs the block had to sort   pad[4] tile ticket of the fused launch
//   pad[6..7] oversize tiles    pad[8..9] keys in oversize tiles       pad[10..11] copy of the fused result count
struct HybridHeaderView {
    uint32_t ticket, err;
    unsigned long long irregular, big_runs;
    uint32_t ls_ticket, pad5;
    unsigned long long over_tiles, over_keys, n_out;
};
static_assert(sizeof(HybridHeaderView) == 56, "layout of the header words");

// `hybrid` = the workspace was carved for (and the call may take) the hybrid finish
// A 16-bit prefix is enough (two passes instead of three) in two situations, judged by the fullest top
// byte (real genomes are skewed enough to need the third pass early):
//  * its buckets stay well under a tile, so that a tile holds a window of a few buckets plus the
//    straddling one (capacity / 2.4);
//  * the keys are spread evenly (fullest top byte within 4 % of the mean, e.g. random sequence) and ONE
//    bucket fits a tile with 6 sigma to spare: every tile then owns exactly one bucket (the windows are
//    made narrower than the smallest bucket, see tile_width).  This is config 3 on 8 GPUs: 387 M keys
//    per rank, buckets of 5913 -- one pass fewer (0.5 ms per 100 M keys) for tiles that are 72 % full.
static int hybrid_tile_cap(int key_bytes, int val_bytes) {
    return key_bytes == 16 ? (val_bytes ? ls_cap<u128, true>() : ls_cap<u128, false>())
                           : (val_bytes ? ls_cap<uint64_t, true>() : ls_cap<uint64_t, false>());
}
static bool hybrid_pb16_ok(uint64_t n, unsigned long long max_top_byte_count, int key_bytes, int val_bytes) {
    // (16-byte keys: tiles of 4096; measured at 100 M keys, k = 63: buckets of 1526 fill a tile to 37 % and
    // the local sort takes 2.57 ms against 1.56 ms + a 0.84 ms pass with the 24-bit prefix)
    const unsigned long long fullest = max_top_byte_count / 256;  // expected size of the largest 16-bit bucket
    if (fullest <= (unsigned long long)(key_bytes == 16 ? 800 : (val_bytes ? 2500 : 3400))) return true;
    if (key_bytes == 16) return false;
    const double avg = (double)n / 65536.0;
    return (double)fullest <= 1.04 * avg && avg + 6.0 * std::sqrt(avg) <= (double)hybrid_tile_cap(key_bytes, val_bytes) - 64.0;
}
int hybrid_choose_pb(uint64_t n, unsigned long long max_top_byte_count, int key_bytes, int val_bytes) {
    if (g_hybrid_pb == 16 || g_hybrid_pb == 24) return g_hybrid_pb;
    return hybrid_pb16_ok(n, max_top_byte_count, key_bytes, val_bytes) ? 16 : 24;
}

// `pre` (fused pipeline): the keys in d_keys are ALREADY grouped by the lowest prefix byte (the first,
// order-free prefix pass ran inside the extraction kernel); pre->top holds the histograms of the
// three top key bytes and pre->pb the prefix width the caller chose.  With pre->bucket_starts the keys
// are grouped by the whole 16-bit prefix (top byte in the extraction, byte 2 in region_partition_kernel):
// no pass runs here at all.
static int sort_impl(void* d_keys, void* d_keys_alt, void* d_vals, void* d_vals_alt, uint64_t n, int key_bytes,
                     int val_bytes, int begin_bit, int end_bit, const uint64_t* d_hist_in, int* h_selector_out,
                     void* d_ws, size_t ws_bytes, cudaStream_t st, bool hybrid, bool allow_hybrid,
                     CountOut* co = nullptr, const PrePartitioned* pre = nullptr) {
    SortWs w = carve_sort_ws(d_ws, n, key_bytes, hybrid, val_bytes);
    KMG_REQUIRE(ws_bytes >= w.total, KMG_ERR_WS, "sort workspace too small: %zu < %zu", ws_bytes, w.total);
    hybrid = hybrid && allow_hybrid;
    KMG_REQUIRE(!pre || hybrid, KMG_ERR_ARG, "pre-partitioned keys need the hybrid finish");
    // (all prefix bits done: no pass runs here, the local sort takes its tile bounds from the bucket starts)
    const bool prefix_done = pre && pre->bucket_starts;
    KMG_REQUIRE(!prefix_done || pre->pb == 16, KMG_ERR_ARG, "bucket starts come with the 16-bit prefix");

    PassPlan plan = make_plan(begin_bit, end_bit);
    int np = plan.num_passes;
    const uint64_t n_parts = (n + PART_MAX - 1) / PART_MAX;

    // header + hist zero; look-back words zero once per sort -- see OnesweepParams::tag
    KMG_CUDA(cudaMemsetAsync(d_ws, 0, w.zero_bytes, st));

    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);

    // Hybrid finish: ordinary passes over the top pb = 16 or 24 bits only, then local_sort_kernel
    // orders everything below them.  The histograms of the three top bytes come from kmg_extract
    // (d_hist_in rows 13..15) or from one sweep; the top byte's tells how skewed the keys are.
    const unsigned long long* hist = w.hist;
    int pb = 0;
    if (hybrid) {
        memset(&plan, 0, sizeof(plan));
        plan.num_passes = 3;
        for (int i = 0; i < 3; ++i) {
            plan.shift[i] = end_bit - 24 + 8 * i;
            plan.bits[i] = 8;
        }
        if (pre) {
            if (!prefix_done)  // (only the passes below read the rows)
                KMG_CUDA(cudaMemcpyAsync(w.hist, pre->top, (size_t)3 * SORT_RADIX * sizeof(uint64_t), cudaMemcpyDeviceToDevice, st));
        } else if (d_hist_in && key_bytes == 8 && (end_bit & 1) == 0) {
            KMG_CUDA(cudaMemcpyAsync(w.hist, d_hist_in + (size_t)13 * SORT_RADIX, (size_t)3 * SORT_RADIX * sizeof(uint64_t),
                                     cudaMemcpyDeviceToDevice, st));
        } else {
            const int grid = (int)std::min<uint64_t>((n + 511) / 512, (uint64_t)sms * 4);
            if (key_bytes == 8)
                radix_hist_kernel<uint64_t, SORT_RADIX_BITS><<<grid, 512, 3 * SORT_RADIX * sizeof(uint32_t), st>>>(
                    (const uint64_t*)d_keys, n, plan, w.hist);
            else
                radix_hist_kernel<u128, SORT_RADIX_BITS><<<grid, 512, 3 * SORT_RADIX * sizeof(uint32_t), st>>>(
                    (const u128*)d_keys, n, plan, w.hist);
            KMG_LAUNCH_CHECK();
        }
        pb = pre ? pre->pb : (g_hybrid_pb == 16 || g_hybrid_pb == 24 ? g_hybrid_pb : 0);
        if (!pb) {
            // 16-bit or 24-bit prefix: see hybrid_pb16_ok (needs the top byte's histogram on the host)
            pb = 24;
            if (n <= (1ull << 29)) {
                unsigned long long h_top[SORT_RADIX];
                KMG_CUDA(cudaMemcpyAsync(h_top, w.hist + 2 * SORT_RADIX, sizeof(h_top), cudaMemcpyDeviceToHost, st));
                KMG_CUDA(cudaStreamSynchronize(st));
                unsigned long long mx = 0;
                for (int i = 0; i < SORT_RADIX; ++i) mx = std::max(mx, h_top[i]);
                if (hybrid_pb16_ok(n, mx, key_bytes, val_bytes)) pb = 16;
            }
        }
        np = pb / 8;
        // passes run over rows [3 - np, 3) of the three-byte plan
        for (int i = 0; i < np; ++i) plan.shift[i] = end_bit - pb + 8 * i;
        plan.num_passes = np;
        hist = w.hist + (size_t)(3 - np) * SORT_RADIX;
    } else if (d_hist_in) {
        // digit histograms of exactly these keys and this plan, produced by kmg_extract
        hist = reinterpret_cast<const unsigned long long*>(d_hist_in);
    } else {
        const int grid = (int)std::min<uint64_t>((n + 511) / 512, (uint64_t)sms * 4);
        const size_t smem = (size_t)np * SORT_RADIX * sizeof(uint32_t);
        if (key_bytes == 8)
            radix_hist_kernel<uint64_t, SORT_RADIX_BITS><<<grid, 512, smem, st>>>((const uint64_t*)d_keys, n, plan, w.hist);
        else
            radix_hist_kernel<u128, SORT_RADIX_BITS><<<grid, 512, smem, st>>>((const u128*)d_keys, n, plan, w.hist);
        KMG_LAUNCH_CHECK();
    }
    if (!prefix_done) {
        radix_scan_kernel<<<np, 32, 0, st>>>(hist, w.bins, SORT_RADIX, 2 * SORT_RADIX, nullptr);
        KMG_LAUNCH_CHECK();
    }

    char* kin = (char*)d_keys;
    char* kout = (char*)d_keys_alt;
    char* vin = (char*)d_vals;
    char* vout = (char*)d_vals_alt;
    if (prefix_done) {
        if (pre->in_alt) {
            std::swap(kin, kout);
            std::swap(vin, vout);
        }
        ++g_stat_sort_passes;  // the caller's region partition: the one prefix pass after the fused extraction
    }
    uint32_t launch = 0;
    for (int pass = prefix_done ? np : (pre ? 1 : 0); pass < np; ++pass) {
        const ShiftDigit op{plan.shift[pass], (1u << plan.bits[pass]) - 1u};
        for (uint64_t part = 0; part < n_parts; ++part) {
            const uint64_t off = part * PART_MAX;
            OnesweepParams p;
            p.keys_in = kin + off * key_bytes;
            p.keys_out = kout;
            p.vals_in = vin ? vin + off * val_bytes : nullptr;
            p.vals_out = vout;
            p.n = (uint32_t)std::min<uint64_t>(PART_MAX, n - off);
            uint64_t* bins = w.bins + (size_t)pass * 2 * SORT_RADIX;
            p.bins_in = bins + (part & 1) * SORT_RADIX;
            p.bins_out = (part + 1 < n_parts) ? bins + ((part + 1) & 1) * SORT_RADIX : nullptr;
            p.lb_agg = w.lookback;
            p.lb_ginc = w.lookback + w.lb_words;
            p.ticket = &w.hdr->ticket;
            p.err = &w.hdr->err;
            if (n_parts > 1) {
                // tile counts differ between parts, so stale words could alias: re-zero
                if (launch > 0)
                    KMG_CUDA(cudaMemsetAsync(w.lookback, 0, (char*)d_ws + w.zero_bytes - (char*)w.lookback, st));
                p.tag = 1u << 30;
            } else {
                // every word is rewritten by every launch, so a 3-cycle of tags tells the
                // current launch's words from the two previous launches' (and from zero)
                p.tag = (launch % 3u + 1u) << 30;
            }
            if (g_ev_used >= MAX_TIMED) timing_collect();
            timing_begin(st);
            // the hybrid finish does not care about the order inside the first pass' digits
            int rcode = dispatch_onesweep(hybrid && pass == 0, key_bytes, val_bytes, p, op, st);
            timing_end(st, 0);
            if (rcode != KMG_OK) return rcode;
            ++launch;
        }
        std::swap(kin, kout);
        std::swap(vin, vout);
        ++g_stat_sort_passes;
    }
    if (!hybrid) {
        *h_selector_out = np & 1;
        return KMG_OK;
    }

    // kin now holds the keys ordered by their top pb bits; finish into kout
    const bool wide_key = key_bytes == 16;
    const bool pairs = val_bytes != 0;
    const int cap = wide_key ? (pairs ? ls_cap<u128, true>() : ls_cap<u128, false>())
                             : (pairs ? ls_cap<uint64_t, true>() : ls_cap<uint64_t, false>());
    HybridParams hp;
    memset(&hp, 0, sizeof(hp));
    hp.keys_in = kin;
    hp.keys_out = kout;
    hp.vals_in = vin;
    hp.vals_out = vout;
    hp.n = n;
    // Tile width: a tile owns WHOLE prefix buckets, so leave room for the straddling one; with a
    // 16-bit prefix the buckets are a sizeable fraction of a tile and a width of k average buckets
    // gives (for evenly filled buckets) every tile the same k buckets instead of k-1 or k
    const double avg = (double)n / (double)(1ull << pb);  // average prefix bucket
    auto tile_width = [&](double want) {
        // (one bucket per tile: windows narrower than the smallest bucket, so that none holds two starts)
        if (avg > cap / 2.4) return (uint32_t)std::max<double>(LS_T_MIN, std::min<double>(cap - 256, avg - 6.0 * std::sqrt(avg) - 8.0));
        double target = std::min<double>(want, cap - std::max(256.0, 1.35 * avg));
        target = std::max<double>(target, LS_T_MIN);
        if (avg < 64) return (uint32_t)target;
        const int kbk = std::max(1, (int)(target / avg));
        return (uint32_t)std::min<double>(cap - 256, std::max<double>(LS_T_MIN, std::ceil(kbk * avg)));
    };
    hp.bounds = w.hyb_bounds;
    hp.flag = w.hyb_flag;
    hp.off = w.hyb_off;
    hp.key_bits = end_bit;
    hp.pb = pb;
    HybridHeaderView* hv = reinterpret_cast<HybridHeaderView*>(w.hdr);
    hp.irregular = &hv->irregular;  // [0] irregular tiles, [1] runs sorted by the block
    hp.over = &hv->over_tiles;      // [0] oversize tiles, [1] their keys
    hp.n_out_copy = &hv->n_out;
    hp.tile_state = w.hyb_state;
    hp.ticket = &hv->ls_ticket;
    hp.err = &w.hdr->err;
    // The persistent fine-cell kernel wins wherever a tile holds several prefix buckets.  With about ONE bucket
    // per tile (a 16-bit prefix under more than ~160 M evenly spread keys: config 3 on 8 GPUs, 387.5 M keys per
    // rank) its tile prefix jams -- 70 % of the warp samples sit behind warp 0's look-back polls, 28 ms against
    // the first kernel's 4.3 ms (profiles/r02_local_sort_one_bucket_tiles.md) -- so tiles narrower than two
    // average buckets keep the first kernel.
    const double avg_bucket = (double)n / (double)(1ull << pb);
    const bool few_bucket_tiles =
        avg_bucket > cap / 2.4 ||
        (avg_bucket >= 64 && std::min<double>(g_local_tile, cap - std::max(256.0, 1.35 * avg_bucket)) < 2.0 * avg_bucket);
    const bool fine = !few_bucket_tiles;
    const size_t smem = fine ? (wide_key ? (pairs ? lsf_smem_bytes<u128, true>() : lsf_smem_bytes<u128, false>())
                                         : (pairs ? lsf_smem_bytes<uint64_t, true>() : lsf_smem_bytes<uint64_t, false>()))
                             : (wide_key ? (pairs ? ls_smem_bytes<u128, true>() : ls_smem_bytes<u128, false>())
                                         : (pairs ? ls_smem_bytes<uint64_t, true>() : ls_smem_bytes<uint64_t, false>()));
    const int sel_in = kin == (char*)d_keys ? 0 : 1;  // where the prefix-ordered keys are
    const int sel_done = sel_in ^ 1;                   // ... and where the finish puts its result
    const bool want_fused = co != nullptr && g_count_fused;

    auto launch_bounds = [&](uint32_t T) -> int {
        hp.tile_t = T;
        hp.n_tiles = (uint32_t)((n + T - 1) / T);
        if (prefix_done) bounds_from_starts_kernel<<<(hp.n_tiles + 1 + 255) / 256, 256, 0, st>>>(hp, pre->bucket_starts, 1u << pb);
        else if (wide_key) tile_bounds_kernel<u128><<<(hp.n_tiles + 1 + 7) / 8, 256, 0, st>>>(hp);
        else tile_bounds_kernel<uint64_t><<<(hp.n_tiles + 1 + 7) / 8, 256, 0, st>>>(hp);
        KMG_LAUNCH_CHECK();
        // tiles that own more keys than the local sort holds (huge prefix buckets: repeats) are known
        // from the bounds alone; the fused launch reads the count from device memory and stands
        // down when there are any (its table would be void), so no host round trip sits between
        KMG_CUDA(cudaMemsetAsync(hp.over, 0, 2 * sizeof(unsigned long long), st));
        oversize_tiles_kernel<<<(hp.n_tiles + 255) / 256, 256, 0, st>>>(hp, (uint32_t)cap, hp.over);
        KMG_LAUNCH_CHECK();
        return KMG_OK;
    };
    auto launch_local = [&](bool fused) -> int {
        hp.counts_out = fused ? co->counts : nullptr;
        hp.n_out = fused ? co->n_out : nullptr;
        if (g_ev_used >= MAX_TIMED) timing_collect();
        timing_begin(st);
#define KMG_LS_LAUNCH(K, E, V)                                                                                   \
    do {                                                                                                         \
        auto kern = fine ? local_sort_fine_kernel<K, E, V> : local_sort_kernel<K, E, V>;                         \
        KMG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));            \
        /* (the fine-cell kernel is persistent: two CTAs per SM take tiles from a ticket) */                     \
        kern<<<fine ? std::min<uint32_t>(hp.n_tiles, 2u * (uint32_t)sms) : hp.n_tiles, LS_BLOCK, smem, st>>>(hp); \
    } while (0)
        if (fused && pairs && wide_key) {
            if (val_bytes == 4) KMG_LS_LAUNCH(u128, 2, 4);
            else KMG_LS_LAUNCH(u128, 2, 8);
        } else if (fused && pairs) {
            if (val_bytes == 4) KMG_LS_LAUNCH(uint64_t, 2, 4);
            else KMG_LS_LAUNCH(uint64_t, 2, 8);
        } else if (fused) {
            if (wide_key) KMG_LS_LAUNCH(u128, 1, 0);
            else KMG_LS_LAUNCH(uint64_t, 1, 0);
        } else if (pairs && wide_key) {
            if (val_bytes == 4) KMG_LS_LAUNCH(u128, 0, 4);
            else KMG_LS_LAUNCH(u128, 0, 8);
        } else if (pairs) {
            if (val_bytes == 4) KMG_LS_LAUNCH(uint64_t, 0, 4);
            else KMG_LS_LAUNCH(uint64_t, 0, 8);
        } else {
            if (wide_key) KMG_LS_LAUNCH(u128, 0, 0);
            else KMG_LS_LAUNCH(uint64_t, 0, 0);
        }
#undef KMG_LS_LAUNCH
        timing_end(st, 1);
        KMG_LAUNCH_CHECK();
        return KMG_OK;
    };
    // ONE read-back per attempt: everything the host needs to know about it
    HybridHeaderView hh;
    auto read_header = [&]() -> int {
        KMG_CUDA(cudaMemcpyAsync(&hh, w.hdr, sizeof(hh), cudaMemcpyDeviceToHost, st));
        KMG_CUDA(cudaStreamSynchronize(st));
        g_stat_hybrid_irregular = (int64_t)hh.irregular;
        g_stat_hybrid_big_runs = (int64_t)hh.big_runs;
        g_stat_last_err = (int64_t)hh.err;
        return KMG_OK;
    };

    // First attempt at the widest tiles: the fused emission when the caller asked for one, else the sort.
    int rcode = launch_bounds(tile_width(g_local_tile));
    if (rcode != KMG_OK) return rcode;
    rcode = launch_local(want_fused);
    if (rcode != KMG_OK) return rcode;
    rcode = read_header();
    if (rcode != KMG_OK) return rcode;
    g_stat_hybrid_path = 1;
    if (hh.irregular == 0 && (!want_fused || hh.over_tiles == 0)) {
        if (want_fused) {
            co->done = true;
            g_stat_last_n_out = (int64_t)hh.n_out;
        }
        *h_selector_out = sel_done;
        return KMG_OK;
    }
    // Some tiles own more keys than the local scheme holds (a huge prefix bucket: repeats) or crowd
    // too many distinct keys into one cell.  The keys get sorted (no fused emission: the caller
    // follows up with kmg_rle_count / kmg_select_singletons), the irregular tiles' ranges are
    // gathered, sorted with the plain passes and put back.
    if (want_fused || hh.over_keys > n / 32) {
        // The widest tiles are the fastest, but a tile owns WHOLE buckets: with big buckets around
        // (repeat families: thousands of keys per 12-mer prefix) wide tiles overflow.  Take the widest
        // candidate width that leaves at most n/32 keys in oversize tiles.
        const uint32_t cand[3] = {tile_width(g_local_tile), tile_width(cap / 2), tile_width(cap / 4)};
        if (hh.over_keys > n / 32) {
            for (int c = 1; c < 3; ++c) {
                if (cand[c] >= cand[c - 1]) continue;
                rcode = launch_bounds(cand[c]);
                if (rcode != KMG_OK) return rcode;
                rcode = read_header();
                if (rcode != KMG_OK) return rcode;
                if (hh.over_keys <= n / 32) break;
            }
        }
        KMG_CUDA(cudaMemsetAsync(hp.irregular, 0, 2 * sizeof(unsigned long long), st));
        KMG_CUDA(cudaMemsetAsync(hp.flag, 0, (size_t)(n / LS_T_MIN + 2) * sizeof(uint32_t), st));
        rcode = launch_local(false);
        if (rcode != KMG_OK) return rcode;
        rcode = read_header();
        if (rcode != KMG_OK) return rcode;
        if (hh.irregular == 0) {
            *h_selector_out = sel_done;
            return KMG_OK;
        }
    }
    irregular_scan_kernel<<<1, 1024, 0, st>>>(hp);
    KMG_LAUNCH_CHECK();
    unsigned long long m_irr = 0;
    KMG_CUDA(cudaMemcpyAsync(&m_irr, hp.off + hp.n_tiles, sizeof(m_irr), cudaMemcpyDeviceToHost, st));
    KMG_CUDA(cudaStreamSynchronize(st));
    if (m_irr <= w.irr_cap) {
        g_stat_hybrid_path = 2;
        const int grid = (int)std::min<uint64_t>(hp.n_tiles, (uint64_t)sms * 8);
        int rc2 = irregular_copy<true>(hp, key_bytes, kin, nullptr, w.irr_buf[0], grid, st);
        if (rc2 == KMG_OK && pairs) rc2 = irregular_copy<true>(hp, val_bytes, vin, nullptr, w.irr_vbuf[0], grid, st);
        if (rc2 != KMG_OK) return rc2;
        int sel2 = 0;
        const int64_t passes = g_stat_sort_passes;
        rcode = sort_impl(w.irr_buf[0], w.irr_buf[1], pairs ? w.irr_vbuf[0] : nullptr, pairs ? w.irr_vbuf[1] : nullptr,
                          m_irr, key_bytes, val_bytes, 0, end_bit, nullptr, &sel2, w.irr_ws, w.irr_ws_bytes, st, false,
                          false);
        g_stat_sort_passes = passes;
        if (rcode != KMG_OK) return rcode;
        rc2 = irregular_copy<false>(hp, key_bytes, nullptr, kout, w.irr_buf[sel2], grid, st);
        if (rc2 == KMG_OK && pairs) rc2 = irregular_copy<false>(hp, val_bytes, nullptr, vout, w.irr_vbuf[sel2], grid, st);
        if (rc2 != KMG_OK) return rc2;
        *h_selector_out = sel_done;
        return KMG_OK;
    }
    g_stat_hybrid_path = 3;
    int sel2 = 0;
    rcode = sort_impl(kin, kout, vin, vout, n, key_bytes, val_bytes, begin_bit, end_bit, nullptr, &sel2, d_ws, ws_bytes, st,
                      true, false);
    if (rcode != KMG_OK) return rcode;
    *h_selector_out = sel_in ^ sel2;
    return KMG_OK;
}

// exclusive scan of one 256-bin histogram row (the cursors of the fused first prefix pass)
void exclusive_scan_256(const unsigned long long* d_hist_row, unsigned long long* d_out, cudaStream_t st) {
    radix_scan_kernel<<<1, 32, 0, st>>>(d_hist_row, reinterpret_cast<uint64_t*>(d_out), SORT_RADIX, SORT_RADIX, nullptr);
    bump_launches();
}

bool hybrid_sort_applies(uint64_t n, int key_bytes, int val_bytes, int end_bit, bool pairs_ok) {
    return hybrid_applies(n, key_bytes, val_bytes, 0, end_bit, pairs_ok);
}
}  // namespace kmg

using namespace kmg;

extern "C" size_t kmg_radix_sort_workspace_bytes(uint64_t n, int key_bytes, int val_bytes, int begin_bit,
                                                 int end_bit) {
    return carve_sort_ws(nullptr, n, key_bytes, hybrid_applies(n, key_bytes, val_bytes, begin_bit, end_bit)).total;
}

extern "C" int kmg_radix_sort(void* d_keys, void* d_keys_alt, void* d_vals, void* d_vals_alt, uint64_t n,
                              int key_bytes, int val_bytes, int begin_bit, int end_bit, const uint64_t* d_hist_in,
                              int* h_selector_out, void* d_ws, size_t ws_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    KMG_REQUIRE(key_bytes == 8 || key_bytes == 16, KMG_ERR_ARG, "key_bytes must be 8 or 16");
    KMG_REQUIRE(val_bytes == 0 || val_bytes == 4 || val_bytes == 8, KMG_ERR_ARG, "val_bytes must be 0, 4 or 8");
    KMG_REQUIRE(begin_bit >= 0 && end_bit <= key_bytes * 8 && begin_bit <= end_bit, KMG_ERR_ARG,
                "bad bit range [%d,%d)", begin_bit, end_bit);
    KMG_REQUIRE(h_selector_out, KMG_ERR_ARG, "h_selector_out is null");
    KMG_REQUIRE((val_bytes == 0) == (d_vals == nullptr), KMG_ERR_ARG, "d_vals / val_bytes mismatch");
    *h_selector_out = 0;
    g_stat_sort_passes = 0;
    g_stat_hybrid_path = 0;
    g_stat_hybrid_irregular = -1;
    g_stat_last_n_out = g_stat_last_err = -1;
    if (n <= 1 || end_bit == begin_bit) return KMG_OK;
    KMG_REQUIRE(d_keys && d_keys_alt && d_ws, KMG_ERR_ARG, "null pointer argument");
    KMG_REQUIRE(val_bytes == 0 || d_vals_alt, KMG_ERR_ARG, "d_vals_alt is null");
    KMG_REQUIRE(((uintptr_t)d_keys % key_bytes) == 0 && ((uintptr_t)d_keys_alt % key_bytes) == 0, KMG_ERR_ARG,
                "key buffers misaligned");
    const bool hybrid = hybrid_applies(n, key_bytes, val_bytes, begin_bit, end_bit);
    return sort_impl(d_keys, d_keys_alt, d_vals, d_vals_alt, n, key_bytes, val_bytes, begin_bit, end_bit, d_hist_in,
                     h_selector_out, d_ws, ws_bytes, st, hybrid, true);
}

extern "C" size_t kmg_rle_workspace_bytes(uint64_t n);
extern "C" int kmg_rle_count(const void* d_sorted_keys, uint64_t n, int key_bytes, void* d_uniq_keys_out,
                             uint32_t* d_counts_out, uint64_t* d_n_out, void* d_ws, size_t ws_bytes, void* stream);

extern "C" size_t kmg_sort_count_workspace_bytes(uint64_t n, int key_bytes, int end_bit) {
    return align_up(kmg_radix_sort_workspace_bytes(n, key_bytes, 0, 0, end_bit), 256) + kmg_rle_workspace_bytes(n);
}

// the run-length / singleton stage keeps its status word in its own workspace header: fold it into the
// sort's, which is the one callers check (kmg_ws_status(d_ws))
__global__ void merge_err_kernel(uint32_t* dst, const uint32_t* src) {
    if (*src) atomicMax(dst, *src);
}

int kmg::sort_count_core(void* d_keys, void* d_keys_alt, uint64_t n, int key_bytes, int end_bit, const uint64_t* d_hist_in,
                         uint32_t* d_counts_out, uint64_t* d_n_out, int* h_selector_out, void* d_ws, size_t ws_bytes,
                         void* stream, const PrePartitioned* pre) {
    cudaStream_t st = (cudaStream_t)stream;
    KMG_REQUIRE(key_bytes == 8 || key_bytes == 16, KMG_ERR_ARG, "key_bytes must be 8 or 16");
    KMG_REQUIRE(end_bit >= 0 && end_bit <= key_bytes * 8, KMG_ERR_ARG, "bad end_bit %d", end_bit);
    KMG_REQUIRE(h_selector_out && d_n_out, KMG_ERR_ARG, "null pointer argument");
    *h_selector_out = 0;
    g_stat_sort_passes = 0;
    g_stat_hybrid_path = 0;
    g_stat_hybrid_irregular = -1;
    g_stat_last_n_out = g_stat_last_err = -1;
    KMG_CUDA(cudaMemsetAsync(d_n_out, 0, sizeof(uint64_t), st));
    if (n == 0) return KMG_OK;
    KMG_REQUIRE(d_keys && d_keys_alt && d_counts_out && d_ws, KMG_ERR_ARG, "null pointer argument");
    KMG_REQUIRE(((uintptr_t)d_keys % key_bytes) == 0 && ((uintptr_t)d_keys_alt % key_bytes) == 0, KMG_ERR_ARG,
                "key buffers misaligned");
    const size_t sort_ws = align_up(kmg_radix_sort_workspace_bytes(n, key_bytes, 0, 0, end_bit), 256);
    KMG_REQUIRE(ws_bytes >= sort_ws + kmg_rle_workspace_bytes(n), KMG_ERR_WS, "sort_count workspace too small");
    int sel = 0;
    CountOut co{d_counts_out, reinterpret_cast<unsigned long long*>(d_n_out), false};
    if (n > 1 && end_bit > 0) {
        const bool hybrid = hybrid_applies(n, key_bytes, 0, 0, end_bit);
        const int rcode = sort_impl(d_keys, d_keys_alt, nullptr, nullptr, n, key_bytes, 0, 0, end_bit, d_hist_in, &sel, d_ws,
                                    sort_ws, st, hybrid, true, &co, pre);
        if (rcode != KMG_OK) return rcode;
    }
    if (co.done) {  // the hybrid finish wrote the table itself
        *h_selector_out = sel;
        return KMG_OK;
    }
    g_stat_last_n_out = g_stat_last_err = -1;  // (whatever the sort read back is not the final word)
    void* sorted = sel ? d_keys_alt : d_keys;
    void* other = sel ? d_keys : d_keys_alt;
    *h_selector_out = sel ^ 1;
    const int rcode = kmg_rle_count(sorted, n, key_bytes, other, d_counts_out, d_n_out, (char*)d_ws + sort_ws,
                                    ws_bytes - sort_ws, stream);
    if (rcode != KMG_OK) return rcode;
    merge_err_kernel<<<1, 1, 0, st>>>(&reinterpret_cast<WsHeader*>(d_ws)->err,
                                      &reinterpret_cast<WsHeader*>((char*)d_ws + sort_ws)->err);
    KMG_LAUNCH_CHECK();
    return KMG_OK;
}

extern "C" int kmg_sort_count(void* d_keys, void* d_keys_alt, uint64_t n, int key_bytes, int end_bit,
                              const uint64_t* d_hist_in, uint32_t* d_counts_out, uint64_t* d_n_out, int* h_selector_out,
                              void* d_ws, size_t ws_bytes, void* stream) {
    return sort_count_core(d_keys, d_keys_alt, n, key_bytes, end_bit, d_hist_in, d_counts_out, d_n_out, h_selector_out, d_ws,
                           ws_bytes, stream, nullptr);
}

extern "C" int kmg_select_singletons(const void* d_sorted_keys, const void* d_vals, uint64_t n, int key_bytes, int val_bytes,
                                     void* d_keys_out, void* d_vals_out, uint64_t* d_n_out, void* d_ws, size_t ws_bytes,
                                     void* stream);

static size_t sort_uniq_sort_ws(uint64_t n, int key_bytes, int val_bytes, int end_bit) {
    return align_up(carve_sort_ws(nullptr, n, key_bytes, hybrid_applies(n, key_bytes, val_bytes, 0, end_bit, true), val_bytes).total,
                    256);
}

extern "C" size_t kmg_sort_uniq_workspace_bytes(uint64_t n, int key_bytes, int val_bytes, int end_bit) {
    return sort_uniq_sort_ws(n, key_bytes, val_bytes, end_bit) + kmg_rle_workspace_bytes(n);
}

int kmg::sort_uniq_core(void* d_keys, void* d_keys_alt, void* d_vals, void* d_vals_alt, uint64_t n, int key_bytes,
                        int val_bytes, int end_bit, const uint64_t* d_hist_in, uint64_t* d_n_out, int* h_selector_out,
                        void* d_ws, size_t ws_bytes, void* stream, const PrePartitioned* pre) {
    cudaStream_t st = (cudaStream_t)stream;
    KMG_REQUIRE(key_bytes == 8 || key_bytes == 16, KMG_ERR_ARG, "key_bytes must be 8 or 16");
    KMG_REQUIRE(val_bytes == 4 || val_bytes == 8, KMG_ERR_ARG, "val_bytes must be 4 or 8");
    KMG_REQUIRE(end_bit >= 0 && end_bit <= key_bytes * 8, KMG_ERR_ARG, "bad end_bit %d", end_bit);
    KMG_REQUIRE(h_selector_out && d_n_out, KMG_ERR_ARG, "null pointer argument");
    *h_selector_out = 0;
    g_stat_sort_passes = 0;
    g_stat_hybrid_path = 0;
    g_stat_hybrid_irregular = -1;
    g_stat_last_n_out = g_stat_last_err = -1;
    KMG_CUDA(cudaMemsetAsync(d_n_out, 0, sizeof(uint64_t), st));
    if (n == 0) return KMG_OK;
    KMG_REQUIRE(d_keys && d_keys_alt && d_vals && d_vals_alt && d_ws, KMG_ERR_ARG, "null pointer argument");
    KMG_REQUIRE(((uintptr_t)d_keys % key_bytes) == 0 && ((uintptr_t)d_keys_alt % key_bytes) == 0, KMG_ERR_ARG,
                "key buffers misaligned");
    const size_t sort_ws = sort_uniq_sort_ws(n, key_bytes, val_bytes, end_bit);
    KMG_REQUIRE(ws_bytes >= sort_ws + kmg_rle_workspace_bytes(n), KMG_ERR_WS, "sort_uniq workspace too small");
    int sel = 0;
    CountOut uo{nullptr, reinterpret_cast<unsigned long long*>(d_n_out), false};
    if (n > 1 && end_bit > 0) {
        // equal keys may come out in any order: only keys that occur once are kept
        const bool hybrid = hybrid_applies(n, key_bytes, val_bytes, 0, end_bit, true);
        const int rcode = sort_impl(d_keys, d_keys_alt, d_vals, d_vals_alt, n, key_bytes, val_bytes, 0, end_bit, d_hist_in, &sel,
                                    d_ws, sort_ws, st, hybrid, true, &uo, pre);
        if (rcode != KMG_OK) return rcode;
    }
    if (uo.done) {  // the hybrid finish emitted the singletons itself
        *h_selector_out = sel;
        return KMG_OK;
    }
    g_stat_last_n_out = g_stat_last_err = -1;
    *h_selector_out = sel ^ 1;
    const int rcode = kmg_select_singletons(sel ? d_keys_alt : d_keys, sel ? d_vals_alt : d_vals, n, key_bytes, val_bytes,
                                            sel ? d_keys : d_keys_alt, sel ? d_vals : d_vals_alt, d_n_out,
                                            (char*)d_ws + sort_ws, ws_bytes - sort_ws, stream);
    if (rcode != KMG_OK) return rcode;
    merge_err_kernel<<<1, 1, 0, st>>>(&reinterpret_cast<WsHeader*>(d_ws)->err,
                                      &reinterpret_cast<WsHeader*>((char*)d_ws + sort_ws)->err);
    KMG_LAUNCH_CHECK();
    return KMG_OK;
}

extern "C" int kmg_sort_uniq(void* d_keys, void* d_keys_alt, void* d_vals, void* d_vals_alt, uint64_t n, int key_bytes,
                             int val_bytes, int end_bit, const uint64_t* d_hist_in, uint64_t* d_n_out, int* h_selector_out,
                             void* d_ws, size_t ws_bytes, void* stream) {
    return sort_uniq_core(d_keys, d_keys_alt, d_vals, d_vals_alt, n, key_bytes, val_bytes, end_bit, d_hist_in, d_n_out,
                          h_selector_out, d_ws, ws_bytes, stream, nullptr);
}

extern "C" size_t kmg_partition_workspace_bytes(uint64_t n, int key_bytes, int val_bytes) {
    return kmg_radix_sort_workspace_bytes(n, key_bytes, val_bytes, 0, 8);
}

extern "C" int kmg_range_partition(const void* d_keys, const void* d_vals, uint64_t n, int key_bytes, int val_bytes,
                                   int key_bits, int n_parts, void* d_keys_out, void* d_vals_out,
                                   uint64_t* d_part_counts, void* d_ws, size_t ws_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    KMG_REQUIRE(key_bytes == 8 || key_bytes == 16, KMG_ERR_ARG, "key_bytes must be 8 or 16");
    KMG_REQUIRE(val_bytes == 0 || val_bytes == 4 || val_bytes == 8, KMG_ERR_ARG, "val_bytes must be 0, 4 or 8");
    KMG_REQUIRE(n_parts >= 1 && n_parts <= SORT_RADIX, KMG_ERR_ARG, "n_parts must be in [1,%d]", SORT_RADIX);
    KMG_REQUIRE(key_bits >= 16 && key_bits <= key_bytes * 8, KMG_ERR_ARG, "key_bits must be in [16,%d]", key_bytes * 8);
    KMG_REQUIRE(d_part_counts && d_ws, KMG_ERR_ARG, "null pointer argument");
    KMG_REQUIRE((val_bytes == 0) == (d_vals == nullptr), KMG_ERR_ARG, "d_vals / val_bytes mismatch");
    KMG_CUDA(cudaMemsetAsync(d_part_counts, 0, sizeof(uint64_t) * n_parts, st));
    if (n == 0) return KMG_OK;
    SortWs w = carve_sort_ws(d_ws, n, key_bytes, false);
    KMG_REQUIRE(ws_bytes >= w.total, KMG_ERR_WS, "partition workspace too small");
    KMG_CUDA(cudaMemsetAsync(d_ws, 0, w.total, st));
    const RangeDigit op{key_bits - 16, (uint32_t)n_parts};
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int grid = (int)std::min<uint64_t>((n + 511) / 512, (uint64_t)sms * 4);
    if (key_bytes == 8)
        digit_hist_kernel<uint64_t, RangeDigit><<<grid, 512, SORT_RADIX * 4, st>>>((const uint64_t*)d_keys, n, op, SORT_RADIX, w.hist);
    else
        digit_hist_kernel<u128, RangeDigit><<<grid, 512, SORT_RADIX * 4, st>>>((const u128*)d_keys, n, op, SORT_RADIX, w.hist);
    KMG_LAUNCH_CHECK();
    radix_scan_kernel<<<1, 32, 0, st>>>(w.hist, w.bins, SORT_RADIX, 2 * SORT_RADIX, nullptr);
    KMG_LAUNCH_CHECK();
    KMG_CUDA(cudaMemcpyAsync(d_part_counts, w.hist, sizeof(uint64_t) * n_parts, cudaMemcpyDeviceToDevice, st));
    const uint64_t n_lb_parts = (n + PART_MAX - 1) / PART_MAX;
    for (uint64_t part = 0; part < n_lb_parts; ++part) {
        const uint64_t off = part * PART_MAX;
        OnesweepParams p;
        p.keys_in = (const char*)d_keys + off * key_bytes;
        p.keys_out = d_keys_out;
        p.vals_in = d_vals ? (const char*)d_vals + off * val_bytes : nullptr;
        p.vals_out = d_vals_out;
        p.n = (uint32_t)std::min<uint64_t>(PART_MAX, n - off);
        p.bins_in = w.bins + (part & 1) * SORT_RADIX;
        p.bins_out = (part + 1 < n_lb_parts) ? w.bins + ((part + 1) & 1) * SORT_RADIX : nullptr;
        p.lb_agg = w.lookback;
        p.lb_ginc = w.lookback + w.lb_words;
        p.ticket = &w.hdr->ticket;
        p.err = &w.hdr->err;
        p.tag = 1u << 30;
        if (part > 0) KMG_CUDA(cudaMemsetAsync(w.lookback, 0, (char*)d_ws + w.total - (char*)w.lookback, st));
        int rcode = dispatch_onesweep(false, key_bytes, val_bytes, p, op, st);
        if (rcode != KMG_OK) return rcode;
    }
    return KMG_OK;
}
