// K4: run-length / singleton selection on sorted keys.
//
// Replaces the grouping loop of Crawler.do_batch (kmermaid/join.py:95-130) and the two emit
// rules: KJoiner.join_sequence_count (join.py:265-285: every group, with its size) and
// KJoiner.join_unique (join.py:243-263: only groups of size exactly one).
//
// A warp walks its contiguous chunk 32 keys at a time; "is the key different from its
// predecessor" becomes one ballot per step, so ranks are popcounts and no shared-memory
// transposition of the keys is needed.
//
// Three launches, no CTA ever waits for another one:
//   1. rle_tile_aggregates: per tile, number of run heads, number of singletons and the
//      position of the last head (reads the keys once);
//   2. rle_scan_tiles: one block turns them into per-tile output offsets and the "run that is
//      open when the tile starts" carry;
//   3. rle_count_kernel / select_singletons_kernel: re-read the keys and emit.
// A single-sweep version with an in-kernel tile prefix was measured first: with B200's tile
// rate the CTAs spent 55-66 % of their time waiting at the barrier behind the prefix
// (profiles/r01_ncu_summary.md); the second read of the keys costs less than that wait.
#include <type_traits>

#include "common.cuh"

namespace kmg {

int64_t g_count_limit = 0;  // kmg_set_option("count_limit", n): test hook, 0 = the real limit 2^32-1

constexpr int RLE_BLOCK = 256;
constexpr int RLE_WARPS = RLE_BLOCK / 32;

template <typename KeyT>
__device__ __forceinline__ KeyT shfl_key(const KeyT& k, int src);
template <>
__device__ __forceinline__ uint64_t shfl_key<uint64_t>(const uint64_t& k, int src) {
    return __shfl_sync(0xffffffffu, k, src);
}
template <>
__device__ __forceinline__ u128 shfl_key<u128>(const u128& k, int src) {
    return u128{__shfl_sync(0xffffffffu, k.lo, src), __shfl_sync(0xffffffffu, k.hi, src)};
}
template <>
__device__ __forceinline__ u256 shfl_key<u256>(const u256& k, int src) {  // wide stream at k > 32 (wide256.cu)
    return u256{shfl_key<u128>(k.lo, src), shfl_key<u128>(k.hi, src)};
}

struct RleParams {
    const void* keys_in;
    const void* vals_in;
    uint64_t n;
    void* keys_out;
    void* vals_out;
    uint32_t* counts_out;
    unsigned long long* n_out;
    uint32_t n_tiles;
    uint32_t* t_heads;    // [tiles] run heads in the tile
    uint32_t* t_singles;  // [tiles] singletons in the tile
    uint32_t* t_last;     // [tiles] tile-local position + 1 of the last head (0 = none)
    uint64_t* t_hpre;     // [tiles] heads before the tile
    uint64_t* t_spre;     // [tiles] singletons before the tile
    uint64_t* t_carry;    // [tiles] position + 1 of the last head before the tile (0 = none)
    uint32_t* err;
    unsigned long long count_limit;  // run lengths above it raise err = 2 (2^32-1; lower only in tests)
};

// lanes of step j whose element exists (tile-local index < n_local)
__device__ __forceinline__ uint32_t valid_mask(uint32_t step_first, uint32_t n_local) {
    if (step_first >= n_local) return 0u;
    const uint32_t left = n_local - step_first;
    return left >= 32 ? 0xffffffffu : ((1u << left) - 1u);
}

// Loads the warp's chunk (IPT steps of 32 consecutive keys starting at tile-local index
// `wfirst`) and returns the extended head ballots: bit l of hb[j] is set iff element
// wfirst + 32*j + l starts a run, where the element one past the end of the whole array counts
// as a head (end sentinel) and anything beyond does not.  hnext = head flag of the element
// right after the chunk.  FULL: every element of the tile exists.
template <typename KeyT, int IPT, bool FULL>
__device__ __forceinline__ void load_heads(const KeyT* __restrict__ kin, uint64_t tile_base, uint32_t n_local,
                                           bool more_after_tile, uint32_t wfirst, KeyT (&keys)[IPT],
                                           uint32_t (&hb)[IPT], uint32_t& hnext) {
    const uint32_t lane = lane_id();
#pragma unroll
    for (int j = 0; j < IPT; ++j) {
        const uint32_t li = wfirst + 32 * j + lane;
        keys[j] = (FULL || li < n_local) ? kin[li] : KeyT{};
    }
    const bool first_of_all = tile_base == 0 && wfirst == 0;
    KeyT before = KeyT{};
    if (lane == 0 && !first_of_all && (FULL || wfirst <= n_local)) before = *(kin + wfirst - 1);
#pragma unroll
    for (int j = 0; j < IPT; ++j) {
        const uint32_t li = wfirst + 32 * j + lane;
        KeyT prev = shfl_key(keys[j], (int)lane - 1);
        if (lane == 0) prev = before;
        bool head = keys[j] != prev || (first_of_all && j == 0 && lane == 0);
        if (!FULL) head = (li < n_local && head) || li == n_local;
        hb[j] = __ballot_sync(0xffffffffu, head);
        before = shfl_key(keys[j], 31);  // only lane 0 uses it
    }
    const uint32_t nli = wfirst + 32 * IPT;
    uint32_t h = 0;
    if (lane == 0) {
        if (nli < n_local || (nli == n_local && more_after_tile)) h = kin[nli] != before ? 1u : 0u;
        else if (nli == n_local) h = 1;  // end of the array
    }
    hnext = __shfl_sync(0xffffffffu, h, 0);
}

// ---- 1. per-tile aggregates ----------------------------------------------------------------------
template <typename KeyT, int IPT, bool FULL>
__device__ __forceinline__ void aggregates_tile(const RleParams& p, const uint32_t tile, uint32_t* s_red) {
    constexpr int TILE = RLE_BLOCK * IPT;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t tile_base = (uint64_t)tile * TILE;
    const uint32_t n_local = FULL ? (uint32_t)TILE : (uint32_t)(p.n - tile_base);
    const uint32_t wfirst = warp * 32 * IPT;
    const KeyT* kin = reinterpret_cast<const KeyT*>(p.keys_in) + tile_base;
    KeyT keys[IPT];
    uint32_t hb[IPT];
    uint32_t hnext;
    load_heads<KeyT, IPT, FULL>(kin, tile_base, n_local, tile_base + TILE < p.n, wfirst, keys, hb, hnext);
    uint32_t heads = 0, singles = 0, last = 0;
#pragma unroll
    for (int j = 0; j < IPT; ++j) {
        const uint32_t vm = FULL ? 0xffffffffu : valid_mask(wfirst + 32 * j, n_local);
        const uint32_t b = hb[j] & vm;
        const uint32_t nb = (j + 1 < IPT) ? hb[j + 1 < IPT ? j + 1 : j] : hnext;
        const uint32_t tb = (hb[j] >> 1) | ((nb & 1u) << 31);
        heads += __popc(b);
        singles += __popc(b & tb);
        if (b) last = wfirst + 32 * j + (31 - __clz(b)) + 1;
    }
    if (lane == 0) {
        s_red[warp] = heads;
        s_red[RLE_WARPS + warp] = singles;
        s_red[2 * RLE_WARPS + warp] = last;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t th = 0, ts = 0, tl = 0;
#pragma unroll
        for (int w = 0; w < RLE_WARPS; ++w) {
            th += s_red[w];
            ts += s_red[RLE_WARPS + w];
            tl = max(tl, s_red[2 * RLE_WARPS + w]);
        }
        p.t_heads[tile] = th;
        p.t_singles[tile] = ts;
        p.t_last[tile] = tl;
    }
}

template <typename KeyT, int IPT>
__global__ void __launch_bounds__(RLE_BLOCK) rle_tile_aggregates(const RleParams p) {
    constexpr int TILE = RLE_BLOCK * IPT;
    __shared__ uint32_t s_red[3 * RLE_WARPS];
    const uint32_t tile = blockIdx.x;
    if ((uint64_t)(tile + 1) * TILE <= p.n) aggregates_tile<KeyT, IPT, true>(p, tile, s_red);
    else aggregates_tile<KeyT, IPT, false>(p, tile, s_red);
}

// ---- 2. scan over the tiles (one block of 32 warps; warp w owns a contiguous segment) ----------------
constexpr int SCAN_BLOCK = 1024;

__device__ __forceinline__ uint64_t warp_incl_max(uint64_t v) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint64_t t = __shfl_up_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) >= (uint32_t)o) v = max(v, t);
    }
    return v;
}

__global__ void __launch_bounds__(SCAN_BLOCK) rle_scan_tiles(const RleParams p, uint32_t tile_keys, int want_singles) {
    __shared__ uint64_t s_h[33], s_s[33], s_c[33];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t per = ((p.n_tiles + 31) / 32 + 31) / 32 * 32;  // tiles per warp, multiple of 32
    const uint32_t b = min(warp * per, p.n_tiles), e = min(b + per, p.n_tiles);
    // pass 1: the segment's totals
    uint64_t h = 0, s = 0, c = 0;
    for (uint32_t i = b + lane; i < e; i += 32) {
        h += p.t_heads[i];
        s += p.t_singles[i];
        const uint32_t l = p.t_last[i];
        if (l) c = max(c, (uint64_t)i * tile_keys + l);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        h += __shfl_xor_sync(0xffffffffu, h, o);
        s += __shfl_xor_sync(0xffffffffu, s, o);
        c = max(c, __shfl_xor_sync(0xffffffffu, c, o));
    }
    if (lane == 0) {
        s_h[warp] = h;
        s_s[warp] = s;
        s_c[warp] = c;
    }
    __syncthreads();
    if (warp == 0) {  // exclusive scan of the 32 segment totals
        const uint64_t hv = s_h[lane], sv = s_s[lane], cv = s_c[lane];
        const uint64_t hi = warp_incl_scan(hv), si = warp_incl_scan(sv), ci = warp_incl_max(cv);
        const uint64_t cprev = __shfl_up_sync(0xffffffffu, ci, 1);
        s_h[lane] = hi - hv;
        s_s[lane] = si - sv;
        s_c[lane] = lane ? cprev : 0;
        if (lane == 31) {
            s_h[32] = hi;
            s_s[32] = si;
        }
    }
    __syncthreads();
    // pass 2: prefixes inside the segment, 32 tiles per step
    uint64_t hrun = s_h[warp], srun = s_s[warp], crun = s_c[warp];
    for (uint32_t i0 = b; i0 < e; i0 += 32) {
        const uint32_t i = i0 + lane;
        const bool ok = i < e;
        const uint64_t hv = ok ? p.t_heads[i] : 0, sv = ok ? p.t_singles[i] : 0;
        const uint32_t l = ok ? p.t_last[i] : 0;
        const uint64_t cv = l ? (uint64_t)i * tile_keys + l : 0;
        const uint64_t hi = warp_incl_scan(hv), si = warp_incl_scan(sv), ci = warp_incl_max(cv);
        const uint64_t cprev = __shfl_up_sync(0xffffffffu, ci, 1);
        if (ok) {
            p.t_hpre[i] = hrun + hi - hv;
            p.t_spre[i] = srun + si - sv;
            p.t_carry[i] = max(crun, lane ? cprev : (uint64_t)0);
        }
        hrun += __shfl_sync(0xffffffffu, hi, 31);
        srun += __shfl_sync(0xffffffffu, si, 31);
        crun = max(crun, __shfl_sync(0xffffffffu, ci, 31));
    }
    if (threadIdx.x == 0) *p.n_out = want_singles ? s_s[32] : s_h[32];
}

// ---- 3a. count: distinct keys + run lengths ----------------------------------------------------------
template <typename KeyT, int IPT, bool FULL>
__device__ __forceinline__ void rle_count_tile(const RleParams& p, const uint32_t tile, uint32_t* s_hpos, uint32_t* s_wheads) {
    constexpr int TILE = RLE_BLOCK * IPT;
    const int t = threadIdx.x;
    const uint32_t lane = t & 31, warp = t >> 5;
    const uint64_t tile_base = (uint64_t)tile * TILE;
    const uint32_t n_local = FULL ? (uint32_t)TILE : (uint32_t)(p.n - tile_base);
    const uint32_t wfirst = warp * 32 * IPT;
    const KeyT* kin = reinterpret_cast<const KeyT*>(p.keys_in) + tile_base;
    const uint64_t excl_heads = p.t_hpre[tile];
    const uint64_t carry = p.t_carry[tile];  // position+1 of the head of the run open at tile start

    KeyT keys[IPT];
    uint32_t hb[IPT];
    uint32_t hnext;
    load_heads<KeyT, IPT, FULL>(kin, tile_base, n_local, tile_base + TILE < p.n, wfirst, keys, hb, hnext);

    uint32_t wheads = 0;
#pragma unroll
    for (int j = 0; j < IPT; ++j) wheads += __popc(FULL ? hb[j] : (hb[j] & valid_mask(wfirst + 32 * j, n_local)));
    if (lane == 0) s_wheads[warp] = wheads;
    __syncthreads();
    uint32_t wexcl = 0;
#pragma unroll
    for (int w = 0; w < RLE_WARPS; ++w)
        if (w < (int)warp) wexcl += s_wheads[w];
    const uint32_t lt = lanemask_lt();
    {
        uint32_t run = wexcl;
#pragma unroll
        for (int j = 0; j < IPT; ++j) {
            const uint32_t b = FULL ? hb[j] : (hb[j] & valid_mask(wfirst + 32 * j, n_local));
            if ((b >> lane) & 1u) s_hpos[run + __popc(b & lt)] = wfirst + 32 * j + lane;
            run += __popc(b);
        }
    }
    __syncthreads();
    KeyT* keys_out = reinterpret_cast<KeyT*>(p.keys_out) + excl_heads;
    uint32_t* counts_out = p.counts_out + excl_heads;  // slot -1 (the run open at tile start) is valid when used
    uint32_t run = wexcl;  // heads of the tile before the current step
#pragma unroll
    for (int j = 0; j < IPT; ++j) {
        const uint32_t li = wfirst + 32 * j + lane;
        const uint32_t vm = FULL ? 0xffffffffu : valid_mask(wfirst + 32 * j, n_local);
        const uint32_t b = hb[j];
        const uint32_t nb = (j + 1 < IPT) ? hb[j + 1 < IPT ? j + 1 : j] : hnext;
        const uint32_t tb = (b >> 1) | ((nb & 1u) << 31);  // tail: the next element is a head
        const uint32_t h_before = run + __popc(b & vm & lt);
        const bool is_head = (b >> lane) & 1u;
        if (FULL || li < n_local) {
            if (is_head) keys_out[h_before] = keys[j];
            if ((tb >> lane) & 1u) {
                const uint32_t h_incl = h_before + (is_head ? 1u : 0u);
                uint64_t len;
                if (h_incl) len = (uint64_t)(li - s_hpos[h_incl - 1]) + 1;
                else len = tile_base + li - (carry - 1) + 1;
                if (len > p.count_limit) atomicExch(p.err, 2u);
                *(counts_out + (int64_t)h_incl - 1) = (uint32_t)len;
            }
        }
        run += __popc(b & vm);
    }
}

template <typename KeyT, int IPT>
__global__ void __launch_bounds__(RLE_BLOCK, 3) rle_count_kernel(const RleParams p) {
    constexpr int TILE = RLE_BLOCK * IPT;
    __shared__ uint32_t s_hpos[TILE];  // local position of the i-th head of the tile
    __shared__ uint32_t s_wheads[RLE_WARPS];
    const uint32_t tile = blockIdx.x;
    if ((uint64_t)(tile + 1) * TILE <= p.n) rle_count_tile<KeyT, IPT, true>(p, tile, s_hpos, s_wheads);
    else rle_count_tile<KeyT, IPT, false>(p, tile, s_hpos, s_wheads);
}

// ---- 3b. singletons: head && tail, compacted in order, with payload ------------------------------------
template <typename KeyT, int VAL_BYTES, int IPT, bool FULL>
__device__ __forceinline__ void select_tile(const RleParams& p, const uint32_t tile, uint32_t* s_wcnt) {
    constexpr int TILE = RLE_BLOCK * IPT;
    using ValT = typename std::conditional<VAL_BYTES == 4, uint32_t, uint64_t>::type;
    const int t = threadIdx.x;
    const uint32_t lane = t & 31, warp = t >> 5;
    const uint64_t tile_base = (uint64_t)tile * TILE;
    const uint32_t n_local = FULL ? (uint32_t)TILE : (uint32_t)(p.n - tile_base);
    const uint32_t wfirst = warp * 32 * IPT;
    const KeyT* kin = reinterpret_cast<const KeyT*>(p.keys_in) + tile_base;
    const uint64_t tile_excl = p.t_spre[tile];

    KeyT keys[IPT];
    uint32_t hb[IPT];
    uint32_t hnext;
    load_heads<KeyT, IPT, FULL>(kin, tile_base, n_local, tile_base + TILE < p.n, wfirst, keys, hb, hnext);

    uint32_t sb[IPT];  // singleton ballots
    uint32_t wcnt = 0;
#pragma unroll
    for (int j = 0; j < IPT; ++j) {
        const uint32_t nb = (j + 1 < IPT) ? hb[j + 1 < IPT ? j + 1 : j] : hnext;
        const uint32_t tb = (hb[j] >> 1) | ((nb & 1u) << 31);
        sb[j] = hb[j] & tb & (FULL ? 0xffffffffu : valid_mask(wfirst + 32 * j, n_local));
        wcnt += __popc(sb[j]);
    }
    if (lane == 0) s_wcnt[warp] = wcnt;
    __syncthreads();
    uint32_t wexcl = 0;
#pragma unroll
    for (int w = 0; w < RLE_WARPS; ++w)
        if (w < (int)warp) wexcl += s_wcnt[w];
    const uint64_t base = tile_excl + wexcl;
    KeyT* keys_out = reinterpret_cast<KeyT*>(p.keys_out) + base;
    const ValT* vals_in = reinterpret_cast<const ValT*>(p.vals_in) + tile_base;
    ValT* vals_out = reinterpret_cast<ValT*>(p.vals_out) + base;
    const uint32_t lt = lanemask_lt();
    uint32_t run = 0;
#pragma unroll
    for (int j = 0; j < IPT; ++j) {
        if ((sb[j] >> lane) & 1u) {
            const uint32_t o = run + __popc(sb[j] & lt);
            keys_out[o] = keys[j];
            if constexpr (VAL_BYTES != 0) vals_out[o] = vals_in[wfirst + 32 * j + lane];
        }
        run += __popc(sb[j]);
    }
}

template <typename KeyT, int VAL_BYTES, int IPT>
__global__ void __launch_bounds__(RLE_BLOCK, 3) select_singletons_kernel(const RleParams p) {
    constexpr int TILE = RLE_BLOCK * IPT;
    __shared__ uint32_t s_wcnt[RLE_WARPS];
    const uint32_t tile = blockIdx.x;
    if ((uint64_t)(tile + 1) * TILE <= p.n) select_tile<KeyT, VAL_BYTES, IPT, true>(p, tile, s_wcnt);
    else select_tile<KeyT, VAL_BYTES, IPT, false>(p, tile, s_wcnt);
}

constexpr int RLE_IPT8 = 16;   // 8-byte keys: 4096-key tiles
constexpr int RLE_IPT16 = 8;   // 16-byte keys: 2048-key tiles

// ---- 4. order-preserving compaction of a count table to the rows in range (kmg_filter_counts) ---------
// One pass with a ticketed tile prefix.  A tile loads its rows into registers before it publishes its
// aggregate, and its rows go to [prefix, prefix + kept) <= its own input's end; a later tile writes only
// once every earlier one has published (it needs their aggregates), so the table can be compacted in place.
struct FilterParams {
    const void* keys_in;
    const uint32_t* counts_in;
    void* keys_out;
    uint32_t* counts_out;
    uint64_t n;
    uint32_t n_tiles;
    uint32_t min_count, max_count;
    unsigned long long* n_out;
    uint64_t* tile_state;
    uint32_t* ticket;
    uint32_t* err;
};

template <typename KeyT, int IPT>
__global__ void __launch_bounds__(RLE_BLOCK) filter_counts_kernel(const FilterParams p) {
    constexpr int TILE = RLE_BLOCK * IPT;
    __shared__ uint32_t s_off[IPT][RLE_WARPS];  // kept rows of warp w in round j, then their exclusive prefix
    __shared__ uint32_t s_tile;
    __shared__ uint64_t s_base;
    const uint32_t t = threadIdx.x, lane = t & 31u, warp = t >> 5;
    if (t == 0) s_tile = atomicAdd(p.ticket, 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint64_t tile_base = (uint64_t)tile * TILE;
    const KeyT* kin = reinterpret_cast<const KeyT*>(p.keys_in) + tile_base;
    const uint32_t* cin = p.counts_in + tile_base;
    const uint64_t left = p.n - tile_base;
    KeyT keys[IPT];
    uint32_t counts[IPT], keep[IPT];
#pragma unroll
    for (int j = 0; j < IPT; ++j) {
        const uint32_t i = j * RLE_BLOCK + t;
        keys[j] = i < left ? kin[i] : KeyT{};
        counts[j] = i < left ? cin[i] : 0u;
    }
#pragma unroll
    for (int j = 0; j < IPT; ++j) {
        keep[j] = __ballot_sync(0xffffffffu, counts[j] >= p.min_count && counts[j] <= p.max_count);
        if (lane == 0) s_off[j][warp] = __popc(keep[j]);
    }
    __syncthreads();  // (every row of the tile is in registers: the tile may publish)
    if (warp == 0) {
        constexpr int PER = IPT * RLE_WARPS / 32;
        uint32_t* flat = &s_off[0][0];
        uint32_t v[PER], sum = 0;
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            v[i] = flat[lane * PER + i];
            sum += v[i];
        }
        const uint32_t incl = warp_incl_scan(sum);
        uint32_t run = incl - sum;
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            flat[lane * PER + i] = run;
            run += v[i];
        }
        const uint32_t agg = __shfl_sync(0xffffffffu, incl, 31);
        if (lane == 0) {
            __threadfence();
            tile_prefix_publish(p.tile_state, tile, agg);
        }
        const uint64_t base = tile_prefix_resolve_warp(p.tile_state, p.n_tiles, tile, agg, p.err);
        if (lane == 0) {
            s_base = base;
            if (tile == p.n_tiles - 1) *p.n_out = base + agg;
        }
    }
    __syncthreads();
    const uint64_t base = s_base;
    KeyT* kout = reinterpret_cast<KeyT*>(p.keys_out) + base;
    uint32_t* cout = p.counts_out + base;
    const uint32_t lt = lanemask_lt();
#pragma unroll
    for (int j = 0; j < IPT; ++j) {
        if ((keep[j] >> lane) & 1u) {
            const uint32_t o = s_off[j][warp] + __popc(keep[j] & lt);
            kout[o] = keys[j];
            cout[o] = counts[j];
        }
    }
}

}  // namespace kmg

using namespace kmg;

static size_t rle_tiles_max(uint64_t n) { return n / 2048 + 2; }

extern "C" size_t kmg_rle_workspace_bytes(uint64_t n) {
    const size_t t = rle_tiles_max(n);
    return sizeof(WsHeader) + 3 * align_up(t * sizeof(uint32_t), 256) + 3 * align_up(t * sizeof(uint64_t), 256);
}

static int rle_setup(RleParams& p, uint64_t n, int key_bytes, void* d_ws, size_t ws_bytes, cudaStream_t st) {
    KMG_REQUIRE(key_bytes == 8 || key_bytes == 16 || key_bytes == 32, KMG_ERR_ARG, "key_bytes must be 8, 16 or 32");
    KMG_REQUIRE(d_ws, KMG_ERR_ARG, "null workspace");
    KMG_REQUIRE(ws_bytes >= kmg_rle_workspace_bytes(n), KMG_ERR_WS, "rle workspace too small");
    const uint64_t tile = key_bytes == 8 ? RLE_BLOCK * RLE_IPT8 : RLE_BLOCK * RLE_IPT16;
    const uint64_t nt = (n + tile - 1) / tile;
    KMG_REQUIRE(nt < (1ull << 31), KMG_ERR_RANGE, "too many tiles");
    KMG_CUDA(cudaMemsetAsync(d_ws, 0, sizeof(WsHeader), st));
    const size_t t = rle_tiles_max(n);
    const size_t a32 = align_up(t * sizeof(uint32_t), 256), a64 = align_up(t * sizeof(uint64_t), 256);
    char* at = (char*)d_ws;
    WsHeader* hdr = reinterpret_cast<WsHeader*>(at);
    at += sizeof(WsHeader);
    p.n = n;
    p.n_tiles = (uint32_t)nt;
    p.t_heads = (uint32_t*)at; at += a32;
    p.t_singles = (uint32_t*)at; at += a32;
    p.t_last = (uint32_t*)at; at += a32;
    p.t_hpre = (uint64_t*)at; at += a64;
    p.t_spre = (uint64_t*)at; at += a64;
    p.t_carry = (uint64_t*)at; at += a64;
    p.err = &hdr->err;
    p.count_limit = g_count_limit > 0 ? (unsigned long long)g_count_limit : 0xffffffffull;
    return KMG_OK;
}

static int rle_prepass(const RleParams& p, int key_bytes, int want_singles, cudaStream_t st) {
    if (key_bytes == 8) rle_tile_aggregates<uint64_t, RLE_IPT8><<<p.n_tiles, RLE_BLOCK, 0, st>>>(p);
    else if (key_bytes == 16) rle_tile_aggregates<u128, RLE_IPT16><<<p.n_tiles, RLE_BLOCK, 0, st>>>(p);
    else rle_tile_aggregates<u256, RLE_IPT16><<<p.n_tiles, RLE_BLOCK, 0, st>>>(p);
    KMG_LAUNCH_CHECK();
    const uint32_t tile_keys = key_bytes == 8 ? RLE_BLOCK * RLE_IPT8 : RLE_BLOCK * RLE_IPT16;
    rle_scan_tiles<<<1, SCAN_BLOCK, 0, st>>>(p, tile_keys, want_singles);
    KMG_LAUNCH_CHECK();
    return KMG_OK;
}

extern "C" int kmg_rle_count(const void* d_sorted_keys, uint64_t n, int key_bytes, void* d_uniq_keys_out,
                             uint32_t* d_counts_out, uint64_t* d_n_out, void* d_ws, size_t ws_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    KMG_REQUIRE(d_n_out, KMG_ERR_ARG, "d_n_out is null");
    KMG_CUDA(cudaMemsetAsync(d_n_out, 0, sizeof(uint64_t), st));
    if (n == 0) return KMG_OK;  // join.py:107-111: nothing to crawl -> empty output
    KMG_REQUIRE(d_sorted_keys && d_uniq_keys_out && d_counts_out, KMG_ERR_ARG, "null pointer argument");
    RleParams p;
    memset(&p, 0, sizeof(p));
    int rcode = rle_setup(p, n, key_bytes, d_ws, ws_bytes, st);
    if (rcode != KMG_OK) return rcode;
    p.keys_in = d_sorted_keys;
    p.keys_out = d_uniq_keys_out;
    p.counts_out = d_counts_out;
    p.n_out = reinterpret_cast<unsigned long long*>(d_n_out);
    rcode = rle_prepass(p, key_bytes, 0, st);
    if (rcode != KMG_OK) return rcode;
    if (key_bytes == 8) rle_count_kernel<uint64_t, RLE_IPT8><<<p.n_tiles, RLE_BLOCK, 0, st>>>(p);
    else if (key_bytes == 16) rle_count_kernel<u128, RLE_IPT16><<<p.n_tiles, RLE_BLOCK, 0, st>>>(p);
    else rle_count_kernel<u256, RLE_IPT16><<<p.n_tiles, RLE_BLOCK, 0, st>>>(p);
    KMG_LAUNCH_CHECK();
    return KMG_OK;
}

extern "C" int kmg_select_singletons(const void* d_sorted_keys, const void* d_vals, uint64_t n, int key_bytes,
                                     int val_bytes, void* d_keys_out, void* d_vals_out, uint64_t* d_n_out,
                                     void* d_ws, size_t ws_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    KMG_REQUIRE(d_n_out, KMG_ERR_ARG, "d_n_out is null");
    KMG_REQUIRE(val_bytes == 0 || val_bytes == 4 || val_bytes == 8, KMG_ERR_ARG, "val_bytes must be 0, 4 or 8");
    KMG_REQUIRE((val_bytes == 0) == (d_vals == nullptr), KMG_ERR_ARG, "d_vals / val_bytes mismatch");
    KMG_REQUIRE(val_bytes == 0 || d_vals_out, KMG_ERR_ARG, "d_vals_out is null");
    KMG_CUDA(cudaMemsetAsync(d_n_out, 0, sizeof(uint64_t), st));
    if (n == 0) return KMG_OK;
    KMG_REQUIRE(d_sorted_keys && d_keys_out, KMG_ERR_ARG, "null pointer argument");
    RleParams p;
    memset(&p, 0, sizeof(p));
    int rcode = rle_setup(p, n, key_bytes, d_ws, ws_bytes, st);
    if (rcode != KMG_OK) return rcode;
    p.keys_in = d_sorted_keys;
    p.vals_in = d_vals;
    p.keys_out = d_keys_out;
    p.vals_out = d_vals_out;
    p.n_out = reinterpret_cast<unsigned long long*>(d_n_out);
    rcode = rle_prepass(p, key_bytes, 1, st);
    if (rcode != KMG_OK) return rcode;
    const uint32_t tiles = p.n_tiles;
    if (key_bytes == 8) {
        if (val_bytes == 0) select_singletons_kernel<uint64_t, 0, RLE_IPT8><<<tiles, RLE_BLOCK, 0, st>>>(p);
        else if (val_bytes == 4) select_singletons_kernel<uint64_t, 4, RLE_IPT8><<<tiles, RLE_BLOCK, 0, st>>>(p);
        else select_singletons_kernel<uint64_t, 8, RLE_IPT8><<<tiles, RLE_BLOCK, 0, st>>>(p);
    } else if (key_bytes == 16) {
        if (val_bytes == 0) select_singletons_kernel<u128, 0, RLE_IPT16><<<tiles, RLE_BLOCK, 0, st>>>(p);
        else if (val_bytes == 4) select_singletons_kernel<u128, 4, RLE_IPT16><<<tiles, RLE_BLOCK, 0, st>>>(p);
        else select_singletons_kernel<u128, 8, RLE_IPT16><<<tiles, RLE_BLOCK, 0, st>>>(p);
    } else {
        if (val_bytes == 0) select_singletons_kernel<u256, 0, RLE_IPT16><<<tiles, RLE_BLOCK, 0, st>>>(p);
        else if (val_bytes == 4) select_singletons_kernel<u256, 4, RLE_IPT16><<<tiles, RLE_BLOCK, 0, st>>>(p);
        else select_singletons_kernel<u256, 8, RLE_IPT16><<<tiles, RLE_BLOCK, 0, st>>>(p);
    }
    KMG_LAUNCH_CHECK();
    return KMG_OK;
}

int kmg::filter_counts(const void* d_keys, const uint32_t* d_counts, uint64_t n, int key_bytes, CountRange range, void* d_keys_out,
                       uint32_t* d_counts_out, uint64_t* d_n_out, void* d_ws, size_t ws_bytes, cudaStream_t st) {
    KMG_REQUIRE(key_bytes == 8 || key_bytes == 16 || key_bytes == 32, KMG_ERR_ARG, "key_bytes must be 8, 16 or 32");
    KMG_REQUIRE(range.min_count >= 1 && range.min_count <= range.max_count, KMG_ERR_ARG, "bad count range [%u, %u]",
                range.min_count, range.max_count);
    KMG_REQUIRE(d_n_out, KMG_ERR_ARG, "d_n_out is null");
    KMG_CUDA(cudaMemsetAsync(d_n_out, 0, sizeof(uint64_t), st));
    if (n == 0) return KMG_OK;
    KMG_REQUIRE(d_keys && d_counts && d_keys_out && d_counts_out && d_ws, KMG_ERR_ARG, "null pointer argument");
    KMG_REQUIRE(ws_bytes >= kmg_rle_workspace_bytes(n), KMG_ERR_WS, "filter workspace too small");
    const uint64_t tile = key_bytes == 8 ? RLE_BLOCK * RLE_IPT8 : RLE_BLOCK * RLE_IPT16;
    const uint64_t nt = (n + tile - 1) / tile;
    KMG_REQUIRE(nt < (1ull << 31), KMG_ERR_RANGE, "too many tiles");
    // header (ticket, status word) | tile prefix state: inside kmg_rle_workspace_bytes(n) for tiles of >= 2048 rows
    const size_t state_bytes = sc_state_words(nt) * sizeof(uint64_t);
    KMG_CUDA(cudaMemsetAsync(d_ws, 0, sizeof(WsHeader) + state_bytes, st));
    WsHeader* hdr = reinterpret_cast<WsHeader*>(d_ws);
    FilterParams p;
    p.keys_in = d_keys;
    p.counts_in = d_counts;
    p.keys_out = d_keys_out;
    p.counts_out = d_counts_out;
    p.n = n;
    p.n_tiles = (uint32_t)nt;
    p.min_count = range.min_count;
    p.max_count = range.max_count;
    p.n_out = reinterpret_cast<unsigned long long*>(d_n_out);
    p.tile_state = reinterpret_cast<uint64_t*>((char*)d_ws + sizeof(WsHeader));
    p.ticket = &hdr->ticket;
    p.err = &hdr->err;
    if (key_bytes == 8) filter_counts_kernel<uint64_t, RLE_IPT8><<<p.n_tiles, RLE_BLOCK, 0, st>>>(p);
    else if (key_bytes == 16) filter_counts_kernel<u128, RLE_IPT16><<<p.n_tiles, RLE_BLOCK, 0, st>>>(p);
    else filter_counts_kernel<u256, RLE_IPT16><<<p.n_tiles, RLE_BLOCK, 0, st>>>(p);
    KMG_LAUNCH_CHECK();
    return KMG_OK;
}

extern "C" int kmg_filter_counts(const void* d_keys, const uint32_t* d_counts, uint64_t n, int key_bytes, uint32_t min_count,
                                 uint32_t max_count, void* d_keys_out, uint32_t* d_counts_out, uint64_t* d_n_out, void* d_ws,
                                 size_t ws_bytes, void* stream) {
    return filter_counts(d_keys, d_counts, n, key_bytes, CountRange{min_count, max_count}, d_keys_out, d_counts_out, d_n_out,
                         d_ws, ws_bytes, (cudaStream_t)stream);
}
