// Hybrid finish of the radix sort: tile bounds, the shared-memory local sort (with its fused
// count / singleton emission) and the helpers that re-sort irregular tiles.  Included by
// radix_sort.cu (inside namespace kmg, after ValType); the host orchestration is sort_impl() there.
#pragma once

// ---- hybrid finish: after the keys are sorted by their top PB bits ---------------------------------
// Every LSD pass pays the full per-key ranking cost again.  For key-only sorts the tail can be
// cheaper: once the top PB = 16 or 24 bits are in order (2-3 ordinary passes), equal-prefix
// buckets are contiguous and small, and a tile of a few thousand keys can finish ALL remaining
// bits at once in shared memory: a counting sort into as many cells as the tile can hold keys
// (monotone key -> cell map, plain shared atomics -- no stability needed) followed by an insertion
// sort of each thread's consecutive cells.  Tiles whose buckets do not fit the scheme (long runs
// of one prefix, crowded cells: repeats) are flagged; the caller re-sorts their ranges with the
// plain LSD passes, so correctness never depends on the data.
// Tile geometry.  PAIRS: a 4- or 8-byte payload follows its key through a 16-bit index array
// (kmg_sort_uniq), which costs shared memory: smaller tiles.
template <typename KeyT, bool PAIRS>
struct LS;
template <>
struct LS<uint64_t, false> {
    static constexpr int IPT = 16;  // keys per thread
    static constexpr int CPT = 16;  // consecutive cells per thread in the prefix / cell-sort phases
};
template <>
struct LS<u128, false> {
    static constexpr int IPT = 8;
    static constexpr int CPT = 8;
};
template <>
struct LS<uint64_t, true> {
    static constexpr int IPT = 12;
    static constexpr int CPT = 12;
};
template <>
struct LS<u128, true> {  // uniq at k > 32
    static constexpr int IPT = 8;
    static constexpr int CPT = 8;
};
constexpr int LS_BLOCK = 512;
template <typename KeyT, bool PAIRS>
__host__ __device__ constexpr int ls_cap() { return LS_BLOCK * LS<KeyT, PAIRS>::IPT; }  // keys a tile can own
template <typename KeyT, bool PAIRS>
__host__ __device__ constexpr int ls_cells() { return LS_BLOCK * LS<KeyT, PAIRS>::CPT; }
// cell counters are padded so that one thread's consecutive cells are conflict-free 128-bit
// accesses: thread stride 16 + 4 = 20 words, 8 + 4 = 12 words, 12 words (no padding needed)
template <typename KeyT, bool PAIRS>
__device__ __forceinline__ uint32_t pc(uint32_t c) {
    constexpr int CPT = LS<KeyT, PAIRS>::CPT;
    return CPT == 16 ? c + ((c >> 4) << 2) : (CPT == 8 ? c + ((c >> 3) << 2) : c);
}
template <typename KeyT, bool PAIRS>
__host__ __device__ constexpr int ls_cell_words() {
    return ls_cells<KeyT, PAIRS>() + (LS<KeyT, PAIRS>::CPT == 12 ? 0 : ls_cells<KeyT, PAIRS>() / LS<KeyT, PAIRS>::CPT * 4) + 4;
}
template <typename KeyT, bool PAIRS>
__host__ __device__ constexpr size_t ls_smem_bytes() {
    return sizeof(KeyT) * ls_cap<KeyT, PAIRS>() + sizeof(uint32_t) * ls_cell_words<KeyT, PAIRS>() +
           (PAIRS ? sizeof(uint16_t) * ls_cap<KeyT, PAIRS>() : 0);
}
constexpr int LS_T_MIN = 1024;             // smallest run-time tile width (workspace sizing)
constexpr int LS_THREAD_RUN_MAX = 24;      // keys a thread insertion-sorts itself
constexpr int LS_WARP_RUN_MAX = 128;       // keys a warp rank-sorts; longer runs go to the whole block
constexpr int LS_MAX_BIG = 48;             // such runs per tile (more: the tile gives up)

// low 64 bits of (key >> s): prefix / cell arithmetic works modulo 2^64 (keys agree above end_bit)
__device__ __forceinline__ uint64_t shr64(uint64_t k, int s) { return k >> s; }
__device__ __forceinline__ uint64_t shr64(const u128& k, int s) {
    if (s >= 64) return k.hi >> (s - 64);
    if (s == 0) return k.lo;
    return (k.lo >> s) | (k.hi << (64 - s));
}

struct HybridParams {
    const void* keys_in;
    void* keys_out;
    const void* vals_in;    // payload sorts (local_sort_kernel<.., VB != 0>)
    void* vals_out;
    uint64_t n;
    uint64_t* bounds;       // [n_tiles + 1], see tile_bounds_kernel
    uint32_t* flag;         // [n_tiles] 1 = the local scheme could not hold the tile (zeroed by the host)
    uint64_t* off;          // [n_tiles + 1] offsets of the flagged tiles' keys in the gather buffer
    uint32_t n_tiles;
    uint32_t tile_t;        // positions per tile
    int key_bits, pb;
    unsigned long long* irregular;  // [0] tiles the local scheme could not handle, [1] runs the block had to sort
    unsigned long long* over;       // [0] tiles that own more keys than the local sort holds, [1] their keys
                                    // (oversize_tiles_kernel); a fused launch stands down when there are any
    unsigned long long* n_out_copy; // second home of *n_out, next to the status words the host reads back
    // fused run-length count (local_sort_kernel<.., true>): distinct keys -> keys_out, compacted
    uint32_t* counts_out;
    unsigned long long* n_out;      // number of distinct keys
    uint64_t* tile_state;           // tile prefix over the tiles' distinct-key counts
    uint32_t* ticket;
    uint32_t* err;
    HistoOut histo;                 // multiplicity histogram (EMIT 3)
    uint32_t min_count, max_count;  // EMIT 4: the rows of the count table that are kept
    uint32_t pad[2];                // (keeps the parameters that follow HybridParams 16-byte aligned as before)
};

// ---- multiplicity histogram (EMIT 3, kmg_sort_histo, kmg_count_histogram) ---------------------------
// The small multiplicities (nearly all of them) go to per-CTA shared bins that are flushed with one
// global atomic per non-empty bin; larger ones take a global atomic, and those >= KMG_HISTO_BINS an entry
// of the `big` list.
constexpr int HISTO_SMEM_BINS = 64;
__device__ __forceinline__ void histo_add_global(const HistoOut& h, uint64_t m) {
    if (m < (uint64_t)KMG_HISTO_BINS) atomicAdd(&h.hist[m], 1ull);
    else if (m <= 0xFFFFFFFFull) h.big[atomicAdd(h.n_big, 1ull)] = (uint32_t)m;
    else atomicMax(h.err, 2u);  // (the count path's limit: a multiplicity must fit uint32)
}
__device__ __forceinline__ void histo_add(uint32_t* s_h, const HistoOut& h, uint64_t m) {
    if (m < (uint64_t)HISTO_SMEM_BINS) atomicAdd(&s_h[m], 1u);
    else histo_add_global(h, m);
}
__device__ __forceinline__ void histo_flush(const uint32_t* s_h, const HistoOut& h) {
    for (uint32_t i = threadIdx.x; i < (uint32_t)HISTO_SMEM_BINS; i += blockDim.x)
        if (s_h[i]) atomicAdd(&h.hist[i], (unsigned long long)s_h[i]);
}

// First i in [lo, hi) whose prefix differs from `ref`, or hi; the prefixes are non-decreasing.
// Whole-warp 32-ary search: the common case (buckets of a few keys) ends after one probe round.
template <typename KeyT>
__device__ __forceinline__ uint64_t prefix_run_end(const KeyT* __restrict__ keys, uint64_t lo, uint64_t hi,
                                                   uint64_t ref, int sh) {
    const uint32_t lane = threadIdx.x & 31u;
    uint64_t step = 1;  // first round: 32 consecutive keys
    while (lo < hi) {
        const uint64_t i = lo + lane * step;
        const bool ne = i < hi ? shr64(keys[i], sh) != ref : true;
        const uint32_t bal = __ballot_sync(0xffffffffu, ne);
        const uint32_t first = bal ? __ffs(bal) - 1 : 32u;  // 32: all probes still match
        if (first == 0) return lo;
        if (step == 1) {
            if (first < 32) return min(lo + first, hi);
            lo += 32;
        } else {
            const uint64_t nlo = lo + (uint64_t)(first - 1) * step + 1;
            hi = first < 32 ? min(hi, lo + (uint64_t)first * step) : hi;
            lo = nlo;
        }
        const uint64_t span = hi - lo;
        step = span <= 32 ? 1 : (span + 31) / 32;
    }
    return hi;
}

// bounds[tile] = first position >= tile * tile_t where a new prefix bucket starts (one warp per tile);
// tile owns [bounds[tile], bounds[tile + 1])
template <typename KeyT>
__global__ void __launch_bounds__(256) tile_bounds_kernel(const HybridParams p) {
    const uint32_t tile = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (tile > p.n_tiles) return;
    const KeyT* keys_in = reinterpret_cast<const KeyT*>(p.keys_in);
    const uint32_t lane = threadIdx.x & 31u;
    const int sh_pref = p.key_bits - p.pb;
    const uint64_t pos = min((uint64_t)tile * p.tile_t, p.n);
    uint64_t r = pos;
    if (pos > 0 && pos < p.n) {
        const uint64_t hi = p.n;  // exact even for long runs: irregular tiles are re-sorted range by range
        // one round trip in the common case: keys[pos-1 .. pos+30]
        const uint64_t i = pos - 1 + lane;
        const uint64_t v = i < hi ? shr64(keys_in[i], sh_pref) : ~0ull;
        const uint64_t ref = __shfl_sync(0xffffffffu, v, 0);
        const uint32_t bal = __ballot_sync(0xffffffffu, v != ref);
        r = bal ? min(pos - 1 + (uint64_t)(__ffs(bal) - 1), hi) : prefix_run_end(keys_in, pos + 31, hi, ref, sh_pref);
    }
    if (lane == 0) p.bounds[tile] = r;
}

// The same bounds for keys whose bucket starts are known (the fused pipeline's pre-pass):
// starts[0 .. n_buckets] (starts[n_buckets] = n), so the first bucket start >= tile * tile_t is one
// binary search -- an empty bucket starts where the next non-empty one does
__global__ void __launch_bounds__(256) bounds_from_starts_kernel(const HybridParams p, const unsigned long long* __restrict__ starts,
                                                                 uint32_t n_buckets) {
    const uint32_t tile = blockIdx.x * blockDim.x + threadIdx.x;
    if (tile > p.n_tiles) return;
    const uint64_t pos = min((uint64_t)tile * p.tile_t, p.n);
    uint32_t lo = 0, hi = n_buckets;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (starts[mid] >= pos) hi = mid;
        else lo = mid + 1;
    }
    p.bounds[tile] = min((uint64_t)starts[lo], p.n);
}

// Tiles that own more keys than the local sort holds are known from the bounds alone: count them
// before the launch so that a fused count is not attempted in vain (repeats: real genomes always
// have some).  The local sort flags them again, together with the rare crowded-cell tiles.
__global__ void __launch_bounds__(256) oversize_tiles_kernel(const HybridParams p, uint32_t cap, unsigned long long* over) {
    const uint32_t tile = blockIdx.x * blockDim.x + threadIdx.x;
    if (tile >= p.n_tiles) return;
    const uint64_t s = p.bounds[tile], e = p.bounds[tile + 1];
    if (s < min((uint64_t)(tile + 1) * p.tile_t, p.n) && e > s && e - s > cap) {
        atomicAdd(&over[0], 1ull);              // tiles
        atomicAdd(&over[1], (unsigned long long)(e - s));  // keys
    }
}

// monotone map key -> cell of the tile's counting sort (see local_sort_kernel)
template <typename KeyT, int CELLS>
struct CellMap {
    uint64_t base;   // b_lo << w
    uint32_t inv;    // 0: cell = x, else cell = umulhi(x, inv)
    int sh;          // x = (key >> sh) - base
    __device__ __forceinline__ uint32_t operator()(const KeyT& key) const {
        const uint32_t x = (uint32_t)(shr64(key, sh) - base);
        // (the clamp only matters for keys that break the contract: bits >= end_bit not all equal)
        return min(inv ? __umulhi(x, inv) : x, (uint32_t)CELLS - 1u);
    }
};

// COUNT: instead of the sorted keys the tile writes its DISTINCT keys and their multiplicities,
// compacted across tiles with the tile prefix (a run of equal keys never leaves its prefix bucket,
// hence never its tile): kmg_rle_count's result without writing and re-reading the sorted keys.
// Tiles take their ids from a ticket so that waiting for earlier tiles is safe.
// VB != 0: the payload (4 or 8 bytes) follows its key: a 16-bit index array travels with the
// staged keys and the payload is gathered from the tile's (L2-resident) input range at the end.
// Equal keys come out in no particular order (kmg_sort_uniq only keeps keys that occur once).
// EMIT: 0 = the sorted keys (and payload), 1 = the count table (COUNT above), 2 = the keys that
// occur exactly once with their payload, compacted across tiles like the count table (kmg_sort_uniq),
// 3 = nothing but the run lengths, added to the multiplicity histogram p.histo (kmg_sort_histo): no
// output order, so no ticket and no tile prefix, and a tile the scheme cannot hold adds nothing (the
// host re-sorts its range and histograms it on the side), 4 = the count table restricted to the rows with
// p.min_count <= count <= p.max_count, compacted across tiles like the full table.
template <typename KeyT, int EMIT, int VB>
__global__ void __launch_bounds__(LS_BLOCK, 2) local_sort_kernel(const HybridParams p) {
    constexpr bool PAIRS = VB != 0;
    constexpr bool COUNT = EMIT == 1, UNIQ = EMIT == 2, HISTO = EMIT == 3, RANGE = EMIT == 4;
    constexpr bool FUSED = EMIT == 1 || EMIT == 2 || EMIT == 4;
    static_assert(!(PAIRS && (COUNT || HISTO || RANGE)), "the fused count and histogram are key-only");
    static_assert(!UNIQ || PAIRS, "singletons carry their payload");
    constexpr int IPT = LS<KeyT, PAIRS>::IPT, CPT = LS<KeyT, PAIRS>::CPT;
    constexpr int CAP = ls_cap<KeyT, PAIRS>(), CELLS = ls_cells<KeyT, PAIRS>(), CELL_WORDS = ls_cell_words<KeyT, PAIRS>();
    constexpr int CELL_BITS = CELLS > 4096 ? 13 : 12;
    static_assert((1 << CELL_BITS) >= CELLS && CAP <= (1 << 16), "cell / index widths");
    using ValT = typename ValType<VB == 0 ? 8 : VB>::type;
    extern __shared__ __align__(16) unsigned char ls_smem[];
    KeyT* s_stage = reinterpret_cast<KeyT*>(ls_smem);                                 // [CAP]
    uint32_t* s_cell = reinterpret_cast<uint32_t*>(ls_smem + sizeof(KeyT) * CAP);     // [CELL_WORDS]
    uint16_t* s_idx = reinterpret_cast<uint16_t*>(s_cell + CELL_WORDS);               // [CAP] (PAIRS)
    __shared__ uint32_t s_scan[LS_BLOCK / 32 + 1];
    __shared__ int s_bad;
    __shared__ uint32_t s_tile;
    __shared__ uint64_t s_base;
    __shared__ uint32_t s_big_n;
    __shared__ uint32_t s_big[LS_MAX_BIG][2];
    const int t = threadIdx.x;
    const int sh_pref = p.key_bits - p.pb;
    // a fused table cannot be patched up afterwards: with oversize tiles around the host falls back to
    // sort + run-length stage, and this launch has nothing to do (every CTA takes the same exit)
    if (FUSED && p.over[0] != 0) return;

    if (t == 0) {
        s_bad = 0;
        s_big_n = 0;
        if (FUSED) s_tile = atomicAdd(p.ticket, 1u);
    }
    {
        uint4* z = reinterpret_cast<uint4*>(s_cell);
        for (uint32_t i = t; i < (uint32_t)CELL_WORDS / 4; i += LS_BLOCK) z[i] = make_uint4(0, 0, 0, 0);
    }
    if (FUSED) __syncthreads();
    const uint32_t tile = FUSED ? s_tile : blockIdx.x;
    // a tile without output still takes part in the tile prefix (and the last one reports the total)
    auto finish_without_output = [&]() {
        if constexpr (FUSED) {
            if (t < 32) {
                if (t == 0) tile_prefix_publish(p.tile_state, tile, 0);
                const uint64_t base = tile_prefix_resolve_warp(p.tile_state, p.n_tiles, tile, 0, p.err);
                if (t == 0 && tile == p.n_tiles - 1) *p.n_out = *p.n_out_copy = base;
            }
        }
    };
    const uint64_t s = p.bounds[tile], e = p.bounds[tile + 1];
    if (s >= min((uint64_t)(tile + 1) * p.tile_t, p.n) || e <= s) {  // no bucket starts in this tile
        finish_without_output();
        return;
    }
    const uint64_t m64 = e - s;
    if (m64 > (uint64_t)CAP) {
        if (t == 0) {
            atomicAdd(p.irregular, 1ull);
            p.flag[tile] = 1;
        }
        finish_without_output();
        return;
    }
    const uint32_t m = (uint32_t)m64;
    const KeyT* kin = reinterpret_cast<const KeyT*>(p.keys_in) + s;
    const uint64_t p_first = shr64(kin[0], sh_pref), p_last = shr64(kin[m - 1], sh_pref);
    KeyT keys[IPT];
#pragma unroll
    for (int j = 0; j < IPT; ++j) {
        const uint32_t idx = t + j * LS_BLOCK;
        keys[j] = idx < m ? kin[idx] : KeyT{};
    }
    // Counting sort into <= CELLS cells through a monotone map of the key: the w bits after the
    // prefix, relative to the tile's first bucket, scaled down to the cell range when the tile
    // spans more than CELLS such values.  Monotone, so sorting inside cells finishes it.
    CellMap<KeyT, CELLS> cm;
    {
        const uint64_t R = p_last - p_first + 1;  // <= 2^24
        int w = min(CELL_BITS, sh_pref);
        w = max(0, min(w, 30 - (63 - __clzll((long long)R))));  // (R << w) < 2^31
        cm.sh = sh_pref - w;
        cm.base = p_first << w;
        const uint64_t range = R << w;
        cm.inv = range <= (uint64_t)CELLS ? 0u : (uint32_t)((((uint64_t)CELLS) << 32) / range);
    }
    __syncthreads();     // cells are zero
#pragma unroll
    for (int j = 0; j < IPT; ++j) {
        if (t + j * LS_BLOCK < m) atomicAdd(&s_cell[pc<KeyT, PAIRS>(cm(keys[j]))], 1u);
    }
    __syncthreads();
    // exclusive prefix over the cells: CPT consecutive cells per thread, 128 bits at a time
    uint4* cv = reinterpret_cast<uint4*>(s_cell + pc<KeyT, PAIRS>(t * CPT));
    uint4 q[CPT / 4];
    uint32_t sum = 0;
#pragma unroll
    for (int i = 0; i < CPT / 4; ++i) {
        q[i] = cv[i];
        sum += q[i].x + q[i].y + q[i].z + q[i].w;
    }
    uint32_t total;
    uint32_t run = block_excl_scan<LS_BLOCK, uint32_t>(sum, s_scan, total);
#pragma unroll
    for (int i = 0; i < CPT / 4; ++i) {
        uint32_t v;
#define KMG_LS_STEP(f) v = f; f = run; run += v;
        KMG_LS_STEP(q[i].x) KMG_LS_STEP(q[i].y) KMG_LS_STEP(q[i].z) KMG_LS_STEP(q[i].w)
#undef KMG_LS_STEP
        cv[i] = q[i];
    }
    __syncthreads();
    // Placement: a second atomic on the cell's running start hands out the slots (arrival order), so
    // nothing but the keys lives in registers between the phases -- a per-key (cell, slot) word kept
    // from the counting pass cost 16 more registers and spilled under the 64-register cap
    // (profiles/r02_ncu_local_sort_experiments.md).  Afterwards a cell's word is its END.
#pragma unroll
    for (int j = 0; j < IPT; ++j) {
        const uint32_t idx = t + j * LS_BLOCK;
        if (idx < m) {
            const uint32_t at = atomicAdd(&s_cell[pc<KeyT, PAIRS>(cm(keys[j]))], 1u);
            s_stage[at] = keys[j];
            if constexpr (PAIRS) s_idx[at] = (uint16_t)idx;
        }
    }
    __syncthreads();
    // Order every cell in place.  The cells are already in order among themselves, so a thread
    // simply insertion-sorts the contiguous run of its CPT cells (~11 / ~6 keys): a key moves only
    // inside its own cell, equal keys cost one compare each.
    const uint32_t lo = t ? s_cell[pc<KeyT, PAIRS>(t * CPT - 1)] : 0u, hi = s_cell[pc<KeyT, PAIRS>((t + 1) * CPT - 1)];
    // COUNT: equal keys share a cell, hence a thread's run, so the run heads (distinct keys) can be
    // counted while inserting: a key is new unless it lands right after an equal one
    uint32_t hc = 0;
    bool my_run_is_big = false;   // sorted by the warp or by the block: heads are recounted afterwards
    const uint32_t run_len = hi - lo;
    // Who sorts a run: its thread by insertion (the normal ~11 keys), its WARP by rank sort when it
    // holds 25..128 keys (a crowded cell: near-copies of a repeat; one thread would spend hundreds of
    // serial moves while the block waits), the whole BLOCK (bitonic, below) beyond that.
    const bool by_block = run_len > (uint32_t)LS_WARP_RUN_MAX;
    const bool by_warp = !by_block && run_len > (uint32_t)LS_THREAD_RUN_MAX;
    uint32_t warp_runs = __ballot_sync(0xffffffffu, by_warp);
    if (by_block) {
        my_run_is_big = true;
        const uint32_t slot = atomicAdd(&s_big_n, 1u);
        if (slot < (uint32_t)LS_MAX_BIG) {
            s_big[slot][0] = lo;
            s_big[slot][1] = hi;
        } else {
            s_bad = 1;
        }
    } else if (by_warp) {
        my_run_is_big = true;
    } else {
        KeyT prev{};
        for (uint32_t i = lo; i < hi; ++i) {
            const KeyT key = s_stage[i];
            if (!(key < prev)) {
                if (COUNT) hc += (i == lo || key != prev) ? 1u : 0u;
                prev = key;
                continue;
            }
            uint32_t qi = i;
            KeyT below{};
            bool more;
            uint16_t my_idx = 0;
            if constexpr (PAIRS) my_idx = s_idx[i];
            do {
                s_stage[qi] = s_stage[qi - 1];
                if constexpr (PAIRS) s_idx[qi] = s_idx[qi - 1];
                --qi;
                more = qi > lo;
                if (more) below = s_stage[qi - 1];
            } while (more && key < below);
            s_stage[qi] = key;
            if constexpr (PAIRS) s_idx[qi] = my_idx;
            if (COUNT) hc += (!more || below != key) ? 1u : 0u;
        }
    }
    while (warp_runs) {  // (warp-uniform)
        const int src = __ffs(warp_runs) - 1;
        warp_runs &= warp_runs - 1;
        const uint32_t rlo = __shfl_sync(0xffffffffu, lo, src), rlen = __shfl_sync(0xffffffffu, run_len, src);
        constexpr int Q = LS_WARP_RUN_MAX / 32;
        const uint32_t lane = t & 31u;
        KeyT kq[Q];
        uint32_t rk[Q];
        uint16_t iq[Q];
#pragma unroll
        for (int q = 0; q < Q; ++q) {
            const uint32_t e = lane + 32u * q;
            kq[q] = e < rlen ? s_stage[rlo + e] : KeyT{};
            if constexpr (PAIRS) iq[q] = e < rlen ? s_idx[rlo + e] : (uint16_t)0;
            rk[q] = 0;
        }
        for (uint32_t j = 0; j < rlen; ++j) {
            const KeyT o = s_stage[rlo + j];  // one address for the whole warp: a broadcast
#pragma unroll
            for (int q = 0; q < Q; ++q) rk[q] += (o < kq[q] || (o == kq[q] && j < lane + 32u * q)) ? 1u : 0u;
        }
        __syncwarp();  // every lane has read the run
#pragma unroll
        for (int q = 0; q < Q; ++q) {
            if (lane + 32u * q < rlen) {
                s_stage[rlo + rk[q]] = kq[q];
                if constexpr (PAIRS) s_idx[rlo + rk[q]] = iq[q];
            }
        }
        __syncwarp();
    }
    __syncthreads();
    if (s_big_n != 0 && !s_bad) {
        // bitonic sort of every big run by the whole block, in the (now dead) cell array, padded to a
        // power of two with all-ones keys (O(s log^2 s): a repeat family puts hundreds of distinct
        // keys into one cell, and there are thousands of such cells in a genome)
        constexpr uint32_t TEMP_CAP = (uint32_t)(CELL_WORDS * sizeof(uint32_t) / (sizeof(KeyT) + (PAIRS ? 2 : 0)));
        constexpr uint32_t TEMP_POW2 = TEMP_CAP >= 4096 ? 4096 : (TEMP_CAP >= 2048 ? 2048 : 1024);
        static_assert(TEMP_POW2 <= TEMP_CAP, "bitonic buffer");
        KeyT* tmp_k = reinterpret_cast<KeyT*>(s_cell);
        uint16_t* tmp_i = reinterpret_cast<uint16_t*>(tmp_k + TEMP_POW2);
        const uint32_t nb = s_big_n;
        if (t == 0) atomicAdd(&p.irregular[1], (unsigned long long)nb);
        for (uint32_t b = 0; b < nb; ++b) {
            const uint32_t blo = s_big[b][0], sz = s_big[b][1] - blo;
            if (sz > TEMP_POW2) {
                s_bad = 1;  // (every thread takes the same branch)
                break;
            }
            uint32_t N = 64;
            while (N < sz) N <<= 1;
            for (uint32_t e = t; e < N; e += LS_BLOCK) {
                tmp_k[e] = e < sz ? s_stage[blo + e] : key_all_ones(KeyT{});
                if constexpr (PAIRS) tmp_i[e] = e < sz ? s_idx[blo + e] : (uint16_t)0xFFFF;  // padding sorts last
            }
            __syncthreads();
            for (uint32_t kk = 2; kk <= N; kk <<= 1) {
                for (uint32_t jj = kk >> 1; jj > 0; jj >>= 1) {
                    for (uint32_t e = t; e < N / 2; e += LS_BLOCK) {
                        // e-th compare-exchange of this stage: partner indices i < l = i ^ jj
                        const uint32_t i = ((e & ~(jj - 1)) << 1) | (e & (jj - 1));
                        const uint32_t l = i | jj;
                        const bool up = (i & kk) == 0;
                        const KeyT a0 = tmp_k[i], a1 = tmp_k[l];
                        bool less = a1 < a0;
                        if constexpr (PAIRS) {  // total order (key, index): the padding can never displace a real pair
                            const uint16_t i0 = tmp_i[i], i1 = tmp_i[l];
                            less = less || (a1 == a0 && i1 < i0);
                            if (less == up) {
                                tmp_i[i] = i1;
                                tmp_i[l] = i0;
                            }
                        }
                        if (less == up) {
                            tmp_k[i] = a1;
                            tmp_k[l] = a0;
                        }
                    }
                    __syncthreads();
                }
            }
            for (uint32_t e = t; e < sz; e += LS_BLOCK) {
                s_stage[blo + e] = tmp_k[e];
                if constexpr (PAIRS) s_idx[blo + e] = tmp_i[e];
            }
            __syncthreads();
        }
    }
    if (COUNT && my_run_is_big && !s_bad) {  // heads of my run, now that the warp / the block has sorted it
        hc = 0;
        KeyT prev{};
        for (uint32_t i = lo; i < hi; ++i) {
            const KeyT key = s_stage[i];
            hc += (i == lo || key != prev) ? 1u : 0u;
            prev = key;
        }
    }
    __syncthreads();
    if (s_bad) {  // too many distinct keys crowded into one cell: leave the tile to the fallback
        if (t == 0) {
            atomicAdd(p.irregular, 1ull);
            p.flag[tile] = 1;
        }
        finish_without_output();
        return;
    }
    if constexpr (HISTO) {
        // a run of equal keys lies inside one thread's run of cells: every thread measures its own runs
        uint32_t* s_h = s_cell;  // [HISTO_SMEM_BINS] (the cell array is dead by now)
        if (t < HISTO_SMEM_BINS) s_h[t] = 0;
        __syncthreads();
        uint32_t start = lo;
        KeyT prev{};
        for (uint32_t i = lo; i < hi; ++i) {
            const KeyT key = s_stage[i];
            if (i != lo && key != prev) {
                histo_add(s_h, p.histo, i - start);
                start = i;
            }
            prev = key;
        }
        if (hi > lo) histo_add(s_h, p.histo, hi - start);
        __syncthreads();
        histo_flush(s_h, p.histo);
    } else if constexpr (!FUSED) {
        KeyT* kout = reinterpret_cast<KeyT*>(p.keys_out) + s;
#pragma unroll
        for (int j = 0; j < IPT; ++j) {
            const uint32_t idx = t + j * LS_BLOCK;
            if (idx < m) kout[idx] = s_stage[idx];
        }
        if constexpr (PAIRS) {
            const ValT* vin = reinterpret_cast<const ValT*>(p.vals_in) + s;
            ValT* vout = reinterpret_cast<ValT*>(p.vals_out) + s;
#pragma unroll
            for (int j = 0; j < IPT; ++j) {
                const uint32_t idx = t + j * LS_BLOCK;
                if (idx < m) vout[idx] = vin[s_idx[idx]];
            }
        }
    } else if constexpr (RANGE) {
        // the runs whose length is in range: every thread measures its own runs (as the histogram does),
        // a block scan ranks the kept ones, and every thread writes its own after the tile prefix
        auto walk = [&](auto&& emit) {
            uint32_t start = lo;
            KeyT prev{};
            for (uint32_t i = lo; i < hi; ++i) {
                const KeyT key = s_stage[i];
                if (i != lo && key != prev) {
                    if (i - start >= p.min_count && i - start <= p.max_count) emit(start, i - start);
                    start = i;
                }
                prev = key;
            }
            if (hi > lo && hi - start >= p.min_count && hi - start <= p.max_count) emit(start, hi - start);
        };
        uint32_t hk = 0;
        walk([&](uint32_t, uint32_t) { ++hk; });
        uint32_t H;
        uint32_t hoff = block_excl_scan<LS_BLOCK, uint32_t>(hk, s_scan, H);
        if (t == 0) tile_prefix_publish(p.tile_state, tile, H);
        if (t < 32) {
            const uint64_t base = tile_prefix_resolve_warp(p.tile_state, p.n_tiles, tile, H, p.err);
            if (t == 0) {
                s_base = base;
                if (tile == p.n_tiles - 1) *p.n_out = *p.n_out_copy = base + H;
            }
        }
        __syncthreads();
        const uint64_t base = s_base;
        KeyT* kout = reinterpret_cast<KeyT*>(p.keys_out);
        walk([&](uint32_t i, uint32_t len) {
            kout[base + hoff] = s_stage[i];
            p.counts_out[base + hoff] = len;
            ++hoff;
        });
    } else if constexpr (UNIQ) {
        // keys that occur once: a run of equal keys lies inside one thread's run, so every thread
        // finds the singletons of its own run; a block scan ranks them, the tile prefix places them
        uint32_t* s_pos = s_cell;  // [m] positions of the singletons in order (the cell array is dead by now)
        static_assert(CAP <= CELL_WORDS, "singleton positions must fit the cell array");
        auto walk = [&](auto&& emit) {
            KeyT prev{}, key{}, next{};
            if (lo < hi) next = s_stage[lo];
            for (uint32_t i = lo; i < hi; ++i) {
                key = next;
                const bool last = i + 1 == hi;
                if (!last) next = s_stage[i + 1];
                if ((i == lo || key != prev) && (last || key != next)) emit(i);
                prev = key;
            }
        };
        uint32_t hs = 0;
        walk([&](uint32_t) { ++hs; });
        uint32_t S;
        uint32_t soff = block_excl_scan<LS_BLOCK, uint32_t>(hs, s_scan, S);  // (barriers: everyone is done with s_cell)
        if (t == 0) tile_prefix_publish(p.tile_state, tile, S);
        walk([&](uint32_t i) { s_pos[soff++] = i; });
        if (t < 32) {
            const uint64_t base = tile_prefix_resolve_warp(p.tile_state, p.n_tiles, tile, S, p.err);
            if (t == 0) {
                s_base = base;
                if (tile == p.n_tiles - 1) *p.n_out = *p.n_out_copy = base + S;
            }
        }
        __syncthreads();
        const uint64_t base = s_base;
        KeyT* kout = reinterpret_cast<KeyT*>(p.keys_out);
        const ValT* vin = reinterpret_cast<const ValT*>(p.vals_in) + s;
        ValT* vout = reinterpret_cast<ValT*>(p.vals_out);
        for (uint32_t h = t; h < S; h += LS_BLOCK) {
            const uint32_t i = s_pos[h];
            kout[base + h] = s_stage[i];
            vout[base + h] = vin[s_idx[i]];
        }
    } else {
        // the runs tile [0, m) in thread order, so a block scan of the per-thread head counts ranks
        // the heads; a second walk over the (now sorted) run records their positions
        uint32_t* s_pos = s_cell;  // [m] positions of the heads in order (the cell array is dead by now)
        static_assert(CAP <= CELL_WORDS, "head positions must fit the cell array");
        uint32_t H;
        uint32_t hoff = block_excl_scan<LS_BLOCK, uint32_t>(hc, s_scan, H);  // (barriers: everyone is done with s_cell)
        if (t == 0) tile_prefix_publish(p.tile_state, tile, H);
        {
            KeyT prev{};
            for (uint32_t i = lo; i < hi; ++i) {
                const KeyT key = s_stage[i];
                if (i == lo || key != prev) s_pos[hoff++] = i;  // (a run's first key differs from every other run's keys)
                prev = key;
            }
        }
        if (t < 32) {
            const uint64_t base = tile_prefix_resolve_warp(p.tile_state, p.n_tiles, tile, H, p.err);
            if (t == 0) {
                s_base = base;
                if (tile == p.n_tiles - 1) *p.n_out = *p.n_out_copy = base + H;
            }
        }
        __syncthreads();
        const uint64_t base = s_base;
        KeyT* kout = reinterpret_cast<KeyT*>(p.keys_out);
        for (uint32_t h = t; h < H; h += LS_BLOCK) {
            const uint32_t i = s_pos[h], nxt = h + 1 < H ? s_pos[h + 1] : m;
            kout[base + h] = s_stage[i];
            p.counts_out[base + h] = nxt - i;
        }
    }
}

// Flagged tiles: off[tile] = exclusive prefix of their key counts (one block), total in off[n_tiles]
__global__ void __launch_bounds__(1024) irregular_scan_kernel(const HybridParams p) {
    __shared__ uint64_t s_scan[33];
    const uint32_t t = threadIdx.x;
    const uint32_t per = (p.n_tiles + 1023) / 1024;
    const uint32_t b = min(t * per, p.n_tiles), e = min(b + per, p.n_tiles);
    uint64_t sum = 0;
    for (uint32_t i = b; i < e; ++i) sum += p.flag[i] ? p.bounds[i + 1] - p.bounds[i] : 0;
    uint64_t total;
    uint64_t run = block_excl_scan<1024, uint64_t>(sum, s_scan, total);
    for (uint32_t i = b; i < e; ++i) {
        p.off[i] = run;
        run += p.flag[i] ? p.bounds[i + 1] - p.bounds[i] : 0;
    }
    if (t == 0) p.off[p.n_tiles] = total;
}

// TO_BUFFER: in[bounds[tile]...] -> buf[off[tile]...] for the flagged tiles; else buf -> out (keys, and
// again for the payload).  The ranges are whole prefix buckets in ascending order, so sorting the
// gathered items and putting them back range by range leaves the output fully sorted.
template <typename T, bool TO_BUFFER>
__global__ void __launch_bounds__(256) irregular_copy_kernel(const HybridParams p, const T* __restrict__ in,
                                                             T* __restrict__ out, T* __restrict__ buf) {
    for (uint32_t tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
        if (!p.flag[tile]) continue;
        const uint64_t s = p.bounds[tile], m = p.bounds[tile + 1] - s, o = p.off[tile];
        for (uint64_t i = threadIdx.x; i < m; i += 256) {
            if (TO_BUFFER) buf[o + i] = in[s + i];
            else out[s + i] = buf[o + i];
        }
    }
}

template <bool TO_BUFFER>
static int irregular_copy(const HybridParams& hp, int item_bytes, const void* in, void* out, void* buf, int grid,
                          cudaStream_t st) {
    if (item_bytes == 16)
        irregular_copy_kernel<u128, TO_BUFFER><<<grid, 256, 0, st>>>(hp, (const u128*)in, (u128*)out, (u128*)buf);
    else if (item_bytes == 8)
        irregular_copy_kernel<uint64_t, TO_BUFFER><<<grid, 256, 0, st>>>(hp, (const uint64_t*)in, (uint64_t*)out, (uint64_t*)buf);
    else
        irregular_copy_kernel<uint32_t, TO_BUFFER><<<grid, 256, 0, st>>>(hp, (const uint32_t*)in, (uint32_t*)out, (uint32_t*)buf);
    KMG_LAUNCH_CHECK();
    return KMG_OK;
}

