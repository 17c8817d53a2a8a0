// Hybrid finish, local sort with FINE cells in a persistent two-tile pipeline (same contract, tile
// geometry and HybridParams as local_sort_kernel in local_sort.cuh; included right after it by
// radix_sort.cu).
//
// The first kernel counts the tile's keys into as many cells as keys and then WALKS every key twice (a
// per-thread insertion sort over each run of cells, then a walk that records the run heads): 5.1 warp
// instructions per key, half of them in those walks at ~40 % lane efficiency
// (profiles/r02_ncu_local_sort_experiments.md).  Two rewrites that kept one cell per key and made the
// in-cell ordering data-independent (rank by reading the cell; register sorting networks) executed MORE
// instructions, because they still touched every key.  This kernel avoids touching keys at all unless
// they collide:
//   * twice as many cells as keys (16-bit counters, two per word): a key shares its cell with another
//     one with probability ~0.39 instead of 0.63, and -- the point -- a key ALONE in its cell is already
//     in its final place after the placement;
//   * the prefix pass sees every cell's count anyway and writes the cells that hold >= 2 keys to a compact
//     list; the list (not the tile) is what gets sorted: entry by entry, a thread per cell (2..12 keys,
//     the normal case: two), a warp per cell (<= 128), the block for the rest (bitonic);
//   * equal keys always share a cell, so duplicates are found right there and recorded in a bitmask of
//     the tile's positions.  Run heads, run lengths (count) and singletons (uniq) then come from that
//     bitmask with popcounts -- position-parallel, coalesced, no key is compared again; a tile without
//     duplicates (the rule on non-repetitive sequence) is a plain copy.
// The prefix is laid out without padding: thread t owns words 4t..4t+3 of every 2048-word chunk (128-bit
// conflict-free accesses) and ONE 64-bit block scan carries the sums of all chunks in 16-bit fields.
//
// That brought the instruction count from 510 M to 424 M per 100 M keys -- and the launch from 1.13 to
// 1.33 ms: what was left were two exposed latencies per tile, the DRAM round trip of the tile's keys
// (32 % of the stall samples) and the wait for the earlier tiles' aggregates at the tile prefix (26 %).
// Hence the pipeline: CTAs are persistent, and the FRONT of the next tile (load, count, prefix) runs
// between the moment the current tile's aggregate is published and the moment its prefix is resolved:
//     placement(A) | ticket(N), L2 prefetch of N's keys (TMA) | fix-up(A) | publish(A) | load, count, prefix(N)
//     | resolve(A), emission(A) | placement(N) | ...
// N's keys travel from DRAM to L2 while A's crowded cells are sorted, and the other CTAs get a third of a
// tile's time to publish before A asks for their aggregates.
#pragma once

constexpr int LSF_THREAD_MAX = 12;   // keys of a cell its list thread insertion-sorts
constexpr int LSF_PEND = 8;          // tiles without output a CTA may skip over while it holds a tile
// counter words (one per key slot, two cells each) + the list of crowded cells (u16, at most one per two keys)
template <typename KeyT, bool PAIRS>
__host__ __device__ constexpr int lsf_cell_words() { return ls_cap<KeyT, PAIRS>() + ls_cap<KeyT, PAIRS>() / 4; }
template <typename KeyT, bool PAIRS>
__host__ __device__ constexpr size_t lsf_smem_bytes() {
    return sizeof(KeyT) * ls_cap<KeyT, PAIRS>() + sizeof(uint32_t) * lsf_cell_words<KeyT, PAIRS>() +
           (PAIRS ? sizeof(uint16_t) * ls_cap<KeyT, PAIRS>() : 0);
}

template <typename KeyT, int EMIT, int VB>
__global__ void __launch_bounds__(LS_BLOCK, 2) local_sort_fine_kernel(const HybridParams p) {
    constexpr bool PAIRS = VB != 0;
    // (EMIT 3, the histogram: tiles by stride as in the plain sort, no tile prefix; see local_sort_kernel)
    constexpr bool COUNT = EMIT == 1, UNIQ = EMIT == 2, HISTO = EMIT == 3, RANGE = EMIT == 4;
    constexpr bool FUSED = EMIT == 1 || EMIT == 2 || EMIT == 4;
    static_assert(!(PAIRS && (COUNT || HISTO || RANGE)), "the fused count and histogram are key-only");
    static_assert(!UNIQ || PAIRS, "singletons carry their payload");
    constexpr int IPT = LS<KeyT, PAIRS>::IPT;
    constexpr int CAP = ls_cap<KeyT, PAIRS>();  // keys = counter words; cells = 2 * CAP
    constexpr int CELLS = 2 * CAP;
    constexpr int CHUNKS = IPT / 4;             // 2048-word chunks of the counter array
    constexpr int CELL_BITS = 14;
    constexpr int NW = CAP / 32;                // bitmask words
    constexpr int MAX_BIG = CAP / (LS_WARP_RUN_MAX + 1) + 1;
    static_assert(IPT % 4 == 0 && CHUNKS <= 4 && CAP == LS_BLOCK * IPT && CELLS <= (1 << CELL_BITS), "geometry");
    using ValT = typename ValType<VB == 0 ? 8 : VB>::type;
    extern __shared__ __align__(16) unsigned char ls_smem[];
    KeyT* s_stage = reinterpret_cast<KeyT*>(ls_smem);                                 // [CAP]
    uint32_t* s_cell = reinterpret_cast<uint32_t*>(ls_smem + sizeof(KeyT) * CAP);     // [CAP] two 16-bit counters per word
    uint16_t* s_fix = reinterpret_cast<uint16_t*>(s_cell + CAP);                      // [CAP / 2] cells holding >= 2 keys
    uint16_t* s_idx = reinterpret_cast<uint16_t*>(s_cell + lsf_cell_words<KeyT, PAIRS>());  // [CAP] (PAIRS)
    __shared__ uint64_t s_scan64[LS_BLOCK / 32 + 1];
    __shared__ uint32_t s_scan[LS_BLOCK / 32 + 1];
    __shared__ uint32_t s_dup[NW + 1];   // bit p: position p holds the same key as position p - 1
    __shared__ uint32_t s_emit[NW];      // bit p: position p is emitted (run head / singleton)
    __shared__ uint32_t s_epre[NW];      // emitted positions before word w (HISTO: the CTA's shared bins)
    __shared__ int s_bad;
    __shared__ uint32_t s_has_mid, s_big_n, s_ndup;
    __shared__ uint32_t s_nfix[2];       // list lengths: the tile in flight / the next one
    __shared__ uint64_t s_base;
    __shared__ uint32_t s_big[MAX_BIG][2];
    // what thread 0 learns about a ticket: kind 0 = no tile left, 1 = a tile to sort, 2 = a tile without
    // output (no bucket starts in it, or it owns more keys than the scheme holds: flagged)
    __shared__ uint32_t s_t_kind, s_t_tile, s_t_m;
    __shared__ uint32_t s_pend[LSF_PEND];
    __shared__ uint64_t s_t_s;
    const int t = threadIdx.x;
    const uint32_t lane = t & 31u, warp = t >> 5;
    const int sh_pref = p.key_bits - p.pb;
    // a fused table cannot be patched up afterwards: with oversize tiles around the host falls back to
    // sort + run-length stage, and this launch has nothing to do (every CTA takes the same exit)
    if (FUSED && p.over[0] != 0) return;

    struct Tile {
        uint32_t kind, tile, m;
        uint64_t s;
    };
    uint32_t stride_next = blockIdx.x;  // (plain sort: tiles are independent, no ticket needed)
    // take the next tile id and classify it (block-wide; contains barriers)
    auto fetch = [&]() -> Tile {
        __syncthreads();  // the previous descriptor has been read by everyone
        if (t == 0) {
            const uint32_t tile = FUSED ? atomicAdd(p.ticket, 1u) : stride_next;
            uint32_t kind = 0, m = 0;
            uint64_t s = 0;
            if (tile < p.n_tiles) {
                s = p.bounds[tile];
                const uint64_t e = p.bounds[tile + 1];
                if (s >= min((uint64_t)(tile + 1) * p.tile_t, p.n) || e <= s) {
                    kind = 2;  // no bucket starts in this tile
                } else if (e - s > (uint64_t)CAP) {
                    kind = 2;
                    atomicAdd(p.irregular, 1ull);
                    p.flag[tile] = 1;
                } else {
                    kind = 1;
                    m = (uint32_t)(e - s);
                }
            }
            s_t_kind = kind;
            s_t_tile = tile;
            s_t_m = m;
            s_t_s = s;
        }
        __syncthreads();
        stride_next += gridDim.x;
        return Tile{s_t_kind, s_t_tile, s_t_m, s_t_s};
    };
    // a tile without output still takes part in the tile prefix (and the last one reports the total)
    auto publish_nothing = [&](uint32_t tile) {
        if constexpr (FUSED) {
            if (t == 0) tile_prefix_publish(p.tile_state, tile, 0);
        }
    };
    // ... but only its side effects matter: as the last tile of a group (super-group) its resolve publishes
    // the group's sum (the chained prefix), as the last tile of all the total.  Any other tile without output
    // is done once it has published its zero -- no waiting for the earlier tiles.
    auto needs_resolve = [&](uint32_t tile) { return tile % SC_GROUP == SC_GROUP - 1 || tile == p.n_tiles - 1; };
    auto resolve_nothing = [&](uint32_t tile) {
        if constexpr (FUSED) {
            if (t < 32 && needs_resolve(tile)) {
                const uint64_t base = tile_prefix_resolve_warp(p.tile_state, p.n_tiles, tile, 0, p.err);
                if (t == 0 && tile == p.n_tiles - 1) *p.n_out = *p.n_out_copy = base;
            }
        }
    };
    // next tile to SORT; tiles without output met on the way are dealt with on the spot (only legal while
    // this CTA holds no unresolved tile: see the pipeline loop)
    auto fetch_sortable = [&]() -> Tile {
        for (;;) {
            const Tile x = fetch();
            if (x.kind != 2) return x;
            publish_nothing(x.tile);
            resolve_nothing(x.tile);
        }
    };
    auto zero_cells = [&]() {
        uint4* z = reinterpret_cast<uint4*>(s_cell);
        for (uint32_t i = t; i < (uint32_t)CAP / 4; i += LS_BLOCK) z[i] = make_uint4(0, 0, 0, 0);
    };
    auto load_keys = [&](const Tile& x, KeyT (&keys)[IPT]) {
        const KeyT* kin = reinterpret_cast<const KeyT*>(p.keys_in) + x.s;
#pragma unroll
        for (int j = 0; j < IPT; ++j) {
            const uint32_t idx = t + j * LS_BLOCK;
            keys[j] = idx < x.m ? kin[idx] : KeyT{};
        }
    };
    // FRONT of a tile: counting pass (needs zeroed counters), prefix + list of crowded cells.  Leaves in
    // `meta` what every key remembers (cell | arrival order << 14); contains barriers.
    auto front = [&](const Tile& x, const KeyT (&keys)[IPT], uint32_t (&meta)[IPT], int which) {
        // monotone map key -> cell (see local_sort_kernel), onto twice as many cells
        CellMap<KeyT, CELLS> cm;
        {
            const KeyT* kin = reinterpret_cast<const KeyT*>(p.keys_in) + x.s;
            const uint64_t p_first = shr64(kin[0], sh_pref), p_last = shr64(kin[x.m - 1], sh_pref);
            const uint64_t R = p_last - p_first + 1;  // <= 2^24
            int w = min(CELL_BITS, sh_pref);
            w = max(0, min(w, 30 - (63 - __clzll((long long)R))));  // (R << w) < 2^31
            cm.sh = sh_pref - w;
            cm.base = p_first << w;
            const uint64_t range = R << w;
            cm.inv = range <= (uint64_t)CELLS ? 0u : (uint32_t)((((uint64_t)CELLS) << 32) / range);
        }
#pragma unroll
        for (int j = 0; j < IPT; ++j) {
            meta[j] = 0;
            if (t + j * LS_BLOCK < x.m) {
                const uint32_t c = cm(keys[j]);
                const uint32_t sh = (c & 1u) << 4;
                meta[j] = c | (((atomicAdd(&s_cell[c >> 1], 1u << sh) >> sh) & 0xFFFFu) << CELL_BITS);
            }
        }
        __syncthreads();
        // exclusive prefix over the counters; word = start of its even cell | count of the even cell << 16.
        // Cells that hold two keys or more are listed (one bit per cell while scanning, then the set bits).
        uint4 q[CHUNKS];
        uint64_t packed = 0;
        uint32_t crowd = 0;  // bit 8 i + 2 wi + half
#pragma unroll
        for (int i = 0; i < CHUNKS; ++i) {
            q[i] = reinterpret_cast<uint4*>(s_cell)[i * LS_BLOCK + t];
            uint32_t sum = 0;
#define KMG_LSF_SUM(f, wi)                                                    \
    sum += (f & 0xFFFFu) + (f >> 16);                                         \
    crowd |= ((f & 0xFFFEu) ? 1u : 0u) << (8 * i + 2 * wi);                   \
    crowd |= ((f & 0xFFFE0000u) ? 1u : 0u) << (8 * i + 2 * wi + 1);
            KMG_LSF_SUM(q[i].x, 0) KMG_LSF_SUM(q[i].y, 1) KMG_LSF_SUM(q[i].z, 2) KMG_LSF_SUM(q[i].w, 3)
#undef KMG_LSF_SUM
            packed |= (uint64_t)sum << (16 * i);
        }
        uint64_t total64;
        const uint64_t excl64 = block_excl_scan<LS_BLOCK, uint64_t>(packed, s_scan64, total64);
        uint32_t fix_total;
        uint32_t fat = block_excl_scan<LS_BLOCK, uint32_t>((uint32_t)__popc(crowd), s_scan, fix_total);
        uint32_t chunk_base = 0;
#pragma unroll
        for (int i = 0; i < CHUNKS; ++i) {
            uint32_t run = chunk_base + (uint32_t)((excl64 >> (16 * i)) & 0xFFFFu);
            chunk_base += (uint32_t)((total64 >> (16 * i)) & 0xFFFFu);
#define KMG_LSF_STEP(f)                                   \
    {                                                     \
        const uint32_t lo = f & 0xFFFFu, hi = f >> 16;    \
        f = run | (lo << 16);                             \
        run += lo + hi;                                   \
    }
            KMG_LSF_STEP(q[i].x) KMG_LSF_STEP(q[i].y) KMG_LSF_STEP(q[i].z) KMG_LSF_STEP(q[i].w)
#undef KMG_LSF_STEP
            reinterpret_cast<uint4*>(s_cell)[i * LS_BLOCK + t] = q[i];
        }
        while (crowd) {
            const uint32_t b = (uint32_t)__ffs(crowd) - 1u;
            crowd &= crowd - 1u;
            // bit -> cell: chunk b >> 3, word (b >> 1) & 3 of this thread's four, half b & 1
            s_fix[fat++] = (uint16_t)(2u * (((b >> 3) * LS_BLOCK + t) * 4u + ((b >> 1) & 3u)) + (b & 1u));
        }
        if (t == 0) s_nfix[which] = fix_total;
        __syncthreads();
    };
    // placement: start of the cell + arrival order.  A key alone in its cell is in its final place.
    // The keys are read again (the tile's range is L2-resident), so that nothing but `meta` had to stay
    // in registers since the counting pass.
    auto placement = [&](const Tile& x, const uint32_t (&meta)[IPT]) {
        KeyT keys[IPT];
        load_keys(x, keys);
#pragma unroll
        for (int j = 0; j < IPT; ++j) {
            const uint32_t idx = t + j * LS_BLOCK;
            if (idx < x.m) {
                const uint32_t c = meta[j] & ((1u << CELL_BITS) - 1u);
                const uint32_t w = s_cell[c >> 1];
                const uint32_t at = (w & 0xFFFFu) + ((c & 1u) ? (w >> 16) : 0u) + (meta[j] >> CELL_BITS);
                s_stage[at] = keys[j];
                if constexpr (PAIRS) s_idx[at] = (uint16_t)idx;
            }
        }
        __syncthreads();
    };
    // the crowded cells: sorted in place, duplicates recorded.  Returns false when a cell is beyond what the
    // block can sort (the tile is flagged for the fallback).  Contains barriers; leaves the total of
    // duplicates in s_ndup.
    auto fixup = [&](const Tile& x, uint32_t n_fix) -> bool {
        const uint32_t m = x.m;
        uint32_t my_dups = 0;
        auto mark_dup = [&](uint32_t pos) {
            atomicOr(&s_dup[pos >> 5], 1u << (pos & 31u));
            ++my_dups;
        };
        // first position and size of a listed cell (the counter words stay intact until the block's pass)
        auto cell_range = [&](uint32_t c, uint32_t& first, uint32_t& cnt) {
            const uint32_t w = s_cell[c >> 1];
            if (c & 1u) {
                first = (w & 0xFFFFu) + (w >> 16);
                cnt = ((c >> 1) + 1u < (uint32_t)CAP ? (s_cell[(c >> 1) + 1u] & 0xFFFFu) : m) - first;
            } else {
                first = w & 0xFFFFu;
                cnt = w >> 16;
            }
        };
        // a thread per cell: two keys as a rule (one compare), else an insertion sort of up to 12
        for (uint32_t i0 = t; i0 < n_fix; i0 += LS_BLOCK) {
            uint32_t first, cnt;
            cell_range(s_fix[i0], first, cnt);
            if (cnt == 2u) {
                const KeyT a = s_stage[first], b = s_stage[first + 1];
                if (b < a) {
                    s_stage[first] = b;
                    s_stage[first + 1] = a;
                    if constexpr (PAIRS) {
                        const uint16_t ia = s_idx[first];
                        s_idx[first] = s_idx[first + 1];
                        s_idx[first + 1] = ia;
                    }
                } else if (a == b) {
                    mark_dup(first + 1);
                }
                continue;
            }
            if (cnt > (uint32_t)LSF_THREAD_MAX) {
                if (cnt > (uint32_t)LS_WARP_RUN_MAX) {  // the block's share
                    const uint32_t b = atomicAdd(&s_big_n, 1u);
                    s_big[b][0] = first;
                    s_big[b][1] = first + cnt;
                } else {
                    s_has_mid = 1;
                }
                continue;
            }
            for (uint32_t i = first + 1; i < first + cnt; ++i) {
                const KeyT key = s_stage[i];
                if (!(key < s_stage[i - 1])) continue;
                uint16_t my_idx = 0;
                if constexpr (PAIRS) my_idx = s_idx[i];
                uint32_t qi = i;
                do {
                    s_stage[qi] = s_stage[qi - 1];
                    if constexpr (PAIRS) s_idx[qi] = s_idx[qi - 1];
                    --qi;
                } while (qi > first && key < s_stage[qi - 1]);
                s_stage[qi] = key;
                if constexpr (PAIRS) s_idx[qi] = my_idx;
            }
            for (uint32_t i = first + 1; i < first + cnt; ++i)
                if (s_stage[i] == s_stage[i - 1]) mark_dup(i);
        }
        __syncthreads();
        if (s_has_mid) {  // (block-uniform) cells of 13..128 keys: one warp each, rank sort with the keys in registers
            for (uint32_t i0 = warp; i0 < n_fix; i0 += LS_BLOCK / 32) {
                uint32_t rlo, rlen;
                cell_range(s_fix[i0], rlo, rlen);
                if (rlen <= (uint32_t)LSF_THREAD_MAX || rlen > (uint32_t)LS_WARP_RUN_MAX) continue;  // (warp-uniform)
                constexpr int Q = LS_WARP_RUN_MAX / 32;
                KeyT kq[Q];
                uint32_t rk[Q];
                uint16_t iq[Q];
#pragma unroll
                for (int q = 0; q < Q; ++q) {
                    const uint32_t o = lane + 32u * q;
                    kq[q] = o < rlen ? s_stage[rlo + o] : KeyT{};
                    if constexpr (PAIRS) iq[q] = o < rlen ? s_idx[rlo + o] : (uint16_t)0;
                    rk[q] = 0;
                }
                for (uint32_t i = 0; i < rlen; ++i) {
                    const KeyT o = s_stage[rlo + i];  // one address for the whole warp: a broadcast
#pragma unroll
                    for (int q = 0; q < Q; ++q) rk[q] += (o < kq[q] || (o == kq[q] && i < lane + 32u * q)) ? 1u : 0u;
                }
                __syncwarp();  // every lane has read the cell
#pragma unroll
                for (int q = 0; q < Q; ++q) {
                    if (lane + 32u * q < rlen) {
                        s_stage[rlo + rk[q]] = kq[q];
                        if constexpr (PAIRS) s_idx[rlo + rk[q]] = iq[q];
                    }
                }
                __syncwarp();
                for (uint32_t o = lane + 1; o < rlen; o += 32)
                    if (s_stage[rlo + o] == s_stage[rlo + o - 1]) mark_dup(rlo + o);
            }
            __syncthreads();
        }
        const uint32_t n_big = s_big_n;
        if (n_big) {
            // bitonic sort of every bigger cell by the whole block, in the (now dead) counter array, padded
            // to a power of two with all-ones keys
            constexpr uint32_t TEMP_CAP = (uint32_t)((CAP + CAP / 4) * sizeof(uint32_t) / (sizeof(KeyT) + (PAIRS ? 2 : 0)));
            constexpr uint32_t TEMP_POW2 = TEMP_CAP >= 4096 ? 4096 : (TEMP_CAP >= 2048 ? 2048 : 1024);
            static_assert(TEMP_POW2 <= TEMP_CAP, "bitonic buffer");
            KeyT* tmp_k = reinterpret_cast<KeyT*>(s_cell);
            uint16_t* tmp_i = reinterpret_cast<uint16_t*>(tmp_k + TEMP_POW2);
            if (t == 0) atomicAdd(&p.irregular[1], (unsigned long long)n_big);
            for (uint32_t b = 0; b < n_big; ++b) {
                const uint32_t blo = s_big[b][0], sz = s_big[b][1] - blo;
                if (sz > TEMP_POW2) {
                    s_bad = 1;  // (every thread takes the same branch)
                    break;
                }
                uint32_t N = 64;
                while (N < sz) N <<= 1;
                for (uint32_t o = t; o < N; o += LS_BLOCK) {
                    tmp_k[o] = o < sz ? s_stage[blo + o] : key_all_ones(KeyT{});
                    if constexpr (PAIRS) tmp_i[o] = o < sz ? s_idx[blo + o] : (uint16_t)0xFFFF;  // padding sorts last
                }
                __syncthreads();
                for (uint32_t kk = 2; kk <= N; kk <<= 1) {
                    for (uint32_t jj = kk >> 1; jj > 0; jj >>= 1) {
                        for (uint32_t o = t; o < N / 2; o += LS_BLOCK) {
                            // o-th compare-exchange of this stage: partner indices i < l = i ^ jj
                            const uint32_t i = ((o & ~(jj - 1)) << 1) | (o & (jj - 1));
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
                for (uint32_t o = t; o < sz; o += LS_BLOCK) {
                    s_stage[blo + o] = tmp_k[o];
                    if constexpr (PAIRS) s_idx[blo + o] = tmp_i[o];
                    if (o && tmp_k[o] == tmp_k[o - 1]) mark_dup(blo + o);
                }
                __syncthreads();
            }
        }
        if (my_dups) atomicAdd(&s_ndup, my_dups);
        __syncthreads();
        return s_bad == 0;
    };

    // ---- the pipeline ----------------------------------------------------------------------------------
    if (t == 0) {
        s_bad = 0;
        s_has_mid = 0;
        s_big_n = 0;
        s_ndup = 0;
    }
    if (t <= NW) s_dup[t] = 0;
    if constexpr (HISTO) {
        static_assert(NW >= HISTO_SMEM_BINS, "shared bins");
        if (t < HISTO_SMEM_BINS) s_epre[t] = 0;  // kept across the CTA's tiles, flushed once at its end
    }
    zero_cells();
    Tile A = fetch_sortable();  // (its barriers also cover the zeroing above)
    if (A.kind == 0) return;
    {
        KeyT keys[IPT];
        uint32_t meta[IPT];
        load_keys(A, keys);
        front(A, keys, meta, 0);
        placement(A, meta);
    }
    for (;;) {
        // A sits in s_stage in cell order; its list has s_nfix[0] entries.  Take the next ticket and get its
        // keys on their way before A's crowded cells are sorted.
        // Tiles without output met on the way are published on the spot, but RESOLVED only after A: a resolve
        // also publishes its group's (and super-group's) sum, and the one of A's group may be A's own job --
        // every CTA has to meet its obligations (publish, resolve) in ascending tile order, or a tile without
        // output in the group after A waits for a group sum that this very CTA has not written yet.
        Tile N = fetch();
        uint32_t n_pend = 0;  // (block-uniform)
        while (N.kind == 2 && n_pend < (uint32_t)LSF_PEND) {
            publish_nothing(N.tile);
            if (needs_resolve(N.tile)) {
                if (t == 0) s_pend[n_pend] = N.tile;
                ++n_pend;
            }
            N = fetch();
        }
        if (N.kind == 1 && t == 0) {  // (TMA prefetch into L2: no registers held while A is being finished)
            const uintptr_t a0 = reinterpret_cast<uintptr_t>(reinterpret_cast<const KeyT*>(p.keys_in) + N.s);
            const uintptr_t a1 = a0 + (uintptr_t)N.m * sizeof(KeyT);
            tma_prefetch_l2(reinterpret_cast<const void*>(a0 & ~(uintptr_t)15), (uint32_t)(((a1 + 15) & ~(uintptr_t)15) - (a0 & ~(uintptr_t)15)));
        }
        if (N.kind == 2) publish_nothing(N.tile);  // (more of them in a row than the list holds)
        const bool ok = fixup(A, s_nfix[0]);
        const uint32_t ndup = s_ndup;
        // A's aggregate: distinct keys (count), singletons (uniq; known here only without duplicates), kept
        // rows (count in range: without duplicates all of them or none)
        if (!ok && t == 0) {
            atomicAdd(p.irregular, 1ull);
            p.flag[A.tile] = 1;
        }
        if constexpr (FUSED) {
            if (!ok) {
                publish_nothing(A.tile);
            } else if (COUNT || ndup == 0) {
                if (t == 0) tile_prefix_publish(p.tile_state, A.tile, RANGE && p.min_count != 1u ? 0u : A.m - ndup);
            }
        }
        // the next tile's front, between A's publish and A's resolve
        uint32_t meta_n[IPT];
        if (N.kind == 1) {
            KeyT keys[IPT];
            load_keys(N, keys);
            zero_cells();
            __syncthreads();
            front(N, keys, meta_n, 1);
        }
        // ---- emission of A ----
        if constexpr (HISTO) {
            // run lengths from the duplicate bitmask: a run head is a position without a mark, a singleton a
            // head whose successor carries none either (one ballot per word), a longer run the head's mark count
            uint32_t* s_h = s_epre;
            const uint32_t m = A.m;
            if (ok && ndup == 0) {
                if (t == 0) atomicAdd(&s_h[1], m);
            } else if (ok) {
                uint32_t singles = 0;
#pragma unroll
                for (int j = 0; j < IPT; ++j) {
                    const uint32_t pos = t + j * LS_BLOCK;
                    const uint32_t w = pos >> 5;
                    const uint64_t window = ((uint64_t)s_dup[w] | ((uint64_t)s_dup[w + 1] << 32)) >> lane;
                    const bool head = pos < m && !(window & 1u);
                    const bool single = head && !(window & 2u);  // (marks stop at m: none beyond the tile)
                    singles += (uint32_t)__popc(__ballot_sync(0xffffffffu, single));
                    if (head && !single) {
                        uint32_t extra = (uint32_t)__ffsll((long long)~(window >> 1)) - 1u;  // marks right after the head
                        if (extra >= 63u - lane) {  // the run leaves the 64-bit window: walk the words (long runs only)
                            uint32_t q = pos + 1u + extra;
                            while (q < m && ((s_dup[q >> 5] >> (q & 31u)) & 1u)) ++q;
                            extra = q - pos - 1u;
                        }
                        histo_add(s_h, p.histo, 1u + extra);
                    }
                }
                if (lane == 0 && singles) atomicAdd(&s_h[1], singles);
            }
        } else if constexpr (!FUSED) {
            if (ok) {
                KeyT* kout = reinterpret_cast<KeyT*>(p.keys_out) + A.s;
#pragma unroll
                for (int j = 0; j < IPT; ++j) {
                    const uint32_t idx = t + j * LS_BLOCK;
                    if (idx < A.m) kout[idx] = s_stage[idx];
                }
                if constexpr (PAIRS) {
                    const ValT* vin = reinterpret_cast<const ValT*>(p.vals_in) + A.s;
                    ValT* vout = reinterpret_cast<ValT*>(p.vals_out) + A.s;
#pragma unroll
                    for (int j = 0; j < IPT; ++j) {
                        const uint32_t idx = t + j * LS_BLOCK;
                        if (idx < A.m) vout[idx] = vin[s_idx[idx]];
                    }
                }
            }
        } else {
            const uint32_t m = A.m;
            KeyT* kout_all = reinterpret_cast<KeyT*>(p.keys_out);
            if (!ok || (RANGE && ndup == 0 && p.min_count != 1u)) {
                resolve_nothing(A.tile);
            } else if (ndup == 0) {
                // every key of the tile is distinct (the rule on non-repetitive sequence): positions ARE
                // ranks, every count is one, every key a singleton -- a plain coalesced copy
                if (t < 32) {
                    const uint64_t base = tile_prefix_resolve_warp(p.tile_state, p.n_tiles, A.tile, m, p.err);
                    if (t == 0) {
                        s_base = base;
                        if (A.tile == p.n_tiles - 1) *p.n_out = *p.n_out_copy = base + m;
                    }
                }
                __syncthreads();
                const uint64_t base = s_base;
#pragma unroll
                for (int j = 0; j < IPT; ++j) {
                    const uint32_t pos = t + j * LS_BLOCK;
                    if (pos < m) {
                        kout_all[base + pos] = s_stage[pos];
                        if constexpr (COUNT || RANGE) p.counts_out[base + pos] = 1u;
                        else reinterpret_cast<ValT*>(p.vals_out)[base + pos] = (reinterpret_cast<const ValT*>(p.vals_in) + A.s)[s_idx[pos]];
                    }
                }
            } else {
                // what is emitted, as a bitmask over the positions: COUNT the run heads (not a duplicate of the
                // key before), UNIQ the singletons (a head whose successor is not its duplicate), RANGE the heads
                // whose run length is in range (every warp classifies its word of each round: one ballot, no
                // atomics); one warp ranks them
                if constexpr (RANGE) {
#pragma unroll
                    for (int j = 0; j < IPT; ++j) {
                        const uint32_t pos = t + j * LS_BLOCK;
                        const uint32_t w = pos >> 5;
                        const uint64_t window = ((uint64_t)s_dup[w] | ((uint64_t)s_dup[w + 1] << 32)) >> lane;
                        const bool head = pos < m && !(window & 1u);
                        uint32_t extra = (uint32_t)__ffsll((long long)~(window >> 1)) - 1u;
                        if (head && extra >= 63u - lane) {  // the run leaves the 64-bit window: walk the words
                            uint32_t q = pos + 1u + extra;
                            while (q < m && ((s_dup[q >> 5] >> (q & 31u)) & 1u)) ++q;
                            extra = q - pos - 1u;
                        }
                        const uint32_t keep = __ballot_sync(0xffffffffu, head && 1u + extra >= p.min_count && 1u + extra <= p.max_count);
                        if (lane == 0) s_emit[w] = keep;
                    }
                    __syncthreads();
                }
                if (warp == 0) {
                    constexpr int PER = NW / 32;
                    uint32_t em[PER], sum = 0;
#pragma unroll
                    for (int i = 0; i < PER; ++i) {
                        const uint32_t w = lane * PER + i;
                        const uint32_t valid = w * 32u >= m ? 0u : (m - w * 32u >= 32u ? 0xffffffffu : ((1u << (m - w * 32u)) - 1u));
                        const uint32_t d0 = s_dup[w];
                        uint32_t x = ~d0 & valid;
                        if constexpr (UNIQ) x &= ~((d0 >> 1) | (s_dup[w + 1] << 31));
                        if constexpr (RANGE) x = s_emit[w];
                        em[i] = x;
                        sum += __popc(x);
                    }
                    const uint32_t incl = warp_incl_scan(sum);
                    uint32_t run = incl - sum;
#pragma unroll
                    for (int i = 0; i < PER; ++i) {
                        s_emit[lane * PER + i] = em[i];
                        s_epre[lane * PER + i] = run;
                        run += __popc(em[i]);
                    }
                    const uint32_t H = __shfl_sync(0xffffffffu, incl, 31);
                    if ((UNIQ || RANGE) && lane == 0) tile_prefix_publish(p.tile_state, A.tile, H);
                    const uint64_t base = tile_prefix_resolve_warp(p.tile_state, p.n_tiles, A.tile, H, p.err);
                    if (lane == 0) {
                        s_base = base;
                        if (A.tile == p.n_tiles - 1) *p.n_out = *p.n_out_copy = base + H;
                    }
                }
                __syncthreads();
                const uint64_t base = s_base;
                KeyT* kout = kout_all + base;
#pragma unroll
                for (int j = 0; j < IPT; ++j) {
                    const uint32_t pos = t + j * LS_BLOCK;
                    const uint32_t w = pos >> 5;  // (one word per warp and round: broadcast loads)
                    const uint32_t em = s_emit[w];
                    if (!((em >> lane) & 1u)) continue;
                    const uint32_t h = s_epre[w] + __popc(em & lanemask_lt());
                    kout[h] = s_stage[pos];
                    if constexpr (COUNT || RANGE) {
                        // run length = 1 + the duplicate marks that follow without a gap
                        const uint64_t window = ((uint64_t)s_dup[w] | ((uint64_t)s_dup[w + 1] << 32)) >> lane >> 1;
                        uint32_t extra = (uint32_t)__ffsll((long long)~window) - 1u;  // marks right after me inside the window
                        if (extra >= 63u - lane) {  // the run leaves the 64-bit window: walk the words (long runs only)
                            uint32_t q = pos + 1u + extra;
                            while (q < m && ((s_dup[q >> 5] >> (q & 31u)) & 1u)) ++q;
                            extra = q - pos - 1u;
                        }
                        p.counts_out[base + h] = 1u + extra;
                    } else {
                        const ValT* vin = reinterpret_cast<const ValT*>(p.vals_in) + A.s;
                        reinterpret_cast<ValT*>(p.vals_out)[base + h] = vin[s_idx[pos]];
                    }
                }
            }
            // the tiles without output taken since A, in ascending order
            if (n_pend != 0 || N.kind == 2) {
                __syncthreads();
                for (uint32_t i = 0; i < n_pend; ++i) resolve_nothing(s_pend[i]);
                if (N.kind == 2) resolve_nothing(N.tile);
            }
        }
        __syncthreads();  // everyone is done with s_stage, the bitmask and the per-tile flags
        if (t <= NW) s_dup[t] = 0;
        if (t == 0) {
            s_bad = 0;
            s_has_mid = 0;
            s_big_n = 0;
            s_ndup = 0;
            s_nfix[0] = s_nfix[1];
        }
        if (N.kind == 2) {  // (dealt with above; nothing of a next tile has been prepared yet)
            zero_cells();
            N = fetch_sortable();
            if (N.kind == 1) {
                KeyT keys[IPT];
                load_keys(N, keys);
                front(N, keys, meta_n, 0);
            }
        }
        if (N.kind == 0) {
            if constexpr (HISTO) histo_flush(s_epre, p.histo);  // (the barrier above covers the last tile's adds)
            return;
        }
        __syncthreads();
        placement(N, meta_n);
        A = N;
    }
}
