// K1+K2: LUT encode + rolling-window key extraction.
//
// Replaces Sequence.yield_kmers (kmermaid/seq.py:284-328), its reverse-complement variant
// (seq.py:245-282) and the second alphabet filter (seq.py:500-509 via batcher.py:559-561).
//
// Narrow stream: the tile front end of extract_tile.cuh (LUT encode once per base, keys by funnel
// shifts out of 64-bit big-endian code words).  Valid keys are compacted in position order
// (block scan + decoupled look-back across tiles), staged in shared memory and written with
// fully coalesced stores.
#include "extract_tile.cuh"

namespace kmg {

constexpr int EX_BLOCK_DEFAULT = 256;  // threads of the position-ordered extraction (MODE 0)

struct ExtractParams {
    const uint8_t* bases;
    uint64_t n_bases;
    uint64_t win_begin, win_end;
    uint64_t first_tile;  // absolute tile index (tile = EX_BLOCK*PPT window starts, buffer-aligned)
    int k;
    const uint8_t* lut;
    const uint8_t* comp16;
    void* keys_out;
    void* vals_out;
    uint64_t pos_offset;
    unsigned long long* counts;  // [0] emitted, [1] wide windows seen
    uint64_t* tile_state;
    uint32_t* ticket;
    uint32_t* err;
    // fused digit histograms (narrow stream): hs[o][x] counts the plain 4-mers x found at window
    // start + hist_off[o]; hs[n_off] is the unshifted 4-mer histogram G (see hist_finalize_kernel)
    unsigned long long* hs;
    int n_off;
    int hist_off[2 * MAX_PASSES];
    // MODE 2 (fused first prefix pass): every key goes straight to the region of its digit
    // (key >> digit_shift) & 255; cursors[256] hold the next free element of every region
    unsigned long long* cursors;
    int digit_shift;
    // range filter (kmg_extract_parts, FILTER instantiations): a key is kept when its part lies in
    // [part_lo, part_hi).  Narrow part = (key >> part_shift) & part_mask (its top log2(n_parts) bits),
    // wide part = wide_parts[top 16 bits of the key] (kmg_wide_part_table).  The wide count-only
    // launch adds every key to part_counts[part] instead.
    int part_shift;
    uint32_t part_mask, part_lo, part_hi;
    const uint8_t* wide_parts;
    unsigned long long* part_counts;
};

__device__ __forceinline__ bool in_parts(uint32_t part, const ExtractParams& p) {
    return part - p.part_lo < p.part_hi - p.part_lo;
}

constexpr int EX_MAX_OFF = 2 * MAX_PASSES;

// 4 consecutive bases starting at base e (0 <= e <= 92) of the 96-base big-endian string X0:X1:X2
__device__ __forceinline__ uint32_t mer4_at(uint64_t X0, uint64_t X1, uint64_t X2, int e) {
    const int w = e >> 5, off = 2 * (e & 31);
    const uint64_t a = w == 0 ? X0 : (w == 1 ? X1 : X2);
    const uint64_t b = w == 0 ? X1 : (w == 1 ? X2 : 0ull);
    const uint64_t v = off == 0 ? a : ((a << off) | (b >> (64 - off)));
    return (uint32_t)(v >> 56);
}
// are the 4 bases starting at base e (0 <= e <= 124) of the 128-base mask string B0:B1 all plain?
__device__ __forceinline__ bool plain4_at(uint64_t B0, uint64_t B1, int e) {
    uint64_t v;
    if (e == 0) v = B0;
    else if (e < 64) v = (B0 << e) | (B1 >> (64 - e));
    else v = B1 << (e - 64);
    return (v >> 60) == 0;
}

// The order-free prefix pass of one tile (extraction MODE 2 and region_partition_kernel): the keys of
// a digit may land in any order inside the digit's region, because the local sort orders everything
// below the prefix.  So a key's place in the tile's run of its digit is what a shared-memory counter
// returns (rank), one thread per digit reserves the tile's run with one global atomic on the region's
// cursor (reserve), the keys are staged in digit order (slot) and leave as runs (write_runs): no tile
// waits for another one and no ranking needs to be stable.
template <int BLOCK>
struct DigitRuns {
    uint32_t* s_cnt;            // [256] keys per digit in this tile (zeroed before the first rank)
    uint32_t* s_off;            // [256] first staging slot of every digit
    unsigned long long* s_gb;   // [256] global slot of staging slot i = s_gb[digit] + i
    uint32_t* s_scan;           // [BLOCK / 32 + 1]

    // digit | rank << 8
    __device__ __forceinline__ uint32_t rank(uint32_t d) const { return d | (atomicAdd(&s_cnt[d], 1u) << 8); }
    // after a __syncthreads() that follows the last rank(); returns the tile's number of keys
    __device__ __forceinline__ uint32_t reserve(unsigned long long* cursors) const {
        const int t = threadIdx.x;
        const uint32_t c = t < 256 ? s_cnt[t] : 0u;
        unsigned long long g = 0;
        if (c) g = atomicAdd(&cursors[t], (unsigned long long)c);
        uint32_t n_tile;
        const uint32_t off = block_excl_scan<BLOCK, uint32_t>(c, s_scan, n_tile);
        if (t < 256) {
            s_off[t] = off;
            s_gb[t] = g - off;
        }
        __syncthreads();
        return n_tile;
    }
    __device__ __forceinline__ uint32_t slot(uint32_t wh) const { return s_off[wh & 255u] + (wh >> 8); }
    // after a __syncthreads() that follows the staging
    template <bool PAY, typename KeyT, typename ValT, typename DigitOf>
    __device__ __forceinline__ void write_runs(const KeyT* s_keys, const ValT* s_vals, uint32_t n_tile, DigitOf digit_of,
                                               KeyT* keys_out, ValT* vals_out) const {
        for (uint32_t i = threadIdx.x; i < n_tile; i += BLOCK) {
            const KeyT key = s_keys[i];
            const unsigned long long at = s_gb[digit_of(key)] + i;
            keys_out[at] = key;
            if constexpr (PAY) vals_out[at] = s_vals[i];
        }
    }
};

// KeyT: uint64_t (k<=32) or u128 (33<=k<=64).  PPT: window starts per thread (8 or 16).
// MODE 0: keys (and payload) of the valid windows in position order (kmg_extract).
// MODE 1: nothing is emitted -- only the 4-mer histograms (HIST) and the window counts: the
//         top-byte histograms of kmg_extract_dest_counts (the fused pipeline has its own pre-pass,
//         prefix16_hist_kernel).
// MODE 2: extraction fused with the FIRST prefix pass of the hybrid sort: that pass may place the
//         keys of one digit in any order (the local sort orders everything below the prefix), so
//         a tile ranks its keys with the return values of shared-memory atomics, reserves its
//         slots in the 256 digit regions with one global atomic per digit and writes digit runs
//         -- no compaction in position order, no tile prefix, no waiting for other tiles, and the
//         keys never make the extra round trip through HBM in extraction order.
// FILTER (MODE 0 only): keep only the keys whose part lies in [p.part_lo, p.part_hi)
// (kmg_extract_parts); the tile counts kept keys instead of valid windows, order is unchanged.
// STRAND (ST_FWD, ST_BOTH, ST_CANON): the strand rule; ST_CANON emits the canonical key of every window
// with its strand bit in the payload (no digit histograms: they describe window offsets).
template <typename KeyT, int PPT, int STRAND, int VAL_BYTES, bool HIST, int MODE, int EX_BLOCK, bool FILTER = false>
__global__ void __launch_bounds__(EX_BLOCK) extract_narrow_kernel(const ExtractParams p) {
    static_assert(MODE != 1 || HIST, "the pre-pass exists for its histograms");
    static_assert(MODE != 2 || !HIST, "the fused pass takes its histograms from the pre-pass");
    static_assert(!FILTER || (MODE == 0 && !HIST), "the range filter is a variant of the position-ordered extraction");
    static_assert(STRAND != ST_CANON || !HIST, "the 4-mer histograms do not describe canonical keys");
    constexpr bool RC = STRAND == ST_BOTH;
    constexpr int TILE = EX_BLOCK * PPT;
    constexpr int WORDS = TILE / 16 + EX_HALO_WORDS;
    constexpr int OUT_PER_WIN = keys_per_window(STRAND);
    using ValT = typename std::conditional<VAL_BYTES == 4, uint32_t, uint64_t>::type;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr uint32_t STAGE = TILE * OUT_PER_WIN;
    constexpr uint32_t STAGE_PAD = STAGE + STAGE / 8 + 8;  // room for pad_idx() of either width
    KeyT* s_keys = reinterpret_cast<KeyT*>(smem_raw);
    ValT* s_vals = reinterpret_cast<ValT*>(smem_raw + sizeof(KeyT) * STAGE_PAD);
    constexpr int KB = sizeof(KeyT);
    constexpr int VB = VAL_BYTES == 0 ? 8 : VAL_BYTES;
    __shared__ uint32_t s_codes[WORDS];
    __shared__ uint16_t s_bad[WORDS];
    __shared__ uint16_t s_inv[WORDS];
    __shared__ uint8_t s_lut[256];
    __shared__ uint32_t s_scan[EX_BLOCK / 32 + 1];
    __shared__ uint32_t s_tile;
    __shared__ uint64_t s_base;
    __shared__ uint32_t s_wide;
    __shared__ uint32_t s_g[HIST ? 256 : 1];                 // 4-mer histogram of the tile's window starts
    uint32_t* s_c = reinterpret_cast<uint32_t*>(smem_raw);  // [n_off][256] corrections for skipped windows;
                                                            // aliases the key staging buffer, used before it
    __shared__ uint32_t s_any_skipped;
    __shared__ uint32_t s_cnt[MODE == 2 ? 256 : 1];            // keys per digit in this tile
    __shared__ uint32_t s_off[MODE == 2 ? 256 : 1];            // first staging slot of every digit
    __shared__ unsigned long long s_gb[MODE == 2 ? 256 : 1];   // global slot of staging slot i = s_gb[digit] + i

    const int t = threadIdx.x;
    if (t == 0) {
        // (only the position-ordered mode waits for earlier tiles: it needs launch-ordered ids)
        s_tile = MODE == 0 ? atomicAdd(p.ticket, 1u) : blockIdx.x;
        s_wide = 0;
        s_any_skipped = 0;
    }
    if (t < 256) {
        if (HIST) s_g[t] = 0;
        if (MODE == 2) s_cnt[t] = 0;
        s_lut[t] = p.lut[t];
    }
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint64_t tile_pos = (p.first_tile + tile) * (uint64_t)TILE;

    encode_tile_words<EX_BLOCK, WORDS>(p.bases, p.n_bases, t, tile_pos, s_lut, s_codes, s_bad, s_inv);
    __syncthreads();

    // ---- K2: rolling windows ---------------------------------------------------------------
    const int k = p.k;
    const int joff = (t * PPT) & 15;
    const auto [X0, X1, X2, B0, B1, I0, I1] = load_tile_words(s_codes, s_bad, s_inv, (t * PPT) >> 4);

    // validity of my PPT windows first: the tile's count is published as early as possible and
    // the prefix over the earlier tiles is resolved only after the keys have been built.  MODE 2 counts
    // no wide windows (the pre-pass does): all-invalid masks let the compiler drop s_inv altogether.
    uint32_t in_range_mask, nwide;
    bool span_clean;
    const uint32_t vf = narrow_window_flags<PPT>(tile_pos + (uint64_t)t * PPT, p.win_begin, p.win_end, k, joff, B0, B1,
                                                 MODE == 2 ? ~0ull : I0, MODE == 2 ? ~0ull : I1, in_range_mask,
                                                 span_clean, nwide);

    // FILTER: bit OUT_PER_WIN*j (+1 for the '-' key) is set when that key of window j is kept
    uint32_t kf = 0;
    if constexpr (FILTER) {
#pragma unroll
        for (int j = 0; j < PPT; ++j) {
            if (!(vf & (1u << j))) continue;
            uint32_t sd;
            const KeyT key = window_key<STRAND, KeyT>(X0, X1, X2, joff + j, k, sd);
            if (in_parts(key_digit(key, p.part_shift, p.part_mask), p)) kf |= 1u << (j * OUT_PER_WIN);
            if constexpr (RC) {
                if (in_parts(key_digit(rc_key(key, k), p.part_shift, p.part_mask), p)) kf |= 1u << (j * 2 + 1);
            }
        }
    }
    // keys per counted item: a valid window yields OUT_PER_WIN keys, a kept key one
    constexpr uint32_t UNIT = FILTER ? 1 : OUT_PER_WIN;
    const uint32_t cnt = FILTER ? __popc(kf) : __popc(vf);
    uint32_t total = 0, excl = 0;
    if constexpr (MODE != 2) excl = block_excl_scan<EX_BLOCK, uint32_t>(cnt, s_scan, total);
    if constexpr (MODE == 0) {
        if (t == 0) tile_prefix_publish(p.tile_state, tile, (uint64_t)total * UNIT);
    }
    if (MODE != 2 && nwide) atomicAdd(&s_wide, nwide);

    if constexpr (HIST) {
        // G: one count per window start whose first 4 bases are plain.  Digit p of a valid
        // window's key IS the 4-mer at window start + (k-4-4p), so every pass' histogram is G
        // over a shifted range minus the contributions of the skipped windows.
#pragma unroll
        for (int j = 0; j < PPT; ++j) {
            const int je = joff + j;
            if (((in_range_mask >> j) & 1u) && (span_clean || plain4_at(B0, B1, je)))
                atomicAdd(&s_g[mer4_at(X0, X1, X2, je)], 1u);
        }
        const uint32_t skipped = in_range_mask & ~vf;
        if (skipped) s_any_skipped = 1;  // the correction table is zeroed lazily: most tiles never touch it
        __syncthreads();
        if (s_any_skipped) {
            for (int i = t; i < p.n_off * 256; i += EX_BLOCK) s_c[i] = 0;
            __syncthreads();
            if (skipped) {
                for (int j = 0; j < PPT; ++j) {
                    if (!((skipped >> j) & 1u)) continue;
                    for (int o = 0; o < p.n_off; ++o) {
                        const int e = joff + j + p.hist_off[o];
                        if (plain4_at(B0, B1, e)) atomicAdd(&s_c[o * 256 + mer4_at(X0, X1, X2, e)], 1u);
                    }
                }
            }
            __syncthreads();
            for (int i = t; i < p.n_off * 256; i += EX_BLOCK) {
                const uint32_t c = s_c[i];
                if (c) atomicAdd(&p.hs[i], 0ull - (unsigned long long)c);
            }
            __syncthreads();  // the staging buffer is about to be reused for the keys
        }
        if (t < 256) {
            const uint32_t c = s_g[t];
            if (c) atomicAdd(&p.hs[p.n_off * 256 + t], (unsigned long long)c);
        }
    }
    if constexpr (MODE == 1) {  // the pre-pass stops here: window counts only
        __syncthreads();
        if (t == 0) {
            if (total) atomicAdd(&p.counts[0], (unsigned long long)total * OUT_PER_WIN);
            if (s_wide) atomicAdd(&p.counts[1], (unsigned long long)s_wide);
        }
        return;
    }

    if constexpr (MODE == 2) {
        // ---- fused first prefix pass: rank inside the tile = what the digit counter returned ----------
        const int dsh = p.digit_shift;
        const DigitRuns<EX_BLOCK> runs{s_cnt, s_off, s_gb, s_scan};
        uint32_t wh[PPT * OUT_PER_WIN];  // digit | rank << 8
#pragma unroll
        for (int j = 0; j < PPT; ++j) {
            if (!(vf & (1u << j))) continue;
            uint32_t sd;
            const KeyT key = window_key<STRAND, KeyT>(X0, X1, X2, joff + j, k, sd);
            wh[j * OUT_PER_WIN] = runs.rank(key_digit(key, dsh, 255u));
            if constexpr (RC) wh[j * 2 + 1] = runs.rank(key_digit(rc_key(key, k), dsh, 255u));
        }
        __syncthreads();
        const uint32_t n_tile = runs.reserve(p.cursors);
#pragma unroll
        for (int j = 0; j < PPT; ++j) {
            if (!(vf & (1u << j))) continue;
            uint32_t sd;
            const KeyT key = window_key<STRAND, KeyT>(X0, X1, X2, joff + j, k, sd);
            const uint64_t pos = tile_pos + (uint64_t)t * PPT + j + p.pos_offset;
            const uint32_t i0 = runs.slot(wh[j * OUT_PER_WIN]);
            s_keys[i0] = key;
            if constexpr (VAL_BYTES != 0) s_vals[i0] = make_val<ValT>(pos, sd);
            if constexpr (RC) {
                const uint32_t i1 = runs.slot(wh[j * 2 + 1]);
                s_keys[i1] = rc_key(key, k);
                if constexpr (VAL_BYTES != 0) s_vals[i1] = make_val<ValT>(pos, 1);
            }
        }
        __syncthreads();
        runs.template write_runs<VAL_BYTES != 0>(s_keys, s_vals, n_tile, [dsh](const KeyT& key) { return key_digit(key, dsh, 255u); },
                                                 reinterpret_cast<KeyT*>(p.keys_out), reinterpret_cast<ValT*>(p.vals_out));
        return;
    }

    // ---- keys of the valid windows, compacted in position order into the staging buffer -----
    uint32_t r = excl;
#pragma unroll
    for (int j = 0; j < PPT; ++j) {
        if (!(vf & (1u << j))) continue;
        uint32_t sd;
        const KeyT key = window_key<STRAND, KeyT>(X0, X1, X2, joff + j, k, sd);
        const uint64_t pos = tile_pos + (uint64_t)t * PPT + j + p.pos_offset;
        if constexpr (FILTER) {
            if ((kf >> (j * OUT_PER_WIN)) & 1u) {
                s_keys[pad_idx<KB>(r)] = key;
                if constexpr (VAL_BYTES != 0) s_vals[pad_idx<VB>(r)] = make_val<ValT>(pos, sd);
                ++r;
            }
            if constexpr (RC) {
                if ((kf >> (j * 2 + 1)) & 1u) {
                    s_keys[pad_idx<KB>(r)] = rc_key(key, k);
                    if constexpr (VAL_BYTES != 0) s_vals[pad_idx<VB>(r)] = make_val<ValT>(pos, 1);
                    ++r;
                }
            }
            continue;
        }
        s_keys[pad_idx<KB>(r * OUT_PER_WIN)] = key;
        if constexpr (VAL_BYTES != 0) s_vals[pad_idx<VB>(r * OUT_PER_WIN)] = make_val<ValT>(pos, sd);
        if constexpr (RC) {
            s_keys[pad_idx<KB>(r * 2 + 1)] = rc_key(key, k);
            if constexpr (VAL_BYTES != 0) s_vals[pad_idx<VB>(r * 2 + 1)] = make_val<ValT>(pos, 1);
        }
        ++r;
    }
    __syncthreads();
    if (t < 32) {
        const uint64_t e = tile_prefix_resolve_warp(p.tile_state, gridDim.x, tile, (uint64_t)total * UNIT, p.err);
        if (t == 0) s_base = e;
    }
    __syncthreads();
    const uint64_t base = s_base;
    const uint32_t n_out = total * UNIT;
    KeyT* keys_out = reinterpret_cast<KeyT*>(p.keys_out) + base;
    for (uint32_t i = t; i < n_out; i += EX_BLOCK) keys_out[i] = s_keys[pad_idx<KB>(i)];
    if constexpr (VAL_BYTES != 0) {
        ValT* vals_out = reinterpret_cast<ValT*>(p.vals_out) + base;
        for (uint32_t i = t; i < n_out; i += EX_BLOCK) vals_out[i] = s_vals[pad_idx<VB>(i)];
    }
    if (t == 0) {
        if (s_wide) atomicAdd(&p.counts[1], (unsigned long long)s_wide);
        if (tile == gridDim.x - 1) p.counts[0] = base + n_out;
    }
}

// ---- wide stream: windows that pass the alphabet test but contain a non-plain symbol -----
// Rare by construction (N runs, IUPAC codes), so the kernel is simple: 4 consecutive window
// starts per thread, bytes staged in shared memory, 4-bit ASCII-rank codes, 128-bit keys.
constexpr int EXW_BLOCK = 256;
constexpr int EXW_PPT = 4;
constexpr int EXW_TILE = EXW_BLOCK * EXW_PPT;

// LIMBS: 64-bit limbs of a key, 2 (k <= 32, u128) or 4 (k <= 64, u256); limb 0 is the least significant
template <int LIMBS>
struct WideKey {
    uint64_t w[LIMBS];
    __device__ __forceinline__ void push(uint32_t code) {  // key = key << 4 | code
#pragma unroll
        for (int i = LIMBS - 1; i > 0; --i) w[i] = (w[i] << 4) | (w[i - 1] >> 60);
        w[0] = (w[0] << 4) | code;
    }
    __device__ __forceinline__ uint32_t pop() {  // lowest nibble; key >>= 4
        const uint32_t c = (uint32_t)w[0] & 0xFu;
#pragma unroll
        for (int i = 0; i < LIMBS - 1; ++i) w[i] = (w[i] >> 4) | (w[i + 1] << 60);
        w[LIMBS - 1] >>= 4;
        return c;
    }
    __device__ __forceinline__ void set_nibble(int q, uint32_t c) { w[q >> 4] |= (uint64_t)c << (4 * (q & 15)); }
};
template <int LIMBS>
__device__ __forceinline__ bool operator<(const WideKey<LIMBS>& a, const WideKey<LIMBS>& b) {
#pragma unroll
    for (int i = LIMBS - 1; i > 0; --i)
        if (a.w[i] != b.w[i]) return a.w[i] < b.w[i];
    return a.w[0] < b.w[0];
}

// first 4 symbols of a wide key (its top 16 bits; k >= 4)
template <int LIMBS>
__device__ __forceinline__ uint32_t wide_top16(const WideKey<LIMBS>& key, int k) {
    const int s = 4 * k - 16;
    const int w = s >> 6, o = s & 63;
    uint64_t v = 0;
#pragma unroll
    for (int i = 0; i < LIMBS; ++i) {
        if (i == w) v |= key.w[i] >> o;
        if (i == w + 1 && o > 48) v |= key.w[i] << (64 - o);
    }
    return (uint32_t)v & 0xFFFFu;
}

// FILTER 0: every wide key (kmg_extract).  1: only keys whose part lies in [p.part_lo, p.part_hi),
// position order as in 0 (kmg_extract_parts).  2: count-only, keys per part into p.part_counts
// (kmg_extract_wide_part_counts; p.part_hi = n_parts).  STRAND: the strand rule, as in extract_narrow_kernel
// (ST_CANON: every window's key is replaced by the smaller of it and its reverse complement up front).
template <int STRAND, int VAL_BYTES, int LIMBS, int FILTER = 0>
__global__ void __launch_bounds__(EXW_BLOCK) extract_wide_kernel(const ExtractParams p) {
    using ValT = typename std::conditional<VAL_BYTES == 4, uint32_t, uint64_t>::type;
    using KeyT = WideKey<LIMBS>;  // same layout as u128 / u256
    constexpr bool RC = STRAND == ST_BOTH;
    constexpr int OUT_PER_WIN = keys_per_window(STRAND);
    __shared__ uint8_t s_e[EXW_TILE + 64];  // LUT entries of the tile bytes (+ halo: k <= 64)
    __shared__ uint8_t s_lut[256];
    __shared__ uint8_t s_comp[16];
    __shared__ uint32_t s_scan[EXW_BLOCK / 32 + 1];
    __shared__ uint32_t s_tile;
    __shared__ uint64_t s_base;
    __shared__ uint32_t s_pc[FILTER == 2 ? 256 : 1];

    const int t = threadIdx.x;
    if (t == 0) s_tile = FILTER == 2 ? blockIdx.x : atomicAdd(p.ticket, 1u);
    s_lut[t] = p.lut[t];
    if (t < 16) s_comp[t] = p.comp16[t];
    if (FILTER == 2) s_pc[t] = 0;
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint64_t tile_pos = (p.first_tile + tile) * (uint64_t)EXW_TILE;
    for (int i = t; i < EXW_TILE + 64; i += EXW_BLOCK) {
        const uint64_t pos = tile_pos + i;
        s_e[i] = pos < p.n_bases ? s_lut[p.bases[pos]] : (uint8_t)KMG_LUT_INVALID;
    }
    __syncthreads();

    const int k = p.k;
    KeyT keys[EXW_PPT];
    uint32_t vf = 0;
#pragma unroll
    for (int j = 0; j < EXW_PPT; ++j) {
        const int o = t * EXW_PPT + j;
        const uint64_t pos = tile_pos + o;
        uint32_t any_inv = 0, any_nonplain = 0;
        KeyT key;
#pragma unroll
        for (int i = 0; i < LIMBS; ++i) key.w[i] = 0;
        for (int q = 0; q < k; ++q) {
            const uint32_t e = s_e[o + q];
            any_inv |= e & 0x80u;
            any_nonplain |= e & 0x40u;
            key.push((e >> 2) & 0xFu);
        }
        keys[j] = key;
        if (pos >= p.win_begin && pos < p.win_end && !any_inv && any_nonplain) vf |= 1u << j;
    }
    // reverse complement: symbol q of the window (nibble k-1-q of the key) becomes nibble q
    auto make_rc = [&](KeyT f) -> KeyT {
        KeyT rcv;
#pragma unroll
        for (int i = 0; i < LIMBS; ++i) rcv.w[i] = 0;
        for (int q = k - 1; q >= 0; --q) rcv.set_nibble(q, s_comp[f.pop()]);
        return rcv;
    };
    uint32_t sb = 0;  // ST_CANON: bit j set when window j's reverse complement is strictly smaller
    if constexpr (STRAND == ST_CANON) {
#pragma unroll
        for (int j = 0; j < EXW_PPT; ++j) {
            if (!(vf & (1u << j))) continue;
            const KeyT r = make_rc(keys[j]);
            if (r < keys[j]) {
                keys[j] = r;
                sb |= 1u << j;
            }
        }
    }
    if constexpr (FILTER != 0) {
        // bit 2j: key of window j kept, bit 2j+1: its reverse complement kept
        KeyT rcs[RC ? EXW_PPT : 1];
        uint32_t kf = 0;
#pragma unroll
        for (int j = 0; j < EXW_PPT; ++j) {
            if (!(vf & (1u << j))) continue;
            const uint32_t pf = p.wide_parts[wide_top16(keys[j], k)];
            if constexpr (FILTER == 2) atomicAdd(&s_pc[pf], 1u);
            else if (in_parts(pf, p)) kf |= 1u << (2 * j);
            if constexpr (RC) {
                rcs[j] = make_rc(keys[j]);
                const uint32_t pr = p.wide_parts[wide_top16(rcs[j], k)];
                if constexpr (FILTER == 2) atomicAdd(&s_pc[pr], 1u);
                else if (in_parts(pr, p)) kf |= 1u << (2 * j + 1);
            }
        }
        if constexpr (FILTER == 2) {
            __syncthreads();
            if (t < (int)p.part_hi && s_pc[t]) atomicAdd(&p.part_counts[t], (unsigned long long)s_pc[t]);
            return;
        }
        uint32_t total;
        const uint32_t excl = block_excl_scan<EXW_BLOCK, uint32_t>(__popc(kf), s_scan, total);
        if (t < 32) {
            const uint64_t e = tile_prefix_exclusive_warp(p.tile_state, gridDim.x, tile, (uint64_t)total, p.err);
            if (t == 0) s_base = e;
        }
        __syncthreads();
        KeyT* keys_out = reinterpret_cast<KeyT*>(p.keys_out);
        ValT* vals_out = reinterpret_cast<ValT*>(p.vals_out);
        uint64_t r = s_base + excl;
#pragma unroll
        for (int j = 0; j < EXW_PPT; ++j) {
            const uint64_t pos = tile_pos + t * EXW_PPT + j + p.pos_offset;
            if ((kf >> (2 * j)) & 1u) {
                keys_out[r] = keys[j];
                if constexpr (VAL_BYTES != 0) vals_out[r] = make_val<ValT>(pos, (sb >> j) & 1u);
                ++r;
            }
            if constexpr (RC) {
                if ((kf >> (2 * j + 1)) & 1u) {
                    keys_out[r] = rcs[j];
                    if constexpr (VAL_BYTES != 0) vals_out[r] = make_val<ValT>(pos, 1);
                    ++r;
                }
            }
        }
        if (t == 0 && tile == gridDim.x - 1) p.counts[0] = s_base + (uint64_t)total;
        return;
    }
    const uint32_t cnt = __popc(vf);
    uint32_t total;
    const uint32_t excl = block_excl_scan<EXW_BLOCK, uint32_t>(cnt, s_scan, total);
    if (t < 32) {
        const uint64_t e = tile_prefix_exclusive_warp(p.tile_state, gridDim.x, tile, (uint64_t)total * OUT_PER_WIN, p.err);
        if (t == 0) s_base = e;
    }
    __syncthreads();
    const uint64_t base = s_base;
    KeyT* keys_out = reinterpret_cast<KeyT*>(p.keys_out);
    ValT* vals_out = reinterpret_cast<ValT*>(p.vals_out);
    uint64_t r = base + (uint64_t)excl * OUT_PER_WIN;
#pragma unroll
    for (int j = 0; j < EXW_PPT; ++j) {
        if (!(vf & (1u << j))) continue;
        const uint64_t pos = tile_pos + t * EXW_PPT + j + p.pos_offset;
        keys_out[r] = keys[j];
        if constexpr (VAL_BYTES != 0) vals_out[r] = make_val<ValT>(pos, (sb >> j) & 1u);
        ++r;
        if constexpr (RC) {
            keys_out[r] = make_rc(keys[j]);
            if constexpr (VAL_BYTES != 0) vals_out[r] = make_val<ValT>(pos, 1);
            ++r;
        }
    }
    if (t == 0 && tile == gridDim.x - 1) p.counts[0] = base + (uint64_t)total * OUT_PER_WIN;
}

template <typename KeyT, int PPT, int STRAND, int VB, bool HIST, int MODE = 0, int BLOCK = EX_BLOCK_DEFAULT, bool FILTER = false>
static int launch_narrow(const ExtractParams& p, uint32_t n_tiles, cudaStream_t st) {
    constexpr int TILE = BLOCK * PPT;
    constexpr uint32_t STAGE = TILE * keys_per_window(STRAND);
    constexpr uint32_t STAGE_PAD = STAGE + STAGE / 8 + 8;
    // (the pre-pass stages no keys: its dynamic shared memory only holds the correction tables)
    const size_t smem = MODE == 1 ? (size_t)8 * 256 * sizeof(uint32_t)
                                  : (sizeof(KeyT) + (VB == 4 ? 4 : (VB == 8 ? 8 : 0))) * (size_t)STAGE_PAD;
    auto kern = extract_narrow_kernel<KeyT, PPT, STRAND, VB, HIST, MODE, BLOCK, FILTER>;
    KMG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<n_tiles, BLOCK, smem, st>>>(p);
    KMG_LAUNCH_CHECK();
    return KMG_OK;
}

template <typename KeyT, int PPT, bool HIST, bool FILTER = false>
static int dispatch_narrow2(const ExtractParams& p, uint32_t n_tiles, int rc, int vb, cudaStream_t st) {
    constexpr int B = EX_BLOCK_DEFAULT;
    if constexpr (!HIST) {  // (extract_impl rejects canonical keys with histograms)
        if (rc == ST_CANON) {
            if (vb == 0) return launch_narrow<KeyT, PPT, ST_CANON, 0, HIST, 0, B, FILTER>(p, n_tiles, st);
            if (vb == 4) return launch_narrow<KeyT, PPT, ST_CANON, 4, HIST, 0, B, FILTER>(p, n_tiles, st);
            return launch_narrow<KeyT, PPT, ST_CANON, 8, HIST, 0, B, FILTER>(p, n_tiles, st);
        }
    }
    if (rc) {
        if (vb == 0) return launch_narrow<KeyT, PPT, ST_BOTH, 0, HIST, 0, B, FILTER>(p, n_tiles, st);
        if (vb == 4) return launch_narrow<KeyT, PPT, ST_BOTH, 4, HIST, 0, B, FILTER>(p, n_tiles, st);
        return launch_narrow<KeyT, PPT, ST_BOTH, 8, HIST, 0, B, FILTER>(p, n_tiles, st);
    }
    if (vb == 0) return launch_narrow<KeyT, PPT, ST_FWD, 0, HIST, 0, B, FILTER>(p, n_tiles, st);
    if (vb == 4) return launch_narrow<KeyT, PPT, ST_FWD, 4, HIST, 0, B, FILTER>(p, n_tiles, st);
    return launch_narrow<KeyT, PPT, ST_FWD, 8, HIST, 0, B, FILTER>(p, n_tiles, st);
}
template <typename KeyT, int PPT>
static int dispatch_narrow(const ExtractParams& p, uint32_t n_tiles, int rc, int vb, bool hist, cudaStream_t st) {
    return hist ? dispatch_narrow2<KeyT, PPT, true>(p, n_tiles, rc, vb, st)
                : dispatch_narrow2<KeyT, PPT, false>(p, n_tiles, rc, vb, st);
}

// fused first prefix pass (MODE 2).  Key-only forward or canonical extraction stages 8192 keys per tile
// in 512 threads (digit runs of ~32 keys = 256 bytes); with payload or reverse complements 256 threads
// keep the staging buffer at 64 KB.
template <typename KeyT, int PPT>
static int dispatch_scatter_digit(const ExtractParams& p, uint64_t n_win_tiles_256, int rc, int vb, cudaStream_t st) {
    const uint32_t t256 = (uint32_t)n_win_tiles_256;
    if (rc == ST_CANON) {
        if (vb == 4) return launch_narrow<KeyT, PPT, ST_CANON, 4, false, 2, 256>(p, t256, st);
        if (vb == 8) return launch_narrow<KeyT, PPT, ST_CANON, 8, false, 2, 256>(p, t256, st);
        return KMG_ERR_ARG;  // (key-only canonical: 512 threads, see extract_digit_scatter)
    }
    if (rc) {
        if (vb == 0) return launch_narrow<KeyT, PPT, ST_BOTH, 0, false, 2, 256>(p, t256, st);
        if (vb == 4) return launch_narrow<KeyT, PPT, ST_BOTH, 4, false, 2, 256>(p, t256, st);
        return launch_narrow<KeyT, PPT, ST_BOTH, 8, false, 2, 256>(p, t256, st);
    }
    if (vb == 4) return launch_narrow<KeyT, PPT, ST_FWD, 4, false, 2, 256>(p, t256, st);
    if (vb == 8) return launch_narrow<KeyT, PPT, ST_FWD, 8, false, 2, 256>(p, t256, st);
    return KMG_ERR_ARG;  // (key-only forward: 512 threads, see extract_digit_scatter)
}

// ---- fused digit histograms: edges and final assembly -----------------------------------------------
__device__ __forceinline__ uint32_t rc4(uint32_t x) {  // reverse complement of a packed 4-mer
    x = ~x & 0xFFu;
    return ((x & 3u) << 6) | ((x & 0xCu) << 2) | ((x >> 2) & 0xCu) | (x >> 6);
}

// hs[o] so far = G over [win_begin, win_end) minus the skipped windows' 4-mers at offset o.  The
// histogram over the SHIFTED range [win_begin+o, win_end+o) differs from G by the two edges.
__global__ void hist_edges_kernel(const ExtractParams p) {
    __shared__ uint8_t s_lut[256];
    s_lut[threadIdx.x] = p.lut[threadIdx.x];
    __syncthreads();
    for (int o = 0; o < p.n_off; ++o) {
        const int off = p.hist_off[o];
        for (int j = threadIdx.x; j < 2 * off; j += blockDim.x) {
            const bool tail = j >= off;  // + 4-mers at [win_end, win_end+off), - those at [win_begin, win_begin+off)
            const uint64_t q = (tail ? p.win_end : p.win_begin) + (uint64_t)(tail ? j - off : j);
            if (q + 4 > p.n_bases) continue;
            uint32_t x = 0;
            bool plain = true;
            for (int b = 0; b < 4; ++b) {
                const uint32_t e = s_lut[p.bases[q + b]];
                plain = plain && !(e & 0xC0u);
                x = (x << 2) | (e & 3u);
            }
            if (plain) atomicAdd(&p.hs[o * 256 + x], tail ? 1ull : 0ull - 1ull);
        }
    }
}

// digit histograms of the sort plan for 2k key bits from the per-offset 4-mer histograms
//   forward key, full digit p : 4-mer at window offset k-4-4p;   top digit (b bits): first b/2 bases
//   rc key,      full digit p : rc4 of the 4-mer at offset 4p;    top digit: rc of the last b/2 bases
// Rows 13..15 (u64 keys, k >= 12): histograms of the three TOP key bytes, i.e. the 4-mers at window
// offsets 8, 4, 0 (rc: rc4 of those at k-12, k-8, k-4), for the prefix passes of the hybrid sort;
// top_idx = index of the first of those extra offsets in hs (fwd 4, fwd 8, [rc k-8, rc k-12]) or -1.
__global__ void hist_finalize_kernel(const unsigned long long* __restrict__ hs, int n_off, int k, int rc, int top_idx,
                                     unsigned long long* __restrict__ hist_out) {
    const int P = (2 * k + 7) / 8;
    const int b = 2 * k - 8 * (P - 1);  // bits of the top digit: 2, 4, 6 or 8
    const unsigned long long* G = hs + (size_t)n_off * 256;
    const int x = threadIdx.x;  // 256 threads
    for (int pss = 0; pss < P; ++pss) hist_out[pss * 256 + x] = 0;
    __syncthreads();
    // offsets were laid out by the host as: [0 .. P-2] forward full digits, [P-1] forward top (offset 0),
    // then, if rc: [P .. 2P-2] rc full digits (offset 4p), [2P-1] rc top (offset k-4)
    for (int pss = 0; pss < P - 1; ++pss) {
        unsigned long long v = G[x] + hs[(size_t)pss * 256 + x];
        if (rc) v += G[rc4(x)] + hs[(size_t)(P + pss) * 256 + rc4(x)];
        hist_out[pss * 256 + x] = v;
    }
    // top digit: marginalise
    {
        const unsigned long long v = G[x] + hs[(size_t)(P - 1) * 256 + x];
        atomicAdd(&hist_out[(P - 1) * 256 + (x >> (8 - b))], v);
        if (rc) {
            const unsigned long long w = G[x] + hs[(size_t)(2 * P - 1) * 256 + x];
            // last b/2 bases of the window = low b bits of x; their reverse complement is the rc key's top digit
            const uint32_t low = x & ((1u << b) - 1u);
            const uint32_t r = rc4(low << (8 - b)) & ((1u << b) - 1u);
            atomicAdd(&hist_out[(P - 1) * 256 + r], w);
        }
    }
    if (top_idx >= 0) {
        // byte 15: offset 0 (hs row P-1) / rc k-4 (row 2P-1); bytes 14, 13: the extra offsets
        for (int j = 0; j < 3; ++j) {
            const int fi = j == 0 ? P - 1 : top_idx + (j - 1);
            unsigned long long v = G[x] + hs[(size_t)fi * 256 + x];
            if (rc) {
                const int ri = j == 0 ? 2 * P - 1 : top_idx + 2 + (j - 1);
                v += G[rc4(x)] + hs[(size_t)ri * 256 + rc4(x)];
            }
            hist_out[(15 - j) * 256 + x] = v;
        }
    }
}

// Top-byte histograms of kmg_extract_dest_counts: histograms of the three TOP key bytes only (rows 0..2 = bits
// [2k-24,2k-16), [2k-16,2k-8), [2k-8,2k)), i.e. of the 4-mers at window offsets 8, 4, 0 (rc keys:
// rc4 of those at k-12, k-8, k-4) -- valid for 8- and 16-byte keys alike.  hs rows as laid out by
// extract_top_hist: [0..2] forward offsets 8, 4, 0, then (rc) [3..5] offsets k-12, k-8, k-4.
// plan[0] = number of keys, plan[1] = largest top-byte count (how skewed the keys are).
__global__ void hist_top_finalize_kernel(const unsigned long long* __restrict__ hs, int n_off, int rc,
                                         unsigned long long* __restrict__ top, unsigned long long* __restrict__ plan) {
    __shared__ unsigned long long s_sum[8], s_max[8];
    const unsigned long long* G = hs + (size_t)n_off * 256;
    const int x = threadIdx.x;  // 256 threads
    unsigned long long v_top = 0;
    for (int j = 0; j < 3; ++j) {
        unsigned long long v = G[x] + hs[(size_t)j * 256 + x];
        if (rc) v += G[rc4(x)] + hs[(size_t)(3 + j) * 256 + rc4(x)];
        top[j * 256 + x] = v;
        v_top = v;
    }
    unsigned long long sum = v_top, mx = v_top;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sum += __shfl_xor_sync(0xffffffffu, sum, o);
        mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if ((x & 31) == 0) {
        s_sum[x >> 5] = sum;
        s_max[x >> 5] = mx;
    }
    __syncthreads();
    if (x == 0) {
        sum = 0;
        mx = 0;
        for (int i = 0; i < 8; ++i) {
            sum += s_sum[i];
            mx = max(mx, s_max[i]);
        }
        plan[0] = sum;
        plan[1] = mx;
    }
}

// ---- pre-pass of the fused pipeline: histogram of the top 16 key bits ------------------------------------
// The top 16 bits of a forward key are the 8-mer at window offset 0, those of a reverse-complement key
// the rc of the 8-mer at offset k-8.  Counting them over the exact valid windows gives the start of every
// 16-bit prefix bucket before the first key is built, which is what lets the fused pass scatter by the
// TOP byte and a second pass (region_partition_kernel) split every top-byte region by byte 2 with
// order-free atomics -- no stable pass, no look-back.
// A persistent grid of one CTA per SM keeps all 65536 counters in 128 KB of shared memory as 16-bit
// halves of 32-bit words; a counter that reaches 2^15 hands 2^15 to a global spill row, so a half never
// carries into its neighbour (poly-A and microsatellites stay exact).  Each CTA then writes its row of
// packed counts; prefix16_reduce_kernel sums the rows.
constexpr int P16_BLOCK = 1024;
constexpr int P16_PPT = 16;  // window starts per thread: one 16-base word, so every window starts in word t
constexpr uint64_t P16_TILE = (uint64_t)P16_BLOCK * P16_PPT;
constexpr int P16_MAX_CTAS = 192;
constexpr uint32_t P16_WORDS = 1u << 15;  // 32-bit words of one row (two counters each)
constexpr uint32_t P16_SPILL = 1u << 15;

struct Prefix16Params {
    const uint8_t* bases;
    uint64_t n_bases;
    uint64_t win_begin, win_end;
    uint64_t first_tile;
    uint32_t n_tiles;
    int k;
    const uint8_t* lut;
    uint32_t* rows;               // [gridDim.x][P16_WORDS] packed counts of every CTA
    unsigned long long* spill;    // [65536] 2^15 for every time a CTA's counter reached 2^15
    unsigned long long* byte3;    // [256] histogram of key bits [2k-24, 2k-16) (the 24-bit prefix)
    unsigned long long* counts;   // [0] valid narrow windows, [1] wide-stream windows
};

// 8 consecutive bases starting at base e (0 <= e <= 88) of the 96-base big-endian string X0:X1:X2
__device__ __forceinline__ uint32_t mer8_at(uint64_t X0, uint64_t X1, uint64_t X2, int e) {
    const int w = e >> 5, off = 2 * (e & 31);
    const uint64_t a = w == 0 ? X0 : (w == 1 ? X1 : X2);
    const uint64_t b = w == 0 ? X1 : (w == 1 ? X2 : 0ull);
    const uint64_t v = off == 0 ? a : ((a << off) | (b >> (64 - off)));
    return (uint32_t)(v >> 48);
}
__device__ __forceinline__ uint32_t rc8(uint32_t x) { return (rc4(x & 0xFFu) << 8) | rc4(x >> 8); }

__device__ __forceinline__ void count16(uint32_t* s_h, unsigned long long* spill, uint32_t b) {
    const uint32_t sh = (b & 1u) << 4;
    const uint32_t old = atomicAdd(&s_h[b >> 1], 1u << sh);
    if (((old >> sh) & 0xFFFFu) == P16_SPILL - 1u) {  // this add took the counter to 2^15: exactly one thread sees it
        atomicSub(&s_h[b >> 1], P16_SPILL << sh);
        atomicAdd(&spill[b], (unsigned long long)P16_SPILL);
    }
}

// STRAND: the strand rule.  ST_CANON needs no key either: a prefix is monotone in the key, so the top bits of
// the smaller key are the smaller of the two keys' top bits -- one count16 per window, as forward-only.
template <int STRAND>
__global__ void __launch_bounds__(P16_BLOCK, 1) prefix16_hist_kernel(const Prefix16Params p) {
    constexpr bool RC = STRAND == ST_BOTH;
    constexpr int WORDS = (int)(P16_TILE / 16) + EX_HALO_WORDS;
    extern __shared__ __align__(16) uint32_t s_h[];  // [P16_WORDS]: counter b is half (b & 1) of word b >> 1
    __shared__ uint32_t s_codes[WORDS];
    __shared__ uint16_t s_bad[WORDS];
    __shared__ uint16_t s_inv[WORDS];
    __shared__ uint8_t s_lut[256];
    __shared__ uint32_t s_b3[256];
    __shared__ unsigned long long s_n[2];
    const int t = threadIdx.x;
    for (uint32_t i = t; i < P16_WORDS / 4; i += P16_BLOCK) reinterpret_cast<uint4*>(s_h)[i] = make_uint4(0, 0, 0, 0);
    if (t < 256) {
        s_lut[t] = p.lut[t];
        s_b3[t] = 0;
    }
    if (t < 2) s_n[t] = 0;
    const int k = p.k;
    uint32_t n_valid = 0, n_wide = 0;
    for (uint32_t tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
        __syncthreads();  // (the previous tile's words are consumed; first round: the tables are zeroed)
        const uint64_t tile_pos = (p.first_tile + tile) * P16_TILE;
        encode_tile_words<P16_BLOCK, WORDS>(p.bases, p.n_bases, t, tile_pos, s_lut, s_codes, s_bad, s_inv);
        __syncthreads();
        const auto [X0, X1, X2, B0, B1, I0, I1] = load_tile_words(s_codes, s_bad, s_inv, t);
        uint32_t in_range_mask, nwide;
        bool span_clean;
        const uint32_t vf = narrow_window_flags<P16_PPT>(tile_pos + (uint64_t)t * P16_PPT, p.win_begin, p.win_end, k, 0, B0, B1,
                                                         I0, I1, in_range_mask, span_clean, nwide);
        n_valid += __popc(vf);
        n_wide += nwide;
#pragma unroll
        for (int j = 0; j < P16_PPT; ++j) {
            if (!(vf & (1u << j))) continue;
            if constexpr (STRAND == ST_CANON) {
                // 16-bit prefixes of the key (8-mer at 0) and of its rc (rc of the 8-mer at k-8); byte 3 = the
                // low byte of the smaller 24-bit prefix (fwd: + 4-mer at 8, rc: + rc of the 4-mer at k-12)
                const uint32_t f8 = mer8_at(X0, X1, X2, j), r8 = rc8(mer8_at(X0, X1, X2, j + k - 8));
                count16(s_h, p.spill, min(f8, r8));
                const uint32_t f12 = (f8 << 8) | mer4_at(X0, X1, X2, j + 8);
                const uint32_t r12 = (r8 << 8) | rc4(mer4_at(X0, X1, X2, j + k - 12));
                atomicAdd(&s_b3[min(f12, r12) & 0xFFu], 1u);
                continue;
            }
            count16(s_h, p.spill, mer8_at(X0, X1, X2, j));
            atomicAdd(&s_b3[mer4_at(X0, X1, X2, j + 8)], 1u);
            if constexpr (RC) {
                count16(s_h, p.spill, rc8(mer8_at(X0, X1, X2, j + k - 8)));
                atomicAdd(&s_b3[rc4(mer4_at(X0, X1, X2, j + k - 12))], 1u);
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        n_valid += __shfl_xor_sync(0xffffffffu, n_valid, o);
        n_wide += __shfl_xor_sync(0xffffffffu, n_wide, o);
    }
    if ((t & 31) == 0) {
        if (n_valid) atomicAdd(&s_n[0], (unsigned long long)n_valid);
        if (n_wide) atomicAdd(&s_n[1], (unsigned long long)n_wide);
    }
    __syncthreads();
    uint4* row = reinterpret_cast<uint4*>(p.rows + (size_t)blockIdx.x * P16_WORDS);
    for (uint32_t i = t; i < P16_WORDS / 4; i += P16_BLOCK) row[i] = reinterpret_cast<const uint4*>(s_h)[i];
    if (t < 256 && s_b3[t]) atomicAdd(&p.byte3[t], (unsigned long long)s_b3[t]);
    if (t < 2 && s_n[t]) atomicAdd(&p.counts[t], s_n[t]);
}

// Block r sums bucket r * 256 + t over the CTA rows: the top-byte row (top[2][r] = region total), the
// byte-2 marginal (top[1]) and the bucket starts INSIDE region r.
__global__ void __launch_bounds__(256) prefix16_reduce_kernel(const uint32_t* __restrict__ rows, int n_rows,
                                                              const unsigned long long* __restrict__ spill,
                                                              unsigned long long* __restrict__ top,
                                                              unsigned long long* __restrict__ starts) {
    __shared__ unsigned long long s_scan[256 / 32 + 1];
    const uint32_t r = blockIdx.x, t = threadIdx.x, b = r * 256 + t;
    const uint32_t* w = rows + (b >> 1);
    const int sh = (int)(b & 1u) << 4;
    uint32_t acc = 0;  // (at most P16_MAX_CTAS * (2^15 - 1))
#pragma unroll 8
    for (int c = 0; c < n_rows; ++c) acc += (w[(size_t)c * P16_WORDS] >> sh) & 0xFFFFu;
    const unsigned long long v = spill[b] + acc;
    unsigned long long tot;
    const unsigned long long ex = block_excl_scan<256, unsigned long long>(v, s_scan, tot);
    starts[b] = ex;
    if (t == 0) top[2 * 256 + r] = tot;
    if (v) atomicAdd(&top[256 + t], v);
}

// Makes the bucket starts absolute (starts[65536] = number of keys) and copies them into the cursors of
// region_partition_kernel; region_starts = exclusive scan of the top-byte row (the cursors of the fused
// top-byte scatter).  plan[0] = number of keys, plan[1] = largest top-byte count.
// tiles: the region partition's tiles of tile_keys keys, region by region (region r owns ceil(count_r /
// tile_keys) of them), then empty entries up to ceil(keys / tile_keys) + 256, the partition's grid.
__global__ void __launch_bounds__(256) prefix16_starts_kernel(const unsigned long long* __restrict__ top,
                                                              unsigned long long* __restrict__ plan,
                                                              unsigned long long* __restrict__ region_starts,
                                                              unsigned long long* __restrict__ starts,
                                                              unsigned long long* __restrict__ cursors,
                                                              RpTile* __restrict__ tiles, uint32_t tile_keys) {
    __shared__ unsigned long long s_scan[256 / 32 + 1], s_max[8], s_base;
    __shared__ uint32_t s_scan32[256 / 32 + 1], s_t0;
    const uint32_t r = blockIdx.x, t = threadIdx.x, b = r * 256 + t;
    const unsigned long long c = top[2 * 256 + t];
    unsigned long long total;
    const unsigned long long ex = block_excl_scan<256, unsigned long long>(c, s_scan, total);
    const uint32_t nt = (uint32_t)((c + tile_keys - 1) / tile_keys);
    uint32_t tiles_all;
    const uint32_t t0 = block_excl_scan<256, uint32_t>(nt, s_scan32, tiles_all);
    if (t == r) {
        s_base = ex;
        s_t0 = t0;
    }
    __syncthreads();
    const unsigned long long s = starts[b] + s_base;
    starts[b] = s;
    cursors[b] = s;
    if (t == 0) region_starts[r] = s_base;
    const unsigned long long c_r = top[2 * 256 + r];
    for (uint32_t i = t; (unsigned long long)i * tile_keys < c_r; i += 256) {
        const unsigned long long first = (unsigned long long)i * tile_keys;
        tiles[s_t0 + i] = RpTile{s_base + first, (uint32_t)min((unsigned long long)tile_keys, c_r - first), r};
    }
    if (r == 255) {
        const unsigned long long grid = (total + tile_keys - 1) / tile_keys + 256;
        for (unsigned long long i = tiles_all + t; i < grid; i += 256) tiles[i] = RpTile{0, 0, 0};
    }
    if (r == 0) {
        unsigned long long mx = c;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        if ((t & 31) == 0) s_max[t >> 5] = mx;
        __syncthreads();
        if (t == 0) {
            for (int i = 1; i < 8; ++i) mx = max(mx, s_max[i]);
            plan[0] = total;
            plan[1] = mx;
            starts[65536] = total;
        }
    }
}

// ---- second prefix pass of the pb = 16 pipeline: split every top-byte region by byte 2 --------------------
// The keys arrive grouped by their top byte (region r = [R_r, R_r + count_r)).  Every 16-bit bucket's start
// is known from the pre-pass, so each region is split on its own with the order-free DigitRuns pass:
// tiles never straddle a region (region r owns ceil(count_r / TILE) consecutive tiles, listed by
// prefix16_starts_kernel), a tile ranks its keys with shared-memory atomics, reserves its runs with one
// global atomic per digit on the bucket cursors and writes them through shared-memory staging.
// A CTA first pulls the tile of the CTA that will start about one wave later into L2, so the DRAM reads
// keep streaming while the resident CTAs rank, reserve and write.
constexpr int RP_BLOCK = 512;
// keys per thread: 48-80 KB of staging and at most 64 registers (two CTAs per SM) without spills
template <typename KeyT, int VB>
constexpr int rp_ipt() { return sizeof(KeyT) == 8 ? (VB == 0 ? 12 : 8) : (VB == 8 ? 6 : 8); }

uint32_t region_tile_keys(int key_bytes, int val_bytes) {
    if (key_bytes == 8) return RP_BLOCK * (val_bytes ? rp_ipt<uint64_t, 4>() : rp_ipt<uint64_t, 0>());
    return RP_BLOCK * (val_bytes == 8 ? rp_ipt<u128, 8>() : rp_ipt<u128, 0>());
}

struct RegionPartParams {
    const void* keys_in;
    void* keys_out;
    const void* vals_in;
    void* vals_out;
    const RpTile* tiles;          // one entry per CTA (prefix16_starts_kernel)
    unsigned long long* cursors;  // [65536] next free slot of every 16-bit bucket
    int digit_shift;              // of byte 2
    uint32_t ahead;               // the tile pulled into L2: this CTA's + ahead (about the CTAs resident at once)
};

// [a, a + bytes) into L2, trimmed to whole 16-byte units inside the range
__device__ __forceinline__ void prefetch_l2_inside(const void* a, size_t bytes) {
    const uintptr_t lo = (reinterpret_cast<uintptr_t>(a) + 15) & ~(uintptr_t)15;
    const uintptr_t hi = (reinterpret_cast<uintptr_t>(a) + bytes) & ~(uintptr_t)15;
    if (hi > lo) tma_prefetch_l2(reinterpret_cast<const void*>(lo), (uint32_t)(hi - lo));
}

template <typename KeyT, int VB>
__global__ void __launch_bounds__(RP_BLOCK, 2) region_partition_kernel(const RegionPartParams p) {
    constexpr int IPT = rp_ipt<KeyT, VB>();
    constexpr uint32_t TILE = RP_BLOCK * IPT;
    using ValT = typename std::conditional<VB == 4, uint32_t, uint64_t>::type;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    KeyT* s_keys = reinterpret_cast<KeyT*>(smem_raw);
    ValT* s_vals = reinterpret_cast<ValT*>(smem_raw + sizeof(KeyT) * TILE);
    __shared__ uint32_t s_cnt[256], s_off[256];
    __shared__ unsigned long long s_gb[256];
    __shared__ uint32_t s_scan[RP_BLOCK / 32 + 1];

    const int t = threadIdx.x;
    const RpTile tile = p.tiles[blockIdx.x];
    if (tile.n == 0) return;  // surplus CTA (the grid is sized for the worst split)
    if (t == 0 && blockIdx.x + p.ahead < gridDim.x) {
        const RpTile nx = p.tiles[blockIdx.x + p.ahead];
        prefetch_l2_inside(reinterpret_cast<const KeyT*>(p.keys_in) + nx.first, (size_t)nx.n * sizeof(KeyT));
        if constexpr (VB != 0)
            prefetch_l2_inside(reinterpret_cast<const ValT*>(p.vals_in) + nx.first, (size_t)nx.n * sizeof(ValT));
    }
    const uint32_t r = tile.region;
    const unsigned long long lo = tile.first;
    const uint32_t n_in = tile.n;
    const KeyT* keys_in = reinterpret_cast<const KeyT*>(p.keys_in) + lo;
    const ValT* vals_in = reinterpret_cast<const ValT*>(p.vals_in) + lo;
    const int dsh = p.digit_shift;
    const DigitRuns<RP_BLOCK> runs{s_cnt, s_off, s_gb, s_scan};
    KeyT key[IPT];
    ValT val[VB ? IPT : 1];
    uint32_t wh[IPT];
#pragma unroll
    for (int q = 0; q < IPT; ++q) {
        const uint32_t i = q * RP_BLOCK + t;
        if (i < n_in) {
            key[q] = keys_in[i];
            if constexpr (VB != 0) val[q] = vals_in[i];
        }
    }
    if (t < 256) s_cnt[t] = 0;  // (after the loads: they are on their way while the CTA waits here)
    __syncthreads();
#pragma unroll
    for (int q = 0; q < IPT; ++q)
        if (q * RP_BLOCK + t < n_in) wh[q] = runs.rank(key_digit(key[q], dsh, 255u));
    __syncthreads();
    const uint32_t n_tile = runs.reserve(p.cursors + (size_t)r * 256);
#pragma unroll
    for (int q = 0; q < IPT; ++q) {
        if (q * RP_BLOCK + t < n_in) {
            const uint32_t i = runs.slot(wh[q]);
            s_keys[i] = key[q];
            if constexpr (VB != 0) s_vals[i] = val[q];
        }
    }
    __syncthreads();
    runs.template write_runs<VB != 0>(s_keys, s_vals, n_tile, [dsh](const KeyT& k_) { return key_digit(k_, dsh, 255u); },
                                      reinterpret_cast<KeyT*>(p.keys_out), reinterpret_cast<ValT*>(p.vals_out));
}

template <typename KeyT, int VB>
static int launch_region_partition(const RegionPartParams& p, uint64_t n, cudaStream_t st) {
    constexpr uint64_t TILE = (uint64_t)RP_BLOCK * rp_ipt<KeyT, VB>();
    const uint64_t grid = (n + TILE - 1) / TILE + 256;  // + one partial tile per region at most
    KMG_REQUIRE(grid < (1ull << 31), KMG_ERR_RANGE, "too many tiles");
    const size_t smem = TILE * (sizeof(KeyT) + VB);
    auto kern = region_partition_kernel<KeyT, VB>;
    KMG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    RegionPartParams q = p;
    q.ahead = 2 * (uint32_t)sms;  // (two CTAs per SM)
    kern<<<(uint32_t)grid, RP_BLOCK, smem, st>>>(q);
    KMG_LAUNCH_CHECK();
    return KMG_OK;
}

template <int STRAND, int LIMBS, int FILTER = 0>
static int dispatch_wide(const ExtractParams& p, uint32_t n_tiles, int vb, cudaStream_t st) {
    if (vb == 0) extract_wide_kernel<STRAND, 0, LIMBS, FILTER><<<n_tiles, EXW_BLOCK, 0, st>>>(p);
    else if (vb == 4) extract_wide_kernel<STRAND, 4, LIMBS, FILTER><<<n_tiles, EXW_BLOCK, 0, st>>>(p);
    else extract_wide_kernel<STRAND, 8, LIMBS, FILTER><<<n_tiles, EXW_BLOCK, 0, st>>>(p);
    KMG_LAUNCH_CHECK();
    return KMG_OK;
}
// FILTER 2 stores nothing: the payload width does not matter
template <int FILTER>
static int dispatch_wide_any(const ExtractParams& p, uint32_t n_tiles, int k, int rc, int vb, cudaStream_t st) {
    if (rc == ST_CANON) return k <= 32 ? dispatch_wide<ST_CANON, 2, FILTER>(p, n_tiles, vb, st)
                                       : dispatch_wide<ST_CANON, 4, FILTER>(p, n_tiles, vb, st);
    if (k <= 32) return rc ? dispatch_wide<ST_BOTH, 2, FILTER>(p, n_tiles, vb, st) : dispatch_wide<ST_FWD, 2, FILTER>(p, n_tiles, vb, st);
    return rc ? dispatch_wide<ST_BOTH, 4, FILTER>(p, n_tiles, vb, st) : dispatch_wide<ST_FWD, 4, FILTER>(p, n_tiles, vb, st);
}

static void fill_common(ExtractParams& p, const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end,
                        uint64_t tile, int k, const uint8_t* d_lut256) {
    memset(&p, 0, sizeof(p));
    p.bases = d_bases;
    p.n_bases = n_bases;
    p.win_begin = win_begin;
    p.win_end = win_end;
    p.first_tile = win_begin / tile;
    p.k = k;
    p.lut = d_lut256;
}

size_t top_hist_workspace_bytes() { return sizeof(WsHeader) + (size_t)(6 + 1) * 256 * sizeof(uint64_t); }

// see common.cuh
int extract_top_hist(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k, int rc,
                     const uint8_t* d_lut256, uint64_t* d_counts, unsigned long long* d_top, unsigned long long* d_plan,
                     void* d_ws, size_t ws_bytes, cudaStream_t st) {
    KMG_REQUIRE(k >= 12 && k <= 64, KMG_ERR_ARG, "the top-byte histograms need 12 <= k <= 64");
    KMG_REQUIRE(ws_bytes >= top_hist_workspace_bytes(), KMG_ERR_WS, "top-hist workspace too small");
    KMG_CUDA(cudaMemsetAsync(d_counts, 0, 2 * sizeof(uint64_t), st));
    KMG_CUDA(cudaMemsetAsync(d_ws, 0, top_hist_workspace_bytes(), st));
    constexpr uint64_t TILE = (uint64_t)EX_BLOCK_DEFAULT * 16;
    ExtractParams p;
    fill_common(p, d_bases, n_bases, win_begin, win_end, TILE, k, d_lut256);
    p.counts = reinterpret_cast<unsigned long long*>(d_counts);
    p.hs = reinterpret_cast<unsigned long long*>((char*)d_ws + sizeof(WsHeader));
    p.hist_off[0] = 8;
    p.hist_off[1] = 4;
    p.hist_off[2] = 0;
    p.n_off = 3;
    if (rc) {
        p.hist_off[3] = k - 12;
        p.hist_off[4] = k - 8;
        p.hist_off[5] = k - 4;
        p.n_off = 6;
    }
    if (win_end > win_begin) {
        const uint64_t n_tiles = (win_end + TILE - 1) / TILE - p.first_tile;
        KMG_REQUIRE(n_tiles < (1ull << 31), KMG_ERR_RANGE, "too many tiles");
        // (the histograms do not depend on the key width; one window per lane and 16 per thread
        // span at most 79 bases, which the 96-base code words cover for every k <= 64)
        const int rcode = launch_narrow<uint64_t, 16, ST_FWD, 0, true, 1, EX_BLOCK_DEFAULT>(p, (uint32_t)n_tiles, st);
        if (rcode != KMG_OK) return rcode;
        hist_edges_kernel<<<1, 256, 0, st>>>(p);
        KMG_LAUNCH_CHECK();
    }
    hist_top_finalize_kernel<<<1, 256, 0, st>>>(p.hs, p.n_off, rc, d_top, d_plan);
    KMG_LAUNCH_CHECK();
    return KMG_OK;
}

// Top-byte histogram of the canonical keys (kmg_extract_dest_counts with rc = KMG_CANONICAL).  The 4-mer shift
// trick of extract_top_hist does not describe the smaller of two keys, but the top byte of the smaller key is
// the smaller of the two top bytes: one shared atomic per window on min(4-mer at 0, rc4(4-mer at k-4)).
constexpr int CT_BLOCK = 256;
constexpr int CT_PPT = 16;  // one 16-base word per thread, as in prefix16_hist_kernel

__global__ void __launch_bounds__(CT_BLOCK) canonical_top_kernel(const ExtractParams p) {
    constexpr int TILE = CT_BLOCK * CT_PPT;
    constexpr int WORDS = TILE / 16 + EX_HALO_WORDS;
    __shared__ uint32_t s_codes[WORDS];
    __shared__ uint16_t s_bad[WORDS];
    __shared__ uint16_t s_inv[WORDS];
    __shared__ uint8_t s_lut[256];
    __shared__ uint32_t s_top[256];
    __shared__ uint32_t s_n[2];
    const int t = threadIdx.x;
    s_lut[t] = p.lut[t];
    s_top[t] = 0;
    if (t < 2) s_n[t] = 0;
    __syncthreads();
    const uint64_t tile_pos = (p.first_tile + blockIdx.x) * (uint64_t)TILE;
    encode_tile_words<CT_BLOCK, WORDS>(p.bases, p.n_bases, t, tile_pos, s_lut, s_codes, s_bad, s_inv);
    __syncthreads();
    const int k = p.k;
    const auto [X0, X1, X2, B0, B1, I0, I1] = load_tile_words(s_codes, s_bad, s_inv, t);
    uint32_t in_range_mask, nwide;
    bool span_clean;
    const uint32_t vf = narrow_window_flags<CT_PPT>(tile_pos + (uint64_t)t * CT_PPT, p.win_begin, p.win_end, k, 0, B0, B1,
                                                    I0, I1, in_range_mask, span_clean, nwide);
#pragma unroll
    for (int j = 0; j < CT_PPT; ++j)
        if (vf & (1u << j)) atomicAdd(&s_top[min(mer4_at(X0, X1, X2, j), rc4(mer4_at(X0, X1, X2, j + k - 4)))], 1u);
    uint32_t n_valid = __popc(vf);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        n_valid += __shfl_xor_sync(0xffffffffu, n_valid, o);
        nwide += __shfl_xor_sync(0xffffffffu, nwide, o);
    }
    if ((t & 31) == 0) {
        if (n_valid) atomicAdd(&s_n[0], n_valid);
        if (nwide) atomicAdd(&s_n[1], nwide);
    }
    __syncthreads();
    if (s_top[t]) atomicAdd(&p.hs[t], (unsigned long long)s_top[t]);
    if (t < 2 && s_n[t]) atomicAdd(&p.counts[t], (unsigned long long)s_n[t]);
}

// see common.cuh
int extract_canonical_top(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k,
                          const uint8_t* d_lut256, unsigned long long* d_top_row, unsigned long long* d_counts,
                          cudaStream_t st) {
    KMG_REQUIRE(k >= 12 && k <= 64, KMG_ERR_ARG, "the top-byte histogram needs 12 <= k <= 64");
    KMG_CUDA(cudaMemsetAsync(d_top_row, 0, 256 * sizeof(uint64_t), st));
    KMG_CUDA(cudaMemsetAsync(d_counts, 0, 2 * sizeof(uint64_t), st));
    if (win_end == win_begin) return KMG_OK;
    constexpr uint64_t TILE = (uint64_t)CT_BLOCK * CT_PPT;
    ExtractParams p;
    fill_common(p, d_bases, n_bases, win_begin, win_end, TILE, k, d_lut256);
    p.hs = d_top_row;
    p.counts = d_counts;
    const uint64_t n_tiles = (win_end + TILE - 1) / TILE - p.first_tile;
    KMG_REQUIRE(n_tiles < (1ull << 31), KMG_ERR_RANGE, "too many tiles");
    canonical_top_kernel<<<(uint32_t)n_tiles, CT_BLOCK, 0, st>>>(p);
    KMG_LAUNCH_CHECK();
    return KMG_OK;
}

int extract_digit_scatter(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k, int rc,
                          const uint8_t* d_lut256, void* d_keys_out, int key_bytes, void* d_vals_out, int val_bytes,
                          uint64_t pos_offset, unsigned long long* d_cursors, int digit_shift, cudaStream_t st) {
    if (win_end == win_begin) return KMG_OK;
    const int ppt = key_bytes == 8 ? 16 : 8;
    const bool big = (!rc || rc == ST_CANON) && val_bytes == 0;  // 512-thread tiles
    const uint64_t tile = (uint64_t)(big ? 512 : 256) * ppt;
    ExtractParams p;
    fill_common(p, d_bases, n_bases, win_begin, win_end, tile, k, d_lut256);
    p.keys_out = d_keys_out;
    p.vals_out = d_vals_out;
    p.pos_offset = pos_offset;
    p.cursors = d_cursors;
    p.digit_shift = digit_shift;
    const uint64_t n_tiles = (win_end + tile - 1) / tile - p.first_tile;
    KMG_REQUIRE(n_tiles < (1ull << 31), KMG_ERR_RANGE, "too many tiles");
    if (big && rc == ST_CANON) {
        if (key_bytes == 8) return launch_narrow<uint64_t, 16, ST_CANON, 0, false, 2, 512>(p, (uint32_t)n_tiles, st);
        return launch_narrow<u128, 8, ST_CANON, 0, false, 2, 512>(p, (uint32_t)n_tiles, st);
    }
    if (big) {
        if (key_bytes == 8) return launch_narrow<uint64_t, 16, ST_FWD, 0, false, 2, 512>(p, (uint32_t)n_tiles, st);
        return launch_narrow<u128, 8, ST_FWD, 0, false, 2, 512>(p, (uint32_t)n_tiles, st);
    }
    if (key_bytes == 8) return dispatch_scatter_digit<uint64_t, 16>(p, n_tiles, rc, val_bytes, st);
    return dispatch_scatter_digit<u128, 8>(p, n_tiles, rc, val_bytes, st);
}

size_t prefix16_rows_bytes() { return (size_t)P16_MAX_CTAS * P16_WORDS * sizeof(uint32_t); }

// see common.cuh
int extract_prefix16_hist(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k, int rc,
                          const uint8_t* d_lut256, const Prefix16Out& o, cudaStream_t st) {
    KMG_REQUIRE(k >= 12 && k <= 64, KMG_ERR_ARG, "the prefix histograms need 12 <= k <= 64");
    KMG_CUDA(cudaMemsetAsync(o.zeroed, 0, P16_ZEROED_WORDS * sizeof(uint64_t), st));
    unsigned long long* spill = o.zeroed;
    unsigned long long* top = p16_top(o.zeroed);
    unsigned long long* plan = p16_plan(o.zeroed);
    Prefix16Params p;
    memset(&p, 0, sizeof(p));
    p.bases = d_bases;
    p.n_bases = n_bases;
    p.win_begin = win_begin;
    p.win_end = win_end;
    p.k = k;
    p.lut = d_lut256;
    p.rows = o.rows;
    p.spill = spill;
    p.byte3 = top;
    p.counts = plan + 2;
    int n_rows = 0;
    if (win_end > win_begin) {
        p.first_tile = win_begin / P16_TILE;
        const uint64_t n_tiles = (win_end + P16_TILE - 1) / P16_TILE - p.first_tile;
        KMG_REQUIRE(n_tiles < (1ull << 31), KMG_ERR_RANGE, "too many tiles");
        p.n_tiles = (uint32_t)n_tiles;
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        n_rows = (int)std::min<uint64_t>(n_tiles, (uint64_t)std::min(sms, P16_MAX_CTAS));
        const size_t smem = P16_WORDS * sizeof(uint32_t);
        auto kern = rc == ST_CANON ? prefix16_hist_kernel<ST_CANON> : rc ? prefix16_hist_kernel<ST_BOTH> : prefix16_hist_kernel<ST_FWD>;
        KMG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<n_rows, P16_BLOCK, smem, st>>>(p);
        KMG_LAUNCH_CHECK();
    }
    prefix16_reduce_kernel<<<256, 256, 0, st>>>(o.rows, n_rows, spill, top, o.starts);
    KMG_LAUNCH_CHECK();
    prefix16_starts_kernel<<<256, 256, 0, st>>>(top, plan, o.region_starts, o.starts, o.cursors, o.tiles, o.tile_keys);
    KMG_LAUNCH_CHECK();
    return KMG_OK;
}

int region_partition(const void* d_keys_in, void* d_keys_out, const void* d_vals_in, void* d_vals_out, uint64_t n,
                     int key_bytes, int val_bytes, const RpTile* d_tiles, unsigned long long* d_cursors, int digit_shift,
                     cudaStream_t st) {
    if (n == 0) return KMG_OK;
    RegionPartParams p;
    p.keys_in = d_keys_in;
    p.keys_out = d_keys_out;
    p.vals_in = d_vals_in;
    p.vals_out = d_vals_out;
    p.tiles = d_tiles;
    p.cursors = d_cursors;
    p.digit_shift = digit_shift;
    if (key_bytes == 8) {
        if (val_bytes == 0) return launch_region_partition<uint64_t, 0>(p, n, st);
        if (val_bytes == 4) return launch_region_partition<uint64_t, 4>(p, n, st);
        return launch_region_partition<uint64_t, 8>(p, n, st);
    }
    if (val_bytes == 0) return launch_region_partition<u128, 0>(p, n, st);
    if (val_bytes == 4) return launch_region_partition<u128, 4>(p, n, st);
    return launch_region_partition<u128, 8>(p, n, st);
}

}  // namespace kmg

using namespace kmg;

// smallest tile any extract kernel uses -> upper bound on the number of tiles
static constexpr uint64_t EX_MIN_TILE = 1024;

extern "C" size_t kmg_extract_workspace_bytes(uint64_t n_windows) {
    // header + tile states (+2 tiles for the unaligned head/tail) + per-offset 4-mer histograms
    return sizeof(WsHeader) + align_up(sc_state_words(n_windows / EX_MIN_TILE + 3) * sizeof(uint64_t), 256) +
           (size_t)(EX_MAX_OFF + 1) * 256 * sizeof(uint64_t);
}

// range filter of kmg_extract_parts
struct PartFilter {
    int n_parts, part_lo, part_hi;
    const uint8_t* wide_parts;
};

static int part_bits(int n_parts) {
    int b = 0;
    while ((1 << b) < n_parts) ++b;
    return b;
}

static int extract_impl(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k, int rc,
                        int wide, const uint8_t* d_lut256, const uint8_t* d_comp16, void* d_keys_out, int key_bytes,
                        void* d_vals_out, int val_bytes, uint64_t pos_offset, uint64_t* d_counts, uint64_t* d_hist_out,
                        void* d_ws, size_t ws_bytes, cudaStream_t st, const PartFilter* f) {
    KMG_REQUIRE(k >= 2, KMG_ERR_ARG, "k must be >= 2, got %d", k);  // batcher.py:477-478
    KMG_REQUIRE(k <= 64, KMG_ERR_RANGE, "k=%d: this build supports k <= 64 (no CPU fallback)", k);
    KMG_REQUIRE(win_begin <= win_end, KMG_ERR_ARG, "win_begin > win_end");
    KMG_REQUIRE(val_bytes == 0 || val_bytes == 4 || val_bytes == 8, KMG_ERR_ARG, "val_bytes must be 0, 4 or 8");
    KMG_REQUIRE((val_bytes == 0) == (d_vals_out == nullptr), KMG_ERR_ARG, "d_vals_out / val_bytes mismatch");
    const int want_kb = wide ? (k <= 32 ? 16 : 32) : (k <= 32 ? 8 : 16);
    KMG_REQUIRE(key_bytes == want_kb, KMG_ERR_ARG, "key_bytes must be %d for k=%d wide=%d", want_kb, k, wide);
    KMG_REQUIRE(((uintptr_t)d_bases & 15) == 0, KMG_ERR_ARG, "d_bases must be 16-byte aligned");
    KMG_REQUIRE(((uintptr_t)d_keys_out & (key_bytes - 1)) == 0, KMG_ERR_ARG, "d_keys_out misaligned");
    KMG_REQUIRE(d_lut256 && d_counts && d_ws, KMG_ERR_ARG, "null pointer argument");
    KMG_REQUIRE(!(wide && rc) || d_comp16, KMG_ERR_ARG, "d_comp16 required for wide rc");
    if (val_bytes == 4)
        KMG_REQUIRE(((pos_offset + n_bases) << 1) < (1ull << 32), KMG_ERR_RANGE, "val_bytes=4 needs < 2^31 positions");
    KMG_REQUIRE(ws_bytes >= kmg_extract_workspace_bytes(win_end - win_begin), KMG_ERR_WS, "extract workspace too small");
    KMG_REQUIRE(!d_hist_out || (!wide && k >= 4), KMG_ERR_ARG, "fused digit histograms need the narrow stream and k >= 4");
    KMG_REQUIRE(!d_hist_out || rc != ST_CANON, KMG_ERR_ARG,
                "fused digit histograms describe window offsets, not canonical keys (d_hist_out must be NULL)");

    KMG_CUDA(cudaMemsetAsync(d_counts, 0, 2 * sizeof(uint64_t), st));
    KMG_CUDA(cudaMemsetAsync(d_ws, 0, sizeof(WsHeader), st));
    if (d_hist_out) KMG_CUDA(cudaMemsetAsync(d_hist_out, 0, sizeof(uint64_t) * MAX_PASSES * 256, st));
    if (win_end == win_begin) return KMG_OK;

    const uint64_t tile = wide ? (uint64_t)EXW_TILE : (uint64_t)(EX_BLOCK_DEFAULT * (key_bytes == 8 ? 16 : 8));
    const uint64_t first_tile = win_begin / tile;
    const uint64_t n_tiles = (win_end + tile - 1) / tile - first_tile;
    KMG_REQUIRE(n_tiles < (1ull << 31), KMG_ERR_RANGE, "too many tiles");
    const size_t state_bytes = align_up(sc_state_words(n_tiles) * sizeof(uint64_t), 256);
    const size_t hs_bytes = (size_t)(EX_MAX_OFF + 1) * 256 * sizeof(uint64_t);
    KMG_REQUIRE(ws_bytes >= sizeof(WsHeader) + state_bytes + hs_bytes, KMG_ERR_WS, "extract workspace too small");
    KMG_CUDA(cudaMemsetAsync(d_ws, 0, sizeof(WsHeader) + state_bytes + (d_hist_out ? hs_bytes : 0), st));
    WsHeader* hdr = reinterpret_cast<WsHeader*>(d_ws);

    ExtractParams p;
    fill_common(p, d_bases, n_bases, win_begin, win_end, tile, k, d_lut256);
    p.comp16 = d_comp16;
    p.keys_out = d_keys_out;
    p.vals_out = d_vals_out;
    p.pos_offset = pos_offset;
    p.counts = reinterpret_cast<unsigned long long*>(d_counts);
    p.tile_state = reinterpret_cast<uint64_t*>(hdr + 1);
    p.ticket = &hdr->ticket;
    p.err = &hdr->err;
    p.hs = reinterpret_cast<unsigned long long*>((char*)d_ws + sizeof(WsHeader) + state_bytes);
    if (f) {
        const int b = part_bits(f->n_parts);
        p.part_shift = b ? 2 * k - b : 0;
        p.part_mask = (1u << b) - 1u;
        p.part_lo = (uint32_t)f->part_lo;
        p.part_hi = (uint32_t)f->part_hi;
        p.wide_parts = f->wide_parts;
        if (wide) return dispatch_wide_any<1>(p, (uint32_t)n_tiles, k, rc, val_bytes, st);
        if (key_bytes == 8) return dispatch_narrow2<uint64_t, 16, false, true>(p, (uint32_t)n_tiles, rc, val_bytes, st);
        return dispatch_narrow2<u128, 8, false, true>(p, (uint32_t)n_tiles, rc, val_bytes, st);
    }
    int top_idx = -1;
    if (d_hist_out) {
        const int P = (2 * k + 7) / 8;
        for (int q = 0; q < P - 1; ++q) p.hist_off[q] = k - 4 - 4 * q;
        p.hist_off[P - 1] = 0;
        p.n_off = P;
        if (rc) {
            for (int q = 0; q < P - 1; ++q) p.hist_off[P + q] = 4 * q;
            p.hist_off[2 * P - 1] = k - 4;
            p.n_off = 2 * P;
        }
        if (key_bytes == 8 && k >= 12) {
            top_idx = p.n_off;
            p.hist_off[p.n_off++] = 4;
            p.hist_off[p.n_off++] = 8;
            if (rc) {
                p.hist_off[p.n_off++] = k - 8;
                p.hist_off[p.n_off++] = k - 12;
            }
        }
    }

    if (wide) return dispatch_wide_any<0>(p, (uint32_t)n_tiles, k, rc, val_bytes, st);
    int rcode;
    if (key_bytes == 8) rcode = dispatch_narrow<uint64_t, 16>(p, (uint32_t)n_tiles, rc, val_bytes, d_hist_out != nullptr, st);
    else rcode = dispatch_narrow<u128, 8>(p, (uint32_t)n_tiles, rc, val_bytes, d_hist_out != nullptr, st);
    if (rcode != KMG_OK || !d_hist_out) return rcode;
    hist_edges_kernel<<<1, 256, 0, st>>>(p);
    KMG_LAUNCH_CHECK();
    hist_finalize_kernel<<<1, 256, 0, st>>>(p.hs, p.n_off, k, rc, top_idx, reinterpret_cast<unsigned long long*>(d_hist_out));
    KMG_LAUNCH_CHECK();
    return KMG_OK;
}

extern "C" int kmg_extract(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k,
                           int rc, int wide, const uint8_t* d_lut256, const uint8_t* d_comp16, void* d_keys_out,
                           int key_bytes, void* d_vals_out, int val_bytes, uint64_t pos_offset,
                           uint64_t* d_counts, uint64_t* d_hist_out, void* d_ws, size_t ws_bytes, void* stream) {
    return extract_impl(d_bases, n_bases, win_begin, win_end, k, rc, wide, d_lut256, d_comp16, d_keys_out, key_bytes,
                        d_vals_out, val_bytes, pos_offset, d_counts, d_hist_out, d_ws, ws_bytes, (cudaStream_t)stream, nullptr);
}

static int check_parts(int k, int n_parts, int part_lo, int part_hi, int wide, const uint8_t* d_wide_parts) {
    KMG_REQUIRE(k >= 4, KMG_ERR_ARG, "the range filter needs k >= 4, got %d", k);
    KMG_REQUIRE(n_parts >= 1 && n_parts <= 256 && (n_parts & (n_parts - 1)) == 0, KMG_ERR_ARG,
                "n_parts must be a power of two <= 256, got %d", n_parts);
    KMG_REQUIRE(0 <= part_lo && part_lo <= part_hi && part_hi <= n_parts, KMG_ERR_ARG,
                "part range [%d, %d) outside [0, %d)", part_lo, part_hi, n_parts);
    KMG_REQUIRE(!wide || d_wide_parts, KMG_ERR_ARG, "the wide stream needs d_wide_parts");
    return KMG_OK;
}

extern "C" int kmg_extract_parts(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k,
                                 int rc, int wide, const uint8_t* d_lut256, const uint8_t* d_comp16, int n_parts,
                                 int part_lo, int part_hi, const uint8_t* d_wide_parts, void* d_keys_out, int key_bytes,
                                 void* d_vals_out, int val_bytes, uint64_t pos_offset, uint64_t* d_counts,
                                 uint64_t* d_hist_out, void* d_ws, size_t ws_bytes, void* stream) {
    KMG_REQUIRE(!d_hist_out, KMG_ERR_ARG, "kmg_extract_parts computes no digit histograms (d_hist_out must be NULL)");
    const int rcode = check_parts(k, n_parts, part_lo, part_hi, wide, d_wide_parts);
    if (rcode != KMG_OK) return rcode;
    const PartFilter f{n_parts, part_lo, part_hi, d_wide_parts};
    return extract_impl(d_bases, n_bases, win_begin, win_end, k, rc, wide, d_lut256, d_comp16, d_keys_out, key_bytes,
                        d_vals_out, val_bytes, pos_offset, d_counts, nullptr, d_ws, ws_bytes, (cudaStream_t)stream, &f);
}

extern "C" int kmg_extract_wide_part_counts(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end,
                                            int k, int rc, const uint8_t* d_lut256, const uint8_t* d_comp16, int n_parts,
                                            const uint8_t* d_wide_parts, uint64_t* d_counts, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    const int rcode = check_parts(k, n_parts, 0, n_parts, 1, d_wide_parts);
    if (rcode != KMG_OK) return rcode;
    KMG_REQUIRE(k <= 64, KMG_ERR_RANGE, "k=%d: this build supports k <= 64 (no CPU fallback)", k);
    KMG_REQUIRE(win_begin <= win_end, KMG_ERR_ARG, "win_begin > win_end");
    KMG_REQUIRE(d_bases && d_lut256 && d_counts && (!rc || d_comp16), KMG_ERR_ARG, "null pointer argument");
    KMG_CUDA(cudaMemsetAsync(d_counts, 0, sizeof(uint64_t) * n_parts, st));
    if (win_end == win_begin) return KMG_OK;
    const uint64_t first_tile = win_begin / EXW_TILE;
    const uint64_t n_tiles = (win_end + EXW_TILE - 1) / EXW_TILE - first_tile;
    KMG_REQUIRE(n_tiles < (1ull << 31), KMG_ERR_RANGE, "too many tiles");
    ExtractParams p;
    fill_common(p, d_bases, n_bases, win_begin, win_end, EXW_TILE, k, d_lut256);
    p.comp16 = d_comp16;
    p.part_lo = 0;
    p.part_hi = (uint32_t)n_parts;
    p.wide_parts = d_wide_parts;
    p.part_counts = reinterpret_cast<unsigned long long*>(d_counts);
    return dispatch_wide_any<2>(p, (uint32_t)n_tiles, k, rc, 0, st);
}
