// Front end of the narrow extraction kernels (extract.cu: extract_narrow_kernel, prefix16_hist_kernel;
// dist_extract.cu: extract_scatter_kernel).
//
// K1: a tile of 16-base words is staged in shared memory as 2-bit codes (first base in the top bits)
// plus two bitmasks (bad-for-narrow, invalid-for-any-stream), so a base is looked up in the LUT
// exactly once.  K2: a thread loads the 96-base code string X0:X1:X2 and the 128-base mask strings
// B0:B1, I0:I1 that start at the word of its first window, decides which of its PPT consecutive
// window starts are valid and builds their keys with funnel shifts.
#pragma once
#include "common.cuh"

namespace kmg {

constexpr int EX_HALO_WORDS = 8;  // 16-base words past the tile that masks/codes may touch

__device__ __forceinline__ uint64_t rev2_64(uint64_t x) {
    x = __brevll(x);
    return ((x >> 1) & 0x5555555555555555ull) | ((x & 0x5555555555555555ull) << 1);
}
__device__ __forceinline__ uint64_t rc_key(uint64_t key, int k) { return rev2_64(~key) >> (64 - 2 * k); }
__device__ __forceinline__ u128 rc_key(const u128& key, int k) {
    uint64_t hi = rev2_64(~key.lo), lo = rev2_64(~key.hi);
    int s = 128 - 2 * k;  // 0 <= s <= 62 because k >= 33
    u128 r;
    if (s == 0) {
        r.lo = lo;
        r.hi = hi;
    } else {
        r.lo = (lo >> s) | (hi << (64 - s));
        r.hi = hi >> s;
    }
    return r;
}

// Strand rule of an extraction kernel (the `rc` argument of kmg.h): the window's key only, the key and its
// reverse complement (two keys per window), or the canonical key (one per window).
constexpr int ST_FWD = 0, ST_BOTH = 1, ST_CANON = KMG_CANONICAL;

// the canonical key: the smaller of the key and its reverse complement (integer order is the string order);
// strand 1 when the reverse complement is strictly smaller, so a palindrome keeps strand 0
template <typename KeyT>
__device__ __forceinline__ KeyT canonical_key(const KeyT& key, int k, uint32_t& strand) {
    const KeyT r = rc_key(key, k);
    strand = r < key ? 1u : 0u;
    return strand ? r : key;
}

template <typename ValT>
__device__ __forceinline__ ValT make_val(uint64_t pos, uint32_t strand) {
    return (ValT)((pos << 1) | strand);
}

// K1: the bases [tile_pos, tile_pos + 16 * WORDS) of bases[0 .. n_bases) as 16-base words of 2-bit codes
// (first base in the top bits) plus the bad-for-narrow and invalid-for-any-stream bitmasks.  (The base
// pointer and count come by value: a reference to the kernel's parameter struct changes its code.)
template <int BLOCK, int WORDS>
__device__ __forceinline__ void encode_tile_words(const uint8_t* bases, uint64_t n_bases, int t, uint64_t tile_pos,
                                                  const uint8_t* s_lut, uint32_t* s_codes, uint16_t* s_bad,
                                                  uint16_t* s_inv) {
    for (int w = t; w < WORDS; w += BLOCK) {
        const uint64_t pos = tile_pos + (uint64_t)w * 16;
        uint32_t b[4];
        if (pos + 16 <= n_bases) {
            const uint4 v = __ldg(reinterpret_cast<const uint4*>(bases + pos));
            b[0] = v.x; b[1] = v.y; b[2] = v.z; b[3] = v.w;
        } else {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                uint32_t x = 0;
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const uint64_t pp = pos + q * 4 + r;
                    // 0xFF is never in an alphabet built by kmg_build_lut; the explicit
                    // range test below does not rely on that.
                    const uint32_t byte = (pp < n_bases) ? bases[pp] : 0xFFu;
                    x |= byte << (8 * r);
                }
                b[q] = x;
            }
        }
        const int nvalid = pos + 16 <= n_bases ? 16 : (pos < n_bases ? (int)(n_bases - pos) : 0);
        uint32_t codes = 0, bad = 0, inv = 0;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const uint32_t byte = (b[j >> 2] >> (8 * (j & 3))) & 0xFFu;
            uint32_t e = s_lut[byte];
            if (j >= nvalid) e = KMG_LUT_INVALID;
            codes |= (e & 3u) << (30 - 2 * j);
            bad |= ((e >> 6) ? 1u : 0u) << (15 - j);
            inv |= (e >> 7) << (15 - j);
        }
        s_codes[w] = codes;
        s_bad[w] = (uint16_t)bad;
        s_inv[w] = (uint16_t)inv;
    }
}

// the 96-base code string X0:X1:X2 and the 128-base mask strings B0:B1 (bad), I0:I1 (invalid) that start
// at word w of the encoded tile
struct TileWords {
    uint64_t X0, X1, X2, B0, B1, I0, I1;
};
__device__ __forceinline__ TileWords load_tile_words(const uint32_t* s_codes, const uint16_t* s_bad, const uint16_t* s_inv,
                                                     int w) {
    TileWords x;
    x.X0 = ((uint64_t)s_codes[w] << 32) | s_codes[w + 1];
    x.X1 = ((uint64_t)s_codes[w + 2] << 32) | s_codes[w + 3];
    x.X2 = ((uint64_t)s_codes[w + 4] << 32) | s_codes[w + 5];
    x.B0 = ((uint64_t)s_bad[w] << 48) | ((uint64_t)s_bad[w + 1] << 32) | ((uint64_t)s_bad[w + 2] << 16) | s_bad[w + 3];
    x.B1 = ((uint64_t)s_bad[w + 4] << 48) | ((uint64_t)s_bad[w + 5] << 32) | ((uint64_t)s_bad[w + 6] << 16) | s_bad[w + 7];
    x.I0 = ((uint64_t)s_inv[w] << 48) | ((uint64_t)s_inv[w + 1] << 32) | ((uint64_t)s_inv[w + 2] << 16) | s_inv[w + 3];
    x.I1 = ((uint64_t)s_inv[w + 4] << 48) | ((uint64_t)s_inv[w + 5] << 32) | ((uint64_t)s_inv[w + 6] << 16) | s_inv[w + 7];
    return x;
}

// Validity of the PPT consecutive window starts first_pos .. first_pos + PPT - 1 (bit j: window j),
// given the 128-base bad / invalid mask strings B0:B1, I0:I1 that start at the word of window 0
// (joff = its base inside that word).  vf: the window lies in [win_begin, win_end) and all its k
// bases are plain (the narrow stream); nwide: windows of the range that belong to the wide stream;
// span_clean: no base of the PPT + k - 1 the windows span is bad (every window of the range is valid).
template <int PPT>
__device__ __forceinline__ uint32_t narrow_window_flags(uint64_t first_pos, uint64_t win_begin, uint64_t win_end, int k,
                                                        int joff, uint64_t B0, uint64_t B1, uint64_t I0, uint64_t I1,
                                                        uint32_t& in_range_mask, bool& span_clean, uint32_t& nwide) {
    {   // window starts [win_begin, win_end) among my PPT positions
        const uint64_t lo = win_begin > first_pos ? win_begin - first_pos : 0;
        const uint64_t hi = win_end > first_pos ? win_end - first_pos : 0;
        const uint32_t l = lo < PPT ? (uint32_t)lo : PPT, h = hi < PPT ? (uint32_t)hi : PPT;
        in_range_mask = h > l ? (((1u << (h - l)) - 1u) << l) : 0u;
    }
    // fast path: no base that is bad for the narrow stream among the PPT+k-1 bases my windows span
    {
        const uint64_t W0 = joff == 0 ? B0 : ((B0 << joff) | (B1 >> (64 - joff)));
        const int span = PPT + k - 1;  // 17 .. 79
        if (span <= 64) span_clean = (W0 >> (64 - span)) == 0;
        else span_clean = W0 == 0 && ((B1 << joff) >> (128 - span)) == 0;
    }
    uint32_t vf = 0;
    nwide = 0;
    if (span_clean) {
        vf = in_range_mask;
    } else {
#pragma unroll
        for (int j = 0; j < PPT; ++j) {
            const int je = joff + j;  // 0..15
            const uint64_t bm = (je == 0 ? B0 : ((B0 << je) | (B1 >> (64 - je)))) >> (64 - k);
            const uint64_t im = (je == 0 ? I0 : ((I0 << je) | (I1 >> (64 - je)))) >> (64 - k);
            const bool in_range = (in_range_mask >> j) & 1u;
            if (in_range && bm == 0) vf |= 1u << j;
            if (in_range && im == 0 && bm != 0) ++nwide;
        }
    }
    return vf;
}

// KeyT: uint64_t (k <= 32) or u128 (33 <= k <= 64).  The key of the window that starts at base je
// (0 <= je <= 15) of the code string X0:X1:X2.
template <typename KeyT>
__device__ __forceinline__ KeyT build_key(uint64_t X0, uint64_t X1, uint64_t X2, int je, int k) {
    const int s2 = 2 * je;
    const uint64_t hi = je == 0 ? X0 : ((X0 << s2) | (X1 >> (64 - s2)));
    KeyT key;
    if constexpr (sizeof(KeyT) == 8) {
        key = hi >> (64 - 2 * k);
    } else {
        const uint64_t lo = je == 0 ? X1 : ((X1 << s2) | (X2 >> (64 - s2)));
        const int s = 128 - 2 * k;
        if (s == 0) {
            key.lo = lo;
            key.hi = hi;
        } else {
            key.lo = (lo >> s) | (hi << (64 - s));
            key.hi = hi >> s;
        }
    }
    return key;
}

// The first key of the window at base je under strand rule STRAND: the window's own key (strand 0), or with
// ST_CANON the canonical key and its strand.
template <int STRAND, typename KeyT>
__device__ __forceinline__ KeyT window_key(uint64_t X0, uint64_t X1, uint64_t X2, int je, int k, uint32_t& strand) {
    const KeyT key = build_key<KeyT>(X0, X1, X2, je, k);
    strand = 0;
    if constexpr (STRAND == ST_CANON) return canonical_key(key, k, strand);
    return key;
}

}  // namespace kmg
