// K6: text emission, and the rank merge between the narrow (2-bit) and wide (4-bit) streams.
//
// Replaces the per-group `%`-formatting of KJoiner.join_sequence_count (kmermaid/join.py:284,
// "SEQ\tCOUNT\n") and KJoiner.join_unique (join.py:262, ">HEADER\nSEQ\n" with HEADER =
// SequenceCoords.__repr__ "ref:start-end:strand", kmermaid/seq.py:103-104).
#include <type_traits>

#include "common.cuh"

namespace kmg {

constexpr int FMT_BLOCK = 256;
constexpr int FMT_RPT = 4;  // records per thread
constexpr int FMT_TILE = FMT_BLOCK * FMT_RPT;

__device__ __forceinline__ uint32_t ndigits_u64(uint64_t v) {
    uint32_t d = 1;
    while (v >= 10) {
        v /= 10;
        ++d;
    }
    return d;
}
__device__ __forceinline__ void put_decimal(uint8_t* at, uint64_t v, uint32_t nd) {
    for (int i = (int)nd - 1; i >= 0; --i) {
        at[i] = (uint8_t)('0' + v % 10);
        v /= 10;
    }
}

// symbol q (0 = first base) of a key
template <typename KeyT>
__device__ __forceinline__ uint32_t key_symbol(const KeyT& key, int k, int q, int bits) {
    return key_digit(key, bits * (k - 1 - q), (1u << bits) - 1u);
}

__device__ __forceinline__ uint8_t sym_ascii(uint32_t code, bool wide, bool rna) {
    if (wide) return (uint8_t)"ABCDGHKMNRSTUVWY"[code];
    return (uint8_t)(rna ? "ACGU" : "ACGT")[code];
}

struct FmtParams {
    const void* keys;
    const void* second;  // counts (u32) or vals
    uint64_t n;
    int k, wide, rna, val_bytes;
    const uint64_t* rec_starts;
    uint32_t n_rec;
    const uint8_t* names;
    const uint64_t* name_offs;
    uint8_t* text;
    unsigned long long* bytes_out;
    uint64_t* state;
    uint32_t* ticket;
    uint32_t* err;
};

// "SEQ\tCOUNT\n": the tile's text is assembled in shared memory, then copied out coalesced.
template <typename KeyT>
__global__ void __launch_bounds__(FMT_BLOCK) format_counts_kernel(const FmtParams p) {
    extern __shared__ uint8_t s_text[];  // FMT_TILE * (k + 12)
    __shared__ uint32_t s_scan[FMT_BLOCK / 32 + 1];
    __shared__ uint32_t s_tile;
    __shared__ uint64_t s_base;
    const int t = threadIdx.x;
    if (t == 0) s_tile = atomicAdd(p.ticket, 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint64_t first = (uint64_t)tile * FMT_TILE + (uint64_t)t * FMT_RPT;
    const KeyT* keys = reinterpret_cast<const KeyT*>(p.keys);
    const uint32_t* counts = reinterpret_cast<const uint32_t*>(p.second);
    const int bits = p.wide ? 4 : 2;

    uint32_t cnt[FMT_RPT], nd[FMT_RPT], len = 0;
#pragma unroll
    for (int r = 0; r < FMT_RPT; ++r) {
        const uint64_t i = first + r;
        cnt[r] = i < p.n ? counts[i] : 0;
        nd[r] = i < p.n ? ndigits_u64(cnt[r]) : 0;
        if (i < p.n) len += p.k + 2 + nd[r];
    }
    uint32_t total;
    uint32_t off = block_excl_scan<FMT_BLOCK, uint32_t>(len, s_scan, total);
    if (t < 32) {
        const uint64_t e = tile_prefix_exclusive_warp(p.state, gridDim.x, tile, total, p.err);
        if (t == 0) {
            s_base = e;
            if (tile == gridDim.x - 1) *p.bytes_out = e + total;
        }
    }
#pragma unroll
    for (int r = 0; r < FMT_RPT; ++r) {
        const uint64_t i = first + r;
        if (i >= p.n) break;
        const KeyT key = keys[i];
        uint8_t* at = s_text + off;
        for (int q = 0; q < p.k; ++q) at[q] = sym_ascii(key_symbol(key, p.k, q, bits), p.wide, p.rna);
        at[p.k] = '\t';
        put_decimal(at + p.k + 1, cnt[r], nd[r]);
        at[p.k + 1 + nd[r]] = '\n';
        off += p.k + 2 + nd[r];
    }
    __syncthreads();
    uint8_t* out = p.text + s_base;
    // head bytes up to 4-byte alignment of the destination, then 32-bit words, then the tail
    const uint32_t mis = (uint32_t)((4 - ((uintptr_t)out & 3)) & 3);
    const uint32_t head = mis < total ? mis : total;
    if ((uint32_t)t < head) out[t] = s_text[t];
    const uint32_t words = (total - head) / 4;
    uint32_t* out32 = reinterpret_cast<uint32_t*>(out + head);
    for (uint32_t w = t; w < words; w += FMT_BLOCK) {
        const uint8_t* s = s_text + head + 4 * w;
        out32[w] = (uint32_t)s[0] | ((uint32_t)s[1] << 8) | ((uint32_t)s[2] << 16) | ((uint32_t)s[3] << 24);
    }
    const uint32_t done = head + 4 * words;
    if (done + t < total) out[done + t] = s_text[done + t];
}

// ">NAME:START-END:STRAND\nSEQ\n": one thread per record writes its own line (names have no
// length bound, so no shared-memory staging here).
template <typename KeyT, int VAL_BYTES>
__global__ void __launch_bounds__(FMT_BLOCK) format_uniq_kernel(const FmtParams p) {
    using ValT = typename std::conditional<VAL_BYTES == 4, uint32_t, uint64_t>::type;
    __shared__ uint64_t s_scan[FMT_BLOCK / 32 + 1];
    __shared__ uint32_t s_tile;
    __shared__ uint64_t s_base;
    const int t = threadIdx.x;
    if (t == 0) s_tile = atomicAdd(p.ticket, 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint64_t i = (uint64_t)tile * FMT_BLOCK + t;
    const KeyT* keys = reinterpret_cast<const KeyT*>(p.keys);
    const ValT* vals = reinterpret_cast<const ValT*>(p.second);
    const int bits = p.wide ? 4 : 2;

    uint64_t len = 0, start = 0, end = 0, noff = 0;
    uint32_t nlen = 0, strand = 0, ds = 0, de = 0;
    if (i < p.n) {
        const uint64_t v = vals[i];
        strand = (uint32_t)(v & 1);
        const uint64_t pos = v >> 1;
        // record = last r with rec_starts[r] <= pos
        uint32_t lo = 0, hi = p.n_rec;
        while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if (p.rec_starts[mid] <= pos) lo = mid;
            else hi = mid;
        }
        start = pos - p.rec_starts[lo];
        end = start + p.k;
        noff = p.name_offs[lo];
        nlen = (uint32_t)(p.name_offs[lo + 1] - noff);
        ds = ndigits_u64(start);
        de = ndigits_u64(end);
        len = 1 + nlen + 1 + ds + 1 + de + 1 + 1 + 1 + p.k + 1;
    }
    uint64_t total;
    const uint64_t off = block_excl_scan<FMT_BLOCK, uint64_t>(len, s_scan, total);
    if (t < 32) {
        const uint64_t e = tile_prefix_exclusive_warp(p.state, gridDim.x, tile, total, p.err);
        if (t == 0) {
            s_base = e;
            if (tile == gridDim.x - 1) *p.bytes_out = e + total;
        }
    }
    __syncthreads();
    if (i < p.n) {
        uint8_t* at = p.text + s_base + off;
        *at++ = '>';
        for (uint32_t q = 0; q < nlen; ++q) *at++ = p.names[noff + q];
        *at++ = ':';
        put_decimal(at, start, ds);
        at += ds;
        *at++ = '-';
        put_decimal(at, end, de);
        at += de;
        *at++ = ':';
        *at++ = strand ? '-' : '+';
        *at++ = '\n';
        const KeyT key = keys[i];
        for (int q = 0; q < p.k; ++q) *at++ = sym_ascii(key_symbol(key, p.k, q, bits), p.wide, p.rna);
        *at++ = '\n';
    }
}

// "COUNT\n" per entry of an abundance vector (abundance.py:168-172): the tile scheme of format_counts_kernel
// with lines of 2..11 bytes.
__global__ void __launch_bounds__(FMT_BLOCK) format_vector_kernel(const FmtParams p) {
    __shared__ uint8_t s_text[FMT_TILE * 11];
    __shared__ uint32_t s_scan[FMT_BLOCK / 32 + 1];
    __shared__ uint32_t s_tile;
    __shared__ uint64_t s_base;
    const int t = threadIdx.x;
    if (t == 0) s_tile = atomicAdd(p.ticket, 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint64_t first = (uint64_t)tile * FMT_TILE + (uint64_t)t * FMT_RPT;
    const uint32_t* counts = reinterpret_cast<const uint32_t*>(p.second);

    uint32_t cnt[FMT_RPT], nd[FMT_RPT], len = 0;
#pragma unroll
    for (int r = 0; r < FMT_RPT; ++r) {
        const uint64_t i = first + r;
        cnt[r] = i < p.n ? counts[i] : 0;
        nd[r] = i < p.n ? ndigits_u64(cnt[r]) : 0;
        if (i < p.n) len += nd[r] + 1;
    }
    uint32_t total;
    uint32_t off = block_excl_scan<FMT_BLOCK, uint32_t>(len, s_scan, total);
    if (t < 32) {
        const uint64_t e = tile_prefix_exclusive_warp(p.state, gridDim.x, tile, total, p.err);
        if (t == 0) {
            s_base = e;
            if (tile == gridDim.x - 1) *p.bytes_out = e + total;
        }
    }
#pragma unroll
    for (int r = 0; r < FMT_RPT; ++r) {
        if (first + r >= p.n) break;
        put_decimal(s_text + off, cnt[r], nd[r]);
        s_text[off + nd[r]] = '\n';
        off += nd[r] + 1;
    }
    __syncthreads();
    uint8_t* out = p.text + s_base;
    const uint32_t mis = (uint32_t)((4 - ((uintptr_t)out & 3)) & 3);
    const uint32_t head = mis < total ? mis : total;
    if ((uint32_t)t < head) out[t] = s_text[t];
    const uint32_t words = (total - head) / 4;
    uint32_t* out32 = reinterpret_cast<uint32_t*>(out + head);
    for (uint32_t w = t; w < words; w += FMT_BLOCK) {
        const uint8_t* s = s_text + head + 4 * w;
        out32[w] = (uint32_t)s[0] | ((uint32_t)s[1] << 8) | ((uint32_t)s[2] << 16) | ((uint32_t)s[3] << 24);
    }
    const uint32_t done = head + 4 * words;
    if (done + t < total) out[done + t] = s_text[done + t];
}

// ---- narrow/wide merge ranks ---------------------------------------------------------------------
// For a wide key W (4-bit ASCII-rank symbols, at least one of them not a plain base) let j be
// the first non-plain symbol and c the number of plain bases whose letter sorts before it.
// A narrow key N sorts before W  <=>  N < T(W) with T = ((prefix_j(W) << 2) + c) << 2(k-1-j),
// and T >= 1 always (no symbol sorts before 'A'), so T' = T-1 fits 64 bits even when T = 2^64.
template <typename NarrowT>
__device__ __forceinline__ NarrowT narrow_from_u128(unsigned __int128 v);
template <>
__device__ __forceinline__ uint64_t narrow_from_u128<uint64_t>(unsigned __int128 v) { return (uint64_t)v; }
template <>
__device__ __forceinline__ u128 narrow_from_u128<u128>(unsigned __int128 v) { return u128{(uint64_t)v, (uint64_t)(v >> 64)}; }

// WideT / NarrowT: u128 / uint64_t (k <= 32) or u256 / u128 (k <= 64).  T' = T - 1 is assembled without
// ever holding T (which can be 2^(2k)): T - 1 = ((prefix << 2) + c - 1) << 2 rem | (4^rem - 1), c >= 1.
template <typename WideT, typename NarrowT>
__global__ void wide_threshold_kernel(const WideT* __restrict__ wide, uint64_t n, int k, int rna,
                                      NarrowT* __restrict__ tprime) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const WideT w = wide[i];
    const uint32_t r3 = rna ? 12u : 11u;  // rank of T / U
    unsigned __int128 A = 0;
    int j = 0;
    for (; j < k; ++j) {
        const uint32_t s = key_digit(w, 4 * (k - 1 - j), 0xFu);
        uint32_t code = 4;
        if (s == 0) code = 0;
        else if (s == 2) code = 1;
        else if (s == 4) code = 2;
        else if (s == r3) code = 3;
        if (code < 4) {
            A = (A << 2) | code;
            continue;
        }
        const uint32_t c = (s > 0) + (s > 2) + (s > 4) + (s > r3);  // >= 1: no symbol sorts before 'A'
        A = (A << 2) + (c - 1);
        break;
    }
    // j == k cannot happen for a wide key; treat it as "right after its own narrow twin" (T' = the twin)
    if (j < k) {
        const int rem = k - 1 - j;
        A = (A << (2 * rem)) | ((((unsigned __int128)1) << (2 * rem)) - 1);
    }
    tprime[i] = narrow_from_u128<NarrowT>(A);
}

// rank_of_narrow[j] = #{i : T'_i < N_j}  (lower bound in the non-decreasing T')
template <typename NarrowT>
__global__ void rank_narrow_kernel(const NarrowT* __restrict__ narrow, uint64_t n_narrow,
                                   const NarrowT* __restrict__ tprime, uint64_t n_wide,
                                   uint64_t* __restrict__ rank_of_narrow) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_narrow) return;
    const NarrowT key = narrow[j];
    uint64_t lo = 0, hi = n_wide;
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (tprime[mid] < key) lo = mid + 1;
        else hi = mid;
    }
    rank_of_narrow[j] = lo;
}

// rank_of_wide[i] = #{j : N_j <= T'_i}  (upper bound); tprime may alias rank_of_wide (8-byte narrow keys)
template <typename NarrowT>
__global__ void rank_wide_kernel(const NarrowT* __restrict__ narrow, uint64_t n_narrow, uint64_t n_wide,
                                 const NarrowT* tprime, uint64_t* rank_of_wide) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_wide) return;
    const NarrowT t = tprime[i];
    uint64_t lo = 0, hi = n_narrow;
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (!(t < narrow[mid])) lo = mid + 1;
        else hi = mid;
    }
    rank_of_wide[i] = lo;
}

}  // namespace kmg

using namespace kmg;

extern "C" size_t kmg_format_workspace_bytes(uint64_t n) {
    return sizeof(WsHeader) + align_up(sc_state_words(n / FMT_BLOCK + 2) * sizeof(uint64_t), 256);
}

static int fmt_setup(FmtParams& p, uint64_t n, uint64_t tile, void* d_ws, size_t ws_bytes, uint32_t& tiles,
                     cudaStream_t st) {
    KMG_REQUIRE(d_ws, KMG_ERR_ARG, "null workspace");
    KMG_REQUIRE(ws_bytes >= kmg_format_workspace_bytes(n), KMG_ERR_WS, "format workspace too small");
    const uint64_t nt = (n + tile - 1) / tile;
    KMG_REQUIRE(nt < (1ull << 31), KMG_ERR_RANGE, "too many tiles");
    tiles = (uint32_t)nt;
    KMG_CUDA(cudaMemsetAsync(d_ws, 0, kmg_format_workspace_bytes(n), st));
    WsHeader* hdr = reinterpret_cast<WsHeader*>(d_ws);
    p.state = reinterpret_cast<uint64_t*>(hdr + 1);
    p.ticket = &hdr->ticket;
    p.err = &hdr->err;
    return KMG_OK;
}

extern "C" int kmg_format_counts(const void* d_keys, const uint32_t* d_counts, uint64_t n, int key_bytes, int k,
                                 int wide, int rna, uint8_t* d_text_out, uint64_t* d_bytes_out, void* d_ws,
                                 size_t ws_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    KMG_REQUIRE(d_bytes_out, KMG_ERR_ARG, "d_bytes_out is null");
    KMG_REQUIRE(key_bytes == 8 || key_bytes == 16 || key_bytes == 32, KMG_ERR_ARG, "key_bytes must be 8, 16 or 32");
    KMG_REQUIRE(k >= 2 && k * (wide ? 4 : 2) <= key_bytes * 8, KMG_ERR_ARG, "k=%d does not fit the key", k);
    KMG_CUDA(cudaMemsetAsync(d_bytes_out, 0, sizeof(uint64_t), st));
    if (n == 0) return KMG_OK;
    KMG_REQUIRE(d_keys && d_counts && d_text_out, KMG_ERR_ARG, "null pointer argument");
    FmtParams p;
    memset(&p, 0, sizeof(p));
    uint32_t tiles = 0;
    int rcode = fmt_setup(p, n, FMT_TILE, d_ws, ws_bytes, tiles, st);
    if (rcode != KMG_OK) return rcode;
    p.keys = d_keys;
    p.second = d_counts;
    p.n = n;
    p.k = k;
    p.wide = wide;
    p.rna = rna;
    p.text = d_text_out;
    p.bytes_out = reinterpret_cast<unsigned long long*>(d_bytes_out);
    const size_t smem = (size_t)FMT_TILE * (k + 12);
    if (key_bytes == 8) {
        KMG_CUDA(cudaFuncSetAttribute(format_counts_kernel<uint64_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        format_counts_kernel<uint64_t><<<tiles, FMT_BLOCK, smem, st>>>(p);
    } else if (key_bytes == 16) {
        KMG_CUDA(cudaFuncSetAttribute(format_counts_kernel<u128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        format_counts_kernel<u128><<<tiles, FMT_BLOCK, smem, st>>>(p);
    } else {
        KMG_CUDA(cudaFuncSetAttribute(format_counts_kernel<u256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        format_counts_kernel<u256><<<tiles, FMT_BLOCK, smem, st>>>(p);
    }
    KMG_LAUNCH_CHECK();
    return KMG_OK;
}

extern "C" int kmg_format_uniq(const void* d_keys, const void* d_vals, uint64_t n, int key_bytes, int val_bytes,
                               int k, int wide, int rna, const uint64_t* d_rec_starts, uint32_t n_rec,
                               const uint8_t* d_names, const uint64_t* d_name_offs, uint8_t* d_text_out,
                               uint64_t* d_bytes_out, void* d_ws, size_t ws_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    KMG_REQUIRE(d_bytes_out, KMG_ERR_ARG, "d_bytes_out is null");
    KMG_REQUIRE(key_bytes == 8 || key_bytes == 16 || key_bytes == 32, KMG_ERR_ARG, "key_bytes must be 8, 16 or 32");
    KMG_REQUIRE(val_bytes == 4 || val_bytes == 8, KMG_ERR_ARG, "val_bytes must be 4 or 8");
    KMG_REQUIRE(k >= 2 && k * (wide ? 4 : 2) <= key_bytes * 8, KMG_ERR_ARG, "k=%d does not fit the key", k);
    KMG_CUDA(cudaMemsetAsync(d_bytes_out, 0, sizeof(uint64_t), st));
    if (n == 0) return KMG_OK;
    KMG_REQUIRE(d_keys && d_vals && d_text_out && d_rec_starts && d_names && d_name_offs && n_rec >= 1, KMG_ERR_ARG,
                "null pointer argument");
    FmtParams p;
    memset(&p, 0, sizeof(p));
    uint32_t tiles = 0;
    int rcode = fmt_setup(p, n, FMT_BLOCK, d_ws, ws_bytes, tiles, st);
    if (rcode != KMG_OK) return rcode;
    p.keys = d_keys;
    p.second = d_vals;
    p.n = n;
    p.k = k;
    p.wide = wide;
    p.rna = rna;
    p.val_bytes = val_bytes;
    p.rec_starts = d_rec_starts;
    p.n_rec = n_rec;
    p.names = d_names;
    p.name_offs = d_name_offs;
    p.text = d_text_out;
    p.bytes_out = reinterpret_cast<unsigned long long*>(d_bytes_out);
    if (key_bytes == 8) {
        if (val_bytes == 4) format_uniq_kernel<uint64_t, 4><<<tiles, FMT_BLOCK, 0, st>>>(p);
        else format_uniq_kernel<uint64_t, 8><<<tiles, FMT_BLOCK, 0, st>>>(p);
    } else if (key_bytes == 16) {
        if (val_bytes == 4) format_uniq_kernel<u128, 4><<<tiles, FMT_BLOCK, 0, st>>>(p);
        else format_uniq_kernel<u128, 8><<<tiles, FMT_BLOCK, 0, st>>>(p);
    } else {
        if (val_bytes == 4) format_uniq_kernel<u256, 4><<<tiles, FMT_BLOCK, 0, st>>>(p);
        else format_uniq_kernel<u256, 8><<<tiles, FMT_BLOCK, 0, st>>>(p);
    }
    KMG_LAUNCH_CHECK();
    return KMG_OK;
}

extern "C" int kmg_format_vector(const uint32_t* d_counts, uint64_t n, uint8_t* d_text_out, uint64_t* d_bytes_out,
                                 void* d_ws, size_t ws_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    KMG_REQUIRE(d_bytes_out, KMG_ERR_ARG, "d_bytes_out is null");
    KMG_CUDA(cudaMemsetAsync(d_bytes_out, 0, sizeof(uint64_t), st));
    if (n == 0) return KMG_OK;
    KMG_REQUIRE(d_counts && d_text_out, KMG_ERR_ARG, "null pointer argument");
    FmtParams p;
    memset(&p, 0, sizeof(p));
    uint32_t tiles = 0;
    int rcode = fmt_setup(p, n, FMT_TILE, d_ws, ws_bytes, tiles, st);
    if (rcode != KMG_OK) return rcode;
    p.second = d_counts;
    p.n = n;
    p.text = d_text_out;
    p.bytes_out = reinterpret_cast<unsigned long long*>(d_bytes_out);
    format_vector_kernel<<<tiles, FMT_BLOCK, 0, st>>>(p);
    KMG_LAUNCH_CHECK();
    return KMG_OK;
}

template <typename WideT, typename NarrowT>
static int merge_ranks_impl(const void* d_narrow_keys, uint64_t n_narrow, const void* d_wide_keys, uint64_t n_wide, int k,
                            int rna, uint64_t* d_rank_of_narrow, uint64_t* d_rank_of_wide, NarrowT* d_tprime,
                            cudaStream_t st) {
    if (n_wide) {
        KMG_REQUIRE(d_wide_keys && d_rank_of_wide && d_tprime, KMG_ERR_ARG, "null pointer argument");
        wide_threshold_kernel<WideT, NarrowT><<<(unsigned)((n_wide + 255) / 256), 256, 0, st>>>((const WideT*)d_wide_keys, n_wide, k,
                                                                                               rna, d_tprime);
        KMG_LAUNCH_CHECK();
    }
    if (n_narrow) {
        KMG_REQUIRE(d_narrow_keys && d_rank_of_narrow, KMG_ERR_ARG, "null pointer argument");
        rank_narrow_kernel<NarrowT><<<(unsigned)((n_narrow + 255) / 256), 256, 0, st>>>((const NarrowT*)d_narrow_keys, n_narrow, d_tprime,
                                                                                        n_wide, d_rank_of_narrow);
        KMG_LAUNCH_CHECK();
    }
    if (n_wide) {
        rank_wide_kernel<NarrowT><<<(unsigned)((n_wide + 255) / 256), 256, 0, st>>>((const NarrowT*)d_narrow_keys, n_narrow, n_wide,
                                                                                    d_tprime, d_rank_of_wide);
        KMG_LAUNCH_CHECK();
    }
    return KMG_OK;
}

extern "C" int kmg_merge_ranks(const void* d_narrow_keys, uint64_t n_narrow, int narrow_key_bytes,
                               const void* d_wide_keys, uint64_t n_wide, int wide_key_bytes, int k, int rna,
                               uint64_t* d_rank_of_narrow, uint64_t* d_rank_of_wide, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    KMG_REQUIRE(k >= 2 && k <= 32, KMG_ERR_RANGE, "8-byte narrow / 16-byte wide keys hold k <= 32, got %d (kmg_merge_ranks_wide)", k);
    KMG_REQUIRE(narrow_key_bytes == 8 && wide_key_bytes == 16, KMG_ERR_ARG, "expected 8-byte narrow and 16-byte wide keys");
    // (the thresholds live in the wide rank array until the last kernel turns them into ranks)
    return merge_ranks_impl<u128, uint64_t>(d_narrow_keys, n_narrow, d_wide_keys, n_wide, k, rna, d_rank_of_narrow, d_rank_of_wide,
                                            d_rank_of_wide, st);
}

extern "C" int kmg_merge_ranks_wide(const void* d_narrow_keys, uint64_t n_narrow, const void* d_wide_keys, uint64_t n_wide, int k,
                                    int rna, uint64_t* d_rank_of_narrow, uint64_t* d_rank_of_wide, void* d_tmp16, void* stream) {
    KMG_REQUIRE(k >= 33 && k <= 64, KMG_ERR_RANGE, "16-byte narrow / 32-byte wide keys are for 33 <= k <= 64, got %d", k);
    KMG_REQUIRE(((uintptr_t)d_tmp16 & 15) == 0, KMG_ERR_ARG, "d_tmp16 misaligned");
    return merge_ranks_impl<u256, u128>(d_narrow_keys, n_narrow, d_wide_keys, n_wide, k, rna, d_rank_of_narrow, d_rank_of_wide,
                                        (u128*)d_tmp16, (cudaStream_t)stream);
}
