// Abundance vectors: `kmer count -m VEC_COUNT / VEC_COUNT_MASKED`.
//
// Replaces KJoiner.join_vector_count / join_vector_count_masked (kmermaid/join.py:287-335) and the
// per-position bookkeeping of AbundanceVector.add_count (kmermaid/abundance.py:104-146): for every group of
// equal k-mers the reference parses each member's header and stores, at the member's start position in
// the vector of its (record, strand), the size of the group -- or, masked, the number of members that
// come from OTHER records (groups living in one record store nothing).
//
// On the device the groups are the runs of the stably sorted keys and the member's coordinates are its
// payload, so the whole mode is one scatter: every element finds the bounds of its run by galloping
// from its own index (no serial walk over long runs: poly-N stretches are runs of 10^5 elements) and
// writes its count to out[strand][position].  Masked: inside a run the payloads ascend (stable sort of
// keys emitted in position order), so the members of my own record are one contiguous stretch whose
// ends are two binary searches on the payloads.
#include "common.cuh"

namespace kmg {

template <typename KeyT>
__device__ __forceinline__ uint64_t run_begin(const KeyT* __restrict__ keys, uint64_t i, const KeyT& key) {
    if (i == 0 || keys[i - 1] != key) return i;
    uint64_t step = 2;  // keys[i - 1] == key
    while (step <= i && keys[i - step] == key) step <<= 1;
    // the first equal key lies in (i - step, i - step / 2]  (or [0, ...] when step > i)
    uint64_t lo = step <= i ? i - step + 1 : 0, hi = i - (step >> 1);
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (keys[mid] == key) hi = mid;
        else lo = mid + 1;
    }
    return lo;
}
template <typename KeyT>
__device__ __forceinline__ uint64_t run_end(const KeyT* __restrict__ keys, uint64_t n, uint64_t i, const KeyT& key) {
    if (i + 1 >= n || keys[i + 1] != key) return i + 1;
    uint64_t step = 2;
    while (i + step < n && keys[i + step] == key) step <<= 1;
    // the first different key lies in [i + step / 2 + 1, i + step]  (or n)
    uint64_t lo = i + (step >> 1) + 1, hi = min(i + step, n);
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (keys[mid] == key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}
// first index in [lo, hi) whose payload is >= v
template <typename ValT>
__device__ __forceinline__ uint64_t vals_lower_bound(const ValT* __restrict__ vals, uint64_t lo, uint64_t hi, uint64_t v) {
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if ((uint64_t)vals[mid] < v) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

template <typename KeyT, typename ValT>
__global__ void __launch_bounds__(256) abundance_scatter_kernel(const KeyT* __restrict__ keys, const ValT* __restrict__ vals,
                                                                uint64_t n, const uint64_t* __restrict__ rec_starts,
                                                                uint32_t n_rec, int masked, uint64_t pos_base,
                                                                uint32_t* __restrict__ out_plus, uint32_t* __restrict__ out_minus,
                                                                uint32_t* __restrict__ err) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const KeyT key = keys[i];
    const uint64_t b = run_begin(keys, i, key), e = run_end(keys, n, i, key);
    uint64_t cnt = e - b;
    const uint64_t v = (uint64_t)vals[i];
    const uint64_t pos = v >> 1;
    if (masked) {
        if (cnt == 1) return;
        // my record: last r with rec_starts[r] <= pos
        uint32_t lo = 0, hi = n_rec;
        while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if (rec_starts[mid] <= pos) lo = mid;
            else hi = mid;
        }
        const uint64_t same = vals_lower_bound(vals, b, e, rec_starts[lo + 1] << 1) - vals_lower_bound(vals, b, e, rec_starts[lo] << 1);
        cnt -= same;
        if (cnt == 0) return;
    }
    if (cnt > 0xffffffffull) {
        atomicExch(err, 2u);
        return;
    }
    ((v & 1) ? out_minus : out_plus)[pos - pos_base] = (uint32_t)cnt;
}

// Length of every (record, strand) vector: its last non-zero position + 1 (abundance.py:137-146 grows a
// vector only up to the positions that were written).  One tile of EXT_TILE positions per block and
// strand; a tile inside one record (all but at most n_rec - 1 of them) reduces to one atomicMax.
constexpr int EXT_BLOCK = 256;
constexpr int EXT_ITEMS = 16;
constexpr uint64_t EXT_TILE = (uint64_t)EXT_BLOCK * EXT_ITEMS;

__device__ __forceinline__ uint32_t record_of(const uint64_t* __restrict__ rec_starts, uint32_t n_rec, uint64_t pos) {
    uint32_t lo = 0, hi = n_rec;  // last r with rec_starts[r] <= pos
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (rec_starts[mid] <= pos) lo = mid;
        else hi = mid;
    }
    return lo;
}

__global__ void __launch_bounds__(EXT_BLOCK) vector_extents_kernel(const uint32_t* __restrict__ plus,
                                                                   const uint32_t* __restrict__ minus, uint64_t n,
                                                                   const uint64_t* __restrict__ rec_starts, uint32_t n_rec,
                                                                   unsigned long long* __restrict__ lengths) {
    __shared__ uint32_t s_rec[2];
    __shared__ unsigned long long s_max[EXT_BLOCK / 32];
    const uint32_t strand = blockIdx.y;
    const uint32_t* __restrict__ v = strand ? minus : plus;
    const uint64_t base = (uint64_t)blockIdx.x * EXT_TILE;
    const uint64_t end = min(base + EXT_TILE, n);
    if (threadIdx.x == 0) {
        s_rec[0] = record_of(rec_starts, n_rec, base);
        s_rec[1] = record_of(rec_starts, n_rec, end - 1);
    }
    __syncthreads();
    const uint32_t r0 = s_rec[0];
    const bool one_record = r0 == s_rec[1];
    unsigned long long last = 0;  // one past the last non-zero position seen (0: none)
#pragma unroll
    for (int j = 0; j < EXT_ITEMS; ++j) {
        const uint64_t i = base + (uint64_t)j * EXT_BLOCK + threadIdx.x;
        if (i >= end || v[i] == 0) continue;
        if (one_record) {
            last = i + 1;
        } else {
            const uint32_t r = record_of(rec_starts, n_rec, i);
            atomicMax(&lengths[2 * r + strand], (unsigned long long)(i + 1 - rec_starts[r]));
        }
    }
    if (!one_record) return;  // (uniform across the block)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
    if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = last;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long m = 0;
#pragma unroll
        for (int w = 0; w < EXT_BLOCK / 32; ++w) m = max(m, s_max[w]);
        if (m) atomicMax(&lengths[2 * r0 + strand], m - rec_starts[r0]);
    }
}

}  // namespace kmg

using namespace kmg;

extern "C" int kmg_abundance_scatter(const void* d_sorted_keys, const void* d_vals, uint64_t n, int key_bytes, int val_bytes,
                                     const uint64_t* d_rec_starts, uint32_t n_rec, int masked, uint64_t pos_base,
                                     uint32_t* d_out_plus, uint32_t* d_out_minus, uint32_t* d_err, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    KMG_REQUIRE(key_bytes == 8 || key_bytes == 16 || key_bytes == 32, KMG_ERR_ARG, "key_bytes must be 8, 16 or 32");
    KMG_REQUIRE(val_bytes == 4 || val_bytes == 8, KMG_ERR_ARG, "val_bytes must be 4 or 8");
    if (n == 0) return KMG_OK;
    KMG_REQUIRE(d_sorted_keys && d_vals && d_rec_starts && d_out_plus && d_out_minus && d_err && n_rec >= 1, KMG_ERR_ARG,
                "null pointer argument");
    const unsigned grid = (unsigned)((n + 255) / 256);
    KMG_REQUIRE((n + 255) / 256 < (1ull << 31), KMG_ERR_RANGE, "too many elements");
#define KMG_AB_LAUNCH(K, V)                                                                                         \
    abundance_scatter_kernel<K, V><<<grid, 256, 0, st>>>((const K*)d_sorted_keys, (const V*)d_vals, n, d_rec_starts, n_rec, \
                                                        masked, pos_base, d_out_plus, d_out_minus, d_err)
    if (key_bytes == 8) {
        if (val_bytes == 4) KMG_AB_LAUNCH(uint64_t, uint32_t);
        else KMG_AB_LAUNCH(uint64_t, uint64_t);
    } else if (key_bytes == 16) {
        if (val_bytes == 4) KMG_AB_LAUNCH(u128, uint32_t);
        else KMG_AB_LAUNCH(u128, uint64_t);
    } else {
        if (val_bytes == 4) KMG_AB_LAUNCH(u256, uint32_t);
        else KMG_AB_LAUNCH(u256, uint64_t);
    }
#undef KMG_AB_LAUNCH
    KMG_LAUNCH_CHECK();
    return KMG_OK;
}

extern "C" int kmg_vector_extents(const uint32_t* d_plus, const uint32_t* d_minus, uint64_t n, const uint64_t* d_rec_starts,
                                  uint32_t n_rec, uint64_t* d_lengths_out, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    KMG_REQUIRE(d_lengths_out && d_rec_starts && n_rec >= 1, KMG_ERR_ARG, "null pointer argument");
    KMG_CUDA(cudaMemsetAsync(d_lengths_out, 0, 2 * (size_t)n_rec * sizeof(uint64_t), st));
    if (n == 0) return KMG_OK;
    KMG_REQUIRE(d_plus && d_minus, KMG_ERR_ARG, "null pointer argument");
    const uint64_t tiles = (n + EXT_TILE - 1) / EXT_TILE;
    KMG_REQUIRE(tiles < (1ull << 31), KMG_ERR_RANGE, "too many positions");
    vector_extents_kernel<<<dim3((unsigned)tiles, 2), EXT_BLOCK, 0, st>>>(d_plus, d_minus, n, d_rec_starts, n_rec,
                                                                         (unsigned long long*)d_lengths_out);
    KMG_LAUNCH_CHECK();
    return KMG_OK;
}
