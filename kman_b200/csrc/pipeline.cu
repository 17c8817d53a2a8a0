// The whole device path of one flat base buffer in one call: what FastaBatcher.do
// (kmermaid/batcher.py:454-487: Sequence.kmerator seq.py:284-359 feeding sorted batches,
// batch.py:156-168) followed by KJoiner.join (kmermaid/join.py:63-130 merge + grouping, :243-263
// unique, :265-285 counts) compute for the narrow (plain ACGT) stream.
//
// Stage calls (kmg_extract -> kmg_sort_count) write every key to HBM in extraction order only to read
// it straight back for the first prefix pass of the hybrid sort -- a pass that does not care about
// the order inside a digit.  Here the extraction kernel IS that pass:
//   1. pre-pass over the bases (prefix16_hist_kernel + two small reduce kernels): histogram of the top
//      16 key bits over the exact valid windows -> every 16-bit bucket start, the histograms of the
//      three top key bytes, number of keys, number of wide-stream windows.  100 MB instead of the
//      800 MB a histogram sweep over the keys would read.
//   2. ONE host read-back (32 bytes): key count (grid sizes), skew of the top byte (prefix width).
//   3. pb = 16: extract_narrow_kernel MODE 2 puts the keys straight into the 256 regions of their TOP
//      byte, region_partition_kernel splits every region by byte 2 (bucket starts known: no look-back,
//      no stable ranking), tile bounds come from the bucket starts, local_sort_kernel with the fused
//      count / singleton emission (radix_sort.cu: sort_impl with `pre`).
//      pb = 24: MODE 2 scatters by byte 3, then the two stable prefix passes (onesweep_kernel), tile
//      bounds and the local sort.
//   4. ONE host read-back (the sort's status words, 56 bytes) carries the result count.
// Inputs the hybrid finish does not take (fewer than 2^20 keys, k < 16)
// run kmg_extract + kmg_sort_count / kmg_sort_uniq inside the same call: same result either way.
#include <algorithm>

#include "common.cuh"

extern "C" size_t kmg_rle_workspace_bytes(uint64_t n);
extern "C" size_t kmg_sort_histo_workspace_bytes(uint64_t n, int key_bytes, int end_bit);

namespace kmg {

namespace {
struct PipeWs {
    unsigned long long* zeroed;   // pre-pass: spill [65536] | top [3][256] | plan [4] (see Prefix16Out)
    unsigned long long* top;      // [3][256]
    unsigned long long* plan;     // [2] + counts [2]
    unsigned long long* cursors;  // [256] region starts of the fused scatter
    unsigned long long* starts;   // [65537] 16-bit bucket starts
    unsigned long long* cursors16;  // [65536] bucket cursors of the region partition
    RpTile* rp_tiles;             // tile list of the region partition
    uint32_t rp_tile_keys;
    uint32_t* rows;               // per-CTA rows of the pre-pass
    uint64_t* hist16;             // [16][256] digit histograms of the stage path
    uint64_t* n_out;              // device result count
    void* ex_ws;                  // kmg_extract workspace (stage path)
    size_t ex_ws_bytes;
    void* sort_ws;
    size_t sort_ws_bytes;
    size_t total;
};

// mode as in run_pipeline: 0 count, 1 uniq (val_bytes 4 / 8), 2 histogram
PipeWs carve_pipe(void* ws, uint64_t n_windows, int k, int rc, int val_bytes, int mode) {
    PipeWs w;
    memset(&w, 0, sizeof(w));
    char* p = (char*)ws;
    auto take = [&](size_t bytes) {
        char* r = p;
        p += align_up(bytes, 256);
        return r;
    };
    const int kb = k <= 32 ? 8 : 16;
    const uint64_t cap = std::max<uint64_t>(n_windows * keys_per_window(rc), 1);
    w.zeroed = (unsigned long long*)take(P16_ZEROED_WORDS * sizeof(uint64_t));
    w.top = p16_top(w.zeroed);
    w.plan = p16_plan(w.zeroed);
    w.cursors = (unsigned long long*)take(256 * sizeof(uint64_t));
    w.starts = (unsigned long long*)take(65537 * sizeof(uint64_t));
    w.cursors16 = (unsigned long long*)take(65536 * sizeof(uint64_t));
    w.rp_tile_keys = region_tile_keys(kb, val_bytes);
    w.rp_tiles = (RpTile*)take((cap / w.rp_tile_keys + 257) * sizeof(RpTile));
    w.rows = (uint32_t*)take(prefix16_rows_bytes());
    w.hist16 = (uint64_t*)take(16 * 256 * sizeof(uint64_t));
    w.n_out = (uint64_t*)take(sizeof(uint64_t));
    w.ex_ws_bytes = kmg_extract_workspace_bytes(n_windows);
    w.ex_ws = take(w.ex_ws_bytes);
    // (the sort workspace is not monotone at the upper end of the hybrid range: cover both)
    const uint64_t caps[2] = {cap, std::min<uint64_t>(cap, 1ull << 33)};
    size_t sw = 0;
    for (uint64_t c : caps) {
        const size_t a = mode == 2 ? kmg_sort_histo_workspace_bytes(c, kb, 2 * k)
                         : val_bytes ? kmg_sort_uniq_workspace_bytes(c, kb, val_bytes, 2 * k)
                                     : kmg_sort_count_workspace_bytes(c, kb, 2 * k);
        sw = std::max(sw, a);
    }
    w.sort_ws_bytes = sw;
    w.sort_ws = take(sw);
    w.total = (size_t)(p - (char*)ws);
    return w;
}

int status_from_err(int64_t err) {
    if (err == 2) {
        set_error("a k-mer occurs more than 2^32-1 times: count does not fit uint32");
        return KMG_ERR_RANGE;
    }
    if (err != 0) {
        set_error("device-side look-back spin limit hit (err=%lld)", (long long)err);
        return KMG_ERR_STATE;
    }
    return KMG_OK;
}

// mode 0: (k-mer, count) table, restricted to `range`; mode 1: singletons with payload; mode 2: the multiplicity
// histogram, added to *histo.  h_result: [0] rows of the result, [1] keys sorted (valid narrow windows, x2 with rc = 1),
// [2] windows that belong to the wide stream, [3] selector (0: result in d_keys / d_vals, 1: in the alt
// buffers); mode 2 has no table: [0] and [3] stay 0
int run_pipeline(int mode, const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k, int rc,
                 const uint8_t* d_lut256, void* d_keys, void* d_keys_alt, void* d_vals, void* d_vals_alt, int val_bytes,
                 uint64_t pos_offset, uint32_t* d_counts_out, uint64_t* h_result, void* d_ws, size_t ws_bytes,
                 cudaStream_t st, const HistoOut* histo = nullptr, CountRange range = {}) {
    KMG_REQUIRE(h_result, KMG_ERR_ARG, "h_result is null");
    h_result[0] = h_result[1] = h_result[2] = h_result[3] = 0;
    KMG_REQUIRE(k >= 2, KMG_ERR_ARG, "k must be >= 2, got %d", k);  // batcher.py:477-478
    KMG_REQUIRE(k <= 64, KMG_ERR_RANGE, "k=%d: this build supports k <= 64 (no CPU fallback)", k);
    KMG_REQUIRE(win_begin <= win_end, KMG_ERR_ARG, "win_begin > win_end");
    KMG_REQUIRE(mode != 1 ? val_bytes == 0 : (val_bytes == 4 || val_bytes == 8), KMG_ERR_ARG,
                "val_bytes must be 0 (count) or 4 / 8 (uniq)");
    KMG_REQUIRE(mode != 2 || (histo && histo->hist && histo->big && histo->n_big), KMG_ERR_ARG, "null histogram argument");
    KMG_REQUIRE(d_bases && d_lut256 && d_ws, KMG_ERR_ARG, "null pointer argument");
    KMG_REQUIRE(((uintptr_t)d_bases & 15) == 0, KMG_ERR_ARG, "d_bases must be 16-byte aligned");
    const uint64_t n_win = win_end - win_begin;
    if (n_win == 0) return KMG_OK;
    const int kb = k <= 32 ? 8 : 16;
    KMG_REQUIRE(d_keys && d_keys_alt && (mode != 0 || d_counts_out) && (mode != 1 || (d_vals && d_vals_alt)), KMG_ERR_ARG,
                "null pointer argument");
    KMG_REQUIRE(((uintptr_t)d_keys % kb) == 0 && ((uintptr_t)d_keys_alt % kb) == 0, KMG_ERR_ARG, "key buffers misaligned");
    if (val_bytes == 4)
        KMG_REQUIRE(((pos_offset + n_bases) << 1) < (1ull << 32), KMG_ERR_RANGE, "val_bytes=4 needs < 2^31 positions");
    const PipeWs w = carve_pipe(d_ws, n_win, k, rc, val_bytes, mode);
    KMG_REQUIRE(ws_bytes >= w.total, KMG_ERR_WS, "pipeline workspace too small: %zu < %zu", ws_bytes, w.total);
    const uint64_t cap = n_win * keys_per_window(rc);
    int sel = 0;
    int rcode;

    uint64_t n = 0;
    bool fused = k >= 16 && hybrid_sort_applies(cap, kb, val_bytes, 2 * k, true);
    if (fused) {
        timing_begin(st);
        const Prefix16Out p16{w.zeroed, w.cursors, w.starts, w.cursors16, w.rows, w.rp_tiles, w.rp_tile_keys};
        rcode = extract_prefix16_hist(d_bases, n_bases, win_begin, win_end, k, rc, d_lut256, p16, st);
        timing_end(st, 2);
        if (rcode != KMG_OK) return rcode;
        unsigned long long h_plan[4] = {0, 0, 0, 0};  // keys, largest top-byte count, windows counted, wide windows
        KMG_CUDA(cudaMemcpyAsync(h_plan, w.plan, sizeof(h_plan), cudaMemcpyDeviceToHost, st));
        KMG_CUDA(cudaStreamSynchronize(st));
        n = h_plan[0];
        h_result[1] = n;
        h_result[2] = h_plan[3];
        KMG_REQUIRE(h_plan[2] * keys_per_window(rc) == n, KMG_ERR_STATE,
                    "prefix histogram (%llu keys) disagrees with the window count (%llu)", h_plan[0],
                    h_plan[2] * keys_per_window(rc));
        if (n == 0) return KMG_OK;
        fused = hybrid_sort_applies(n, kb, val_bytes, 2 * k, true);  // (most windows skipped: small after all)
        if (fused) {
            PrePartitioned pre;
            pre.pb = hybrid_choose_pb(n, h_plan[1], kb, val_bytes);
            pre.top = w.top;
            // pb = 16: the keys go to the regions of their TOP byte (cursors: the pre-pass' region starts),
            // then every region is split by byte 2 on its own -- both passes order-free.
            // pb = 24: byte 3 first, then the two stable passes of sort_impl.
            const bool msd = pre.pb == 16;
            if (!msd) exclusive_scan_256(w.top, w.cursors, st);
            timing_begin(st);
            rcode = extract_digit_scatter(d_bases, n_bases, win_begin, win_end, k, rc, d_lut256, d_keys, kb, d_vals, val_bytes,
                                          pos_offset, w.cursors, msd ? 2 * k - 8 : 2 * k - 24, st);
            timing_end(st, 3);
            if (rcode != KMG_OK) return rcode;
            if (msd) {
                timing_begin(st);
                rcode = region_partition(d_keys, d_keys_alt, d_vals, d_vals_alt, n, kb, val_bytes, w.rp_tiles, w.cursors16,
                                         2 * k - 16, st);
                timing_end(st, 0);
                if (rcode != KMG_OK) return rcode;
                pre.bucket_starts = w.starts;
                pre.in_alt = true;
            }
            if (mode == 2)
                rcode = sort_histo_core(d_keys, d_keys_alt, n, kb, 2 * k, nullptr, *histo, w.sort_ws, w.sort_ws_bytes, st, &pre);
            else if (mode == 0)
                rcode = sort_count_core(d_keys, d_keys_alt, n, kb, 2 * k, nullptr, d_counts_out, w.n_out, &sel, w.sort_ws,
                                        w.sort_ws_bytes, st, &pre, range);
            else
                rcode = sort_uniq_core(d_keys, d_keys_alt, d_vals, d_vals_alt, n, kb, val_bytes, 2 * k, nullptr, w.n_out, &sel,
                                       w.sort_ws, w.sort_ws_bytes, st, &pre);
            if (rcode != KMG_OK) return rcode;
        }
    }
    if (!fused) {
        // stage path: position-ordered extraction with every pass' histogram (canonical keys: the sort's own
        // histogram sweep), then the sort
        uint64_t* hist = k >= 4 && rc != KMG_CANONICAL ? w.hist16 : nullptr;
        rcode = kmg_extract(d_bases, n_bases, win_begin, win_end, k, rc, 0, d_lut256, nullptr, d_keys, kb, d_vals, val_bytes,
                            pos_offset, reinterpret_cast<uint64_t*>(w.plan), hist, w.ex_ws, w.ex_ws_bytes, st);
        if (rcode != KMG_OK) return rcode;
        unsigned long long h_cnt[2] = {0, 0};
        KMG_CUDA(cudaMemcpyAsync(h_cnt, w.plan, sizeof(h_cnt), cudaMemcpyDeviceToHost, st));
        rcode = kmg_ws_status(w.ex_ws, st);  // synchronises
        if (rcode != KMG_OK) return rcode;
        n = h_cnt[0];
        h_result[1] = n;
        h_result[2] = h_cnt[1];
        if (n == 0) return KMG_OK;
        if (mode == 2)
            rcode = sort_histo_core(d_keys, d_keys_alt, n, kb, 2 * k, hist, *histo, w.sort_ws, w.sort_ws_bytes, st, nullptr);
        else if (mode == 0)
            rcode = sort_count_core(d_keys, d_keys_alt, n, kb, 2 * k, hist, d_counts_out, w.n_out, &sel, w.sort_ws,
                                    w.sort_ws_bytes, st, nullptr, range);
        else
            rcode = sort_uniq_core(d_keys, d_keys_alt, d_vals, d_vals_alt, n, kb, val_bytes, 2 * k, hist, w.n_out, &sel,
                                   w.sort_ws, w.sort_ws_bytes, st, nullptr);
        if (rcode != KMG_OK) return rcode;
    }
    if (mode == 2) return kmg_ws_status(w.sort_ws, st);  // (synchronises)
    h_result[3] = (uint64_t)sel;
    if (g_stat_last_n_out >= 0 && g_stat_last_err >= 0) {  // the sort's own read-back already has it all
        h_result[0] = (uint64_t)g_stat_last_n_out;
        return status_from_err(g_stat_last_err);
    }
    unsigned long long h_n = 0;
    KMG_CUDA(cudaMemcpyAsync(&h_n, w.n_out, sizeof(h_n), cudaMemcpyDeviceToHost, st));
    rcode = kmg_ws_status(w.sort_ws, st);  // synchronises
    if (rcode != KMG_OK) return rcode;
    h_result[0] = h_n;
    return KMG_OK;
}
}  // namespace

}  // namespace kmg

using namespace kmg;

// keys per destination of the range partition part = ((key >> (2k-16)) * n_parts) >> 16 for a power-of-two
// number of parts: the top log2(n_parts) bits of the top key byte
__global__ void dest_counts_kernel(const unsigned long long* __restrict__ top_row, const unsigned long long* __restrict__ wide,
                                   int shift, int n_parts, unsigned long long* __restrict__ counts) {
    __shared__ unsigned long long s_c[256];
    const int x = threadIdx.x;
    s_c[x] = 0;
    __syncthreads();
    atomicAdd(&s_c[x >> shift], top_row[x]);
    __syncthreads();
    if (x < n_parts) counts[x] = s_c[x];
    if (x == 0) counts[n_parts] = *wide;
}

extern "C" size_t kmg_dest_counts_workspace_bytes(void) {
    return align_up(top_hist_workspace_bytes(), 256) + (3 * 256 + 4) * sizeof(uint64_t);
}

extern "C" int kmg_extract_dest_counts(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k,
                                       int rc, const uint8_t* d_lut256, int n_parts, uint64_t* d_counts, void* d_ws,
                                       size_t ws_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    KMG_REQUIRE(k >= 12 && k <= 64, KMG_ERR_RANGE, "needs 12 <= k <= 64, got %d", k);
    KMG_REQUIRE(n_parts >= 1 && n_parts <= 256 && (n_parts & (n_parts - 1)) == 0, KMG_ERR_ARG,
                "n_parts must be a power of two <= 256, got %d", n_parts);
    KMG_REQUIRE(d_bases && d_lut256 && d_counts && d_ws, KMG_ERR_ARG, "null pointer argument");
    KMG_REQUIRE(ws_bytes >= kmg_dest_counts_workspace_bytes(), KMG_ERR_WS, "dest-counts workspace too small");
    KMG_REQUIRE(win_begin <= win_end, KMG_ERR_ARG, "win_begin > win_end");
    unsigned long long* top = reinterpret_cast<unsigned long long*>((char*)d_ws + align_up(top_hist_workspace_bytes(), 256));
    unsigned long long* plan = top + 3 * 256;  // [0..1] plan, [2..3] window counts
    const int rcode = rc == KMG_CANONICAL
                          ? extract_canonical_top(d_bases, n_bases, win_begin, win_end, k, d_lut256, top + 2 * 256, plan + 2, st)
                          : extract_top_hist(d_bases, n_bases, win_begin, win_end, k, rc, d_lut256,
                                             reinterpret_cast<uint64_t*>(plan + 2), top, plan, d_ws,
                                             top_hist_workspace_bytes(), st);
    if (rcode != KMG_OK) return rcode;
    int g = 0;
    while ((1 << g) < n_parts) ++g;
    dest_counts_kernel<<<1, 256, 0, st>>>(top + 2 * 256, plan + 3, 8 - g, n_parts,
                                          reinterpret_cast<unsigned long long*>(d_counts));
    KMG_LAUNCH_CHECK();
    return KMG_OK;
}

extern "C" size_t kmg_pipeline_workspace_bytes(uint64_t n_windows, int k, int rc, int val_bytes) {
    if (k < 2 || k > 64) return 0;
    return carve_pipe(nullptr, n_windows, k, rc, val_bytes, val_bytes ? 1 : 0).total;
}

extern "C" size_t kmg_pipeline_histo_workspace_bytes(uint64_t n_windows, int k, int rc) {
    if (k < 2 || k > 64) return 0;
    return carve_pipe(nullptr, n_windows, k, rc, 0, 2).total;
}

extern "C" int kmg_extract_sort_count(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k,
                                      int rc, const uint8_t* d_lut256, void* d_keys, void* d_keys_alt,
                                      uint32_t* d_counts_out, uint64_t* h_result, void* d_ws, size_t ws_bytes,
                                      void* stream) {
    return run_pipeline(0, d_bases, n_bases, win_begin, win_end, k, rc, d_lut256, d_keys, d_keys_alt, nullptr, nullptr, 0, 0,
                        d_counts_out, h_result, d_ws, ws_bytes, (cudaStream_t)stream);
}

extern "C" int kmg_extract_sort_count_range(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end,
                                            int k, int rc, const uint8_t* d_lut256, void* d_keys, void* d_keys_alt,
                                            uint32_t min_count, uint32_t max_count, uint32_t* d_counts_out, uint64_t* h_result,
                                            void* d_ws, size_t ws_bytes, void* stream) {
    KMG_REQUIRE(h_result, KMG_ERR_ARG, "h_result is null");
    h_result[0] = h_result[1] = h_result[2] = h_result[3] = 0;
    KMG_REQUIRE(min_count >= 1 && min_count <= max_count, KMG_ERR_ARG, "bad count range [%u, %u]", min_count, max_count);
    return run_pipeline(0, d_bases, n_bases, win_begin, win_end, k, rc, d_lut256, d_keys, d_keys_alt, nullptr, nullptr, 0, 0,
                        d_counts_out, h_result, d_ws, ws_bytes, (cudaStream_t)stream, nullptr, CountRange{min_count, max_count});
}

extern "C" int kmg_extract_sort_uniq(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k,
                                     int rc, const uint8_t* d_lut256, void* d_keys, void* d_keys_alt, void* d_vals,
                                     void* d_vals_alt, int val_bytes, uint64_t pos_offset, uint64_t* h_result, void* d_ws,
                                     size_t ws_bytes, void* stream) {
    return run_pipeline(1, d_bases, n_bases, win_begin, win_end, k, rc, d_lut256, d_keys, d_keys_alt, d_vals, d_vals_alt,
                        val_bytes, pos_offset, nullptr, h_result, d_ws, ws_bytes, (cudaStream_t)stream);
}

extern "C" int kmg_extract_sort_histo(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k,
                                      int rc, const uint8_t* d_lut256, void* d_keys, void* d_keys_alt, uint64_t* d_hist,
                                      uint32_t* d_big, uint64_t* d_n_big, uint64_t* h_result, void* d_ws, size_t ws_bytes,
                                      void* stream) {
    const HistoOut histo{reinterpret_cast<unsigned long long*>(d_hist), d_big, reinterpret_cast<unsigned long long*>(d_n_big),
                         nullptr};
    return run_pipeline(2, d_bases, n_bases, win_begin, win_end, k, rc, d_lut256, d_keys, d_keys_alt, nullptr, nullptr, 0, 0,
                        nullptr, h_result, d_ws, ws_bytes, (cudaStream_t)stream, &histo);
}
