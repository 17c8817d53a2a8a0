// C-ABI glue: error state, options/stats, LUT builder, and the whole-path host-buffer calls
// (what FastaBatcher.do (kmermaid/batcher.py:454-487) followed by KJoiner.join
// (kmermaid/join.py:376-391) do for one flat base buffer).
#include <stdarg.h>

#include <algorithm>
#include <new>

#include "common.cuh"

namespace kmg {

static thread_local char g_err[512] = "";
static thread_local int64_t g_launches = 0;
extern int g_time_passes;
extern int g_hybrid;
extern int g_hybrid_pb;
extern int g_count_fused;
extern int g_local_tile;
extern thread_local int64_t g_stat_hybrid_irregular;
extern thread_local int64_t g_stat_hybrid_path;
extern thread_local int64_t g_stat_hybrid_big_runs;
extern int64_t g_count_limit;
extern thread_local int64_t g_stat_sort_passes;
void timing_collect();
double timing_total_ms(int kind);
int64_t timing_count(int kind);
void timing_reset();

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
void bump_launches(int n) { g_launches += n; }

}  // namespace kmg

using namespace kmg;

extern "C" int kmg_version(void) { return KMG_VERSION; }
extern "C" const char* kmg_last_error(void) { return g_err; }

extern "C" int kmg_device_count(void) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        set_error("cudaGetDeviceCount: %s", cudaGetErrorString(e));
        cudaGetLastError();
        return KMG_ERR_CUDA;
    }
    return n;
}

extern "C" int kmg_set_option(const char* name, int64_t value) {
    KMG_REQUIRE(name, KMG_ERR_ARG, "option name is null");
    if (!strcmp(name, "local_tile")) {
        KMG_REQUIRE(value >= 2048 && value <= 7936, KMG_ERR_ARG, "local_tile must be in [2048,7936]");
        g_local_tile = (int)value;
        return KMG_OK;
    }
    if (!strcmp(name, "count_fused")) {
        g_count_fused = value != 0;
        return KMG_OK;
    }
    if (!strcmp(name, "hybrid_pb")) {
        g_hybrid_pb = (int)value;
        return KMG_OK;
    }
    if (!strcmp(name, "hybrid")) {
        g_hybrid = value != 0;
        return KMG_OK;
    }
    if (!strcmp(name, "count_limit")) {
        KMG_REQUIRE(value >= 0 && value <= 0xffffffffll, KMG_ERR_ARG, "count_limit must be in [0, 2^32-1]");
        g_count_limit = value;
        return KMG_OK;
    }
    if (!strcmp(name, "time_passes")) {
        g_time_passes = (int)value;
        timing_reset();
        return KMG_OK;
    }
    set_error("unknown option '%s'", name);
    return KMG_ERR_ARG;
}

extern "C" int64_t kmg_get_stat(const char* name) {
    if (!name) return -1;
    if (!strcmp(name, "launches")) return g_launches;
    if (!strcmp(name, "sort_passes")) return g_stat_sort_passes;
    if (!strcmp(name, "hybrid_irregular")) return g_stat_hybrid_irregular;
    if (!strcmp(name, "hybrid_path")) return g_stat_hybrid_path;
    if (!strcmp(name, "hybrid_big_runs")) return g_stat_hybrid_big_runs;
    if (!strcmp(name, "n_out")) return g_stat_last_n_out;
    if (!strcmp(name, "ws_err")) return g_stat_last_err;
    if (!strcmp(name, "sort_pass_ns")) {  // total device time of the timed onesweep launches
        timing_collect();
        return (int64_t)(timing_total_ms(0) * 1e6);
    }
    if (!strcmp(name, "sort_pass_count")) {
        timing_collect();
        return timing_count(0);
    }
    if (!strcmp(name, "local_sort_ns")) {  // same for the hybrid finish's local sort launches
        timing_collect();
        return (int64_t)(timing_total_ms(1) * 1e6);
    }
    if (!strcmp(name, "local_sort_count")) {
        timing_collect();
        return timing_count(1);
    }
    if (!strcmp(name, "prepass_ns") || !strcmp(name, "scatter_ns")) {  // pipeline.cu's two extraction launches
        timing_collect();
        return (int64_t)(timing_total_ms(name[0] == 'p' ? 2 : 3) * 1e6);
    }
    if (!strcmp(name, "prepass_count") || !strcmp(name, "scatter_count")) {
        timing_collect();
        return timing_count(name[0] == 'p' ? 2 : 3);
    }
    if (!strcmp(name, "reset_launches")) {
        g_launches = 0;
        return 0;
    }
    return -1;
}

// 16 IUPAC letters (+U) in ASCII order: the 4-bit rank code of the wide stream
static const char kSymbols16[] = "ABCDGHKMNRSTUVWY";

extern "C" int kmg_build_lut(const char* symbols, const char* complement, uint8_t* h_lut256, uint8_t* h_comp16) {
    KMG_REQUIRE(symbols && complement && h_lut256 && h_comp16, KMG_ERR_ARG, "null pointer argument");
    const size_t ns = strlen(symbols);
    KMG_REQUIRE(ns >= 4 && strlen(complement) == ns, KMG_ERR_ARG, "alphabet rows must have equal length >= 4");
    memset(h_lut256, KMG_LUT_INVALID, 256);
    memset(h_comp16, 0, 16);
    // the first four symbols are the plain bases; they must be sorted (A<C<G<T/U) because
    // the 2-bit code has to be monotone in ASCII
    for (int i = 0; i < 4; ++i) {
        const char c = symbols[i];
        KMG_REQUIRE(c >= 'A' && c <= 'Z', KMG_ERR_ARG, "alphabet symbols must be upper-case letters");
        KMG_REQUIRE(i == 0 || symbols[i - 1] < c, KMG_ERR_ARG, "the four plain bases must be in ASCII order");
    }
    for (size_t i = 0; i < ns; ++i) {
        const char c = symbols[i];
        const char* at = strchr(kSymbols16, c);
        const char* cat = strchr(kSymbols16, complement[i]);
        KMG_REQUIRE(at && cat && c != '\0', KMG_ERR_ARG, "symbol '%c' is not an IUPAC nucleotide code", c);
        const uint8_t rank = (uint8_t)(at - kSymbols16);
        uint8_t e = (uint8_t)(rank << 2);
        if (i < 4) e |= (uint8_t)i;
        else e |= KMG_LUT_NONPLAIN;
        h_lut256[(unsigned char)c] = e;
        h_lut256[(unsigned char)(c + 32)] = e;  // seq.py:313: case-folded
        h_comp16[rank] = (uint8_t)(cat - kSymbols16);
    }
    return KMG_OK;
}

// part of a wide key = part of the largest plain 4-mer m <= s (s = its first 4 symbols; m < s unless s is
// plain, since s is then not a plain 4-mer).  m keeps the plain prefix of s, replaces the first other
// symbol by the largest plain base below it (one exists: 'A' is plain and sorts first) and fills up with
// the largest plain base.
extern "C" int kmg_wide_part_table(int rna, int n_parts, uint8_t* h_table65536) {
    KMG_REQUIRE(h_table65536, KMG_ERR_ARG, "null pointer argument");
    KMG_REQUIRE(n_parts >= 1 && n_parts <= 256 && (n_parts & (n_parts - 1)) == 0, KMG_ERR_ARG,
                "n_parts must be a power of two <= 256, got %d", n_parts);
    const char* plain = rna ? "ACGU" : "ACGT";
    int b = 0;
    while ((1 << b) < n_parts) ++b;
    for (uint32_t x = 0; x < 65536; ++x) {
        uint32_t m = 0;  // packed 2-bit codes of the 4-mer, first symbol in the top bits
        bool below = false;
        for (int i = 0; i < 4; ++i) {
            int code = 3;
            if (!below) {
                const char c = kSymbols16[(x >> (12 - 4 * i)) & 0xFu];
                code = 0;
                while (code < 3 && plain[code + 1] <= c) ++code;  // largest plain base <= c
                below = plain[code] != c;
            }
            m = (m << 2) | (uint32_t)code;
        }
        h_table65536[x] = (uint8_t)(m >> (8 - b));
    }
    return KMG_OK;
}

// read back and clear the error word of a stage workspace (synchronises the stream)
extern "C" int kmg_ws_status(void* d_ws, void* stream) {
    KMG_REQUIRE(d_ws, KMG_ERR_ARG, "null workspace");
    WsHeader h;
    KMG_CUDA(cudaMemcpyAsync(&h, d_ws, sizeof(uint32_t) * 2, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    KMG_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    if (h.err == 2) {
        set_error("a k-mer occurs more than 2^32-1 times: count does not fit uint32");
        return KMG_ERR_RANGE;
    }
    if (h.err != 0) {
        set_error("device-side look-back spin limit hit (err=%u)", h.err);
        return KMG_ERR_STATE;
    }
    return KMG_OK;
}

// ---- whole-path context -----------------------------------------------------------------------
struct kmg_ctx {
    int device;
    cudaStream_t stream;
    char* pool;        // one device allocation, grown on demand
    size_t pool_bytes;
    uint8_t* d_lut;
    uint64_t* d_small;  // counters
    uint64_t* d_hist;   // [16][256] digit histograms handed from extract to sort
};

extern "C" int kmg_ctx_create(int device, kmg_ctx** out) {
    KMG_REQUIRE(out, KMG_ERR_ARG, "out is null");
    *out = nullptr;
    KMG_CUDA(cudaSetDevice(device));
    kmg_ctx* c = new (std::nothrow) kmg_ctx();
    KMG_REQUIRE(c, KMG_ERR_ARG, "out of host memory");
    c->device = device;
    c->pool = nullptr;
    c->pool_bytes = 0;
    KMG_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    KMG_CUDA(cudaMalloc(&c->d_lut, 256));
    KMG_CUDA(cudaMalloc(&c->d_small, 64));
    KMG_CUDA(cudaMalloc(&c->d_hist, sizeof(uint64_t) * 16 * 256));
    *out = c;
    return KMG_OK;
}

extern "C" void kmg_ctx_destroy(kmg_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->pool) cudaFree(c->pool);
    cudaFree(c->d_lut);
    cudaFree(c->d_small);
    cudaFree(c->d_hist);
    cudaStreamDestroy(c->stream);
    delete c;
}

static int ctx_reserve(kmg_ctx* c, size_t bytes) {
    if (bytes <= c->pool_bytes) return KMG_OK;
    if (c->pool) KMG_CUDA(cudaFree(c->pool));
    c->pool = nullptr;
    c->pool_bytes = 0;
    KMG_CUDA(cudaMalloc(&c->pool, bytes));
    c->pool_bytes = bytes;
    return KMG_OK;
}

namespace {
struct Carver {
    char* p;
    size_t used;
    void* take(size_t bytes) {
        void* r = p ? p + used : nullptr;
        used += align_up(bytes, 256);
        return r;
    }
};
}  // namespace

// mode 0: count, mode 1: uniq
static int run_host(kmg_ctx* c, int mode, const uint8_t* h_bases, uint64_t n_bases, int k, int rc,
                    const uint8_t* h_lut256, void* h_keys_out, void* h_second_out, uint64_t cap,
                    uint64_t* h_n_out) {
    KMG_REQUIRE(c && h_n_out && h_lut256, KMG_ERR_ARG, "null pointer argument");
    KMG_REQUIRE(h_bases || n_bases == 0, KMG_ERR_ARG, "h_bases is null");
    KMG_REQUIRE(k >= 2, KMG_ERR_ARG, "k must be >= 2, got %d", k);
    KMG_REQUIRE(k <= 64, KMG_ERR_RANGE, "k=%d: this build supports k <= 64", k);
    *h_n_out = 0;
    KMG_CUDA(cudaSetDevice(c->device));
    const int kb = k <= 32 ? 8 : 16;
    const int vb = mode == 1 ? 8 : 0;
    const uint64_t n_win = n_bases >= (uint64_t)k ? n_bases - k + 1 : 0;
    if (n_win == 0) return KMG_OK;
    const uint64_t n_max = n_win * (rc ? 2 : 1);
    const size_t ws_bytes = kmg_pipeline_workspace_bytes(n_win, k, rc, vb);

    Carver cv{nullptr, 0};
    for (int round = 0; round < 2; ++round) {
        cv.used = 0;
        cv.p = round ? c->pool : nullptr;
        cv.take(align_up(n_bases, 16) + 16);
        cv.take(n_max * kb);
        cv.take(n_max * kb);
        if (vb) {
            cv.take(n_max * vb);
            cv.take(n_max * vb);
        }
        if (mode == 0) cv.take(n_max * 4);
        cv.take(ws_bytes);
        if (!round) {
            int rcode = ctx_reserve(c, cv.used);
            if (rcode != KMG_OK) return rcode;
        }
    }
    cv.used = 0;
    uint8_t* d_bases = (uint8_t*)cv.take(align_up(n_bases, 16) + 16);
    char* d_keys = (char*)cv.take(n_max * kb);
    char* d_keys_alt = (char*)cv.take(n_max * kb);
    char* d_vals = nullptr;
    char* d_vals_alt = nullptr;
    if (vb) {
        d_vals = (char*)cv.take(n_max * vb);
        d_vals_alt = (char*)cv.take(n_max * vb);
    }
    uint32_t* d_counts = mode == 0 ? (uint32_t*)cv.take(n_max * 4) : nullptr;
    void* d_ws = cv.take(ws_bytes);
    cudaStream_t st = c->stream;

    KMG_CUDA(cudaMemcpyAsync(c->d_lut, h_lut256, 256, cudaMemcpyHostToDevice, st));
    KMG_CUDA(cudaMemcpyAsync(d_bases, h_bases, n_bases, cudaMemcpyHostToDevice, st));
    // the fused device path: pre-pass, extraction = first prefix pass, remaining passes, local sort
    uint64_t res[4] = {0, 0, 0, 0};
    int rcode;
    if (mode == 0)
        rcode = kmg_extract_sort_count(d_bases, n_bases, 0, n_win, k, rc, c->d_lut, d_keys, d_keys_alt, d_counts, res, d_ws,
                                       ws_bytes, st);
    else
        rcode = kmg_extract_sort_uniq(d_bases, n_bases, 0, n_win, k, rc, c->d_lut, d_keys, d_keys_alt, d_vals, d_vals_alt, vb,
                                      0, res, d_ws, ws_bytes, st);
    if (rcode != KMG_OK) return rcode;
    KMG_REQUIRE(res[2] == 0, KMG_ERR_STATE,
                "input holds %llu windows with non-ACGT alphabet symbols: use the stage API (wide stream)",
                (unsigned long long)res[2]);
    const uint64_t n_out = res[0];
    char* ok = res[3] ? d_keys_alt : d_keys;  // buffer that holds the compacted output
    char* ov = res[3] ? d_vals_alt : d_vals;
    *h_n_out = n_out;
    KMG_REQUIRE(n_out <= cap, KMG_ERR_RANGE, "output capacity %llu < %llu results", (unsigned long long)cap,
                (unsigned long long)n_out);
    if (n_out) {
        KMG_CUDA(cudaMemcpyAsync(h_keys_out, ok, n_out * kb, cudaMemcpyDeviceToHost, st));
        if (mode == 0) KMG_CUDA(cudaMemcpyAsync(h_second_out, d_counts, n_out * 4, cudaMemcpyDeviceToHost, st));
        else KMG_CUDA(cudaMemcpyAsync(h_second_out, ov, n_out * 8, cudaMemcpyDeviceToHost, st));
        KMG_CUDA(cudaStreamSynchronize(st));
    }
    return KMG_OK;
}

extern "C" int kmg_count_host(kmg_ctx* ctx, const uint8_t* h_bases, uint64_t n_bases, int k, int rc,
                              const uint8_t* h_lut256, void* h_keys_out, uint32_t* h_counts_out, uint64_t cap,
                              uint64_t* h_n_out) {
    return run_host(ctx, 0, h_bases, n_bases, k, rc, h_lut256, h_keys_out, h_counts_out, cap, h_n_out);
}

extern "C" int kmg_uniq_host(kmg_ctx* ctx, const uint8_t* h_bases, uint64_t n_bases, int k, int rc,
                             const uint8_t* h_lut256, void* h_keys_out, uint64_t* h_vals_out, uint64_t cap,
                             uint64_t* h_n_out) {
    return run_host(ctx, 1, h_bases, n_bases, k, rc, h_lut256, h_keys_out, h_vals_out, cap, h_n_out);
}
