/*
 * kmg.h -- C ABI of the B200-native k-mer engine (libkmg.so).
 *
 * This is the drop-in boundary for kmermaid's one data-parallel hot path:
 *   extract  (kmermaid/seq.py:284-328, rc :245-282)
 *   sort     (kmermaid/batch.py:156-168)
 *   join     (kmermaid/join.py:63-130 merge+group, :243-263 uniq, :265-285 count)
 * The reference is pure Python and has no FFI layer; these entry points are what a
 * ctypes binding in kmermaid/batcher.py + kmermaid/join.py would call (INTEGRATION.md).
 *
 * Conventions
 *   - plain C types only; every `d_*` pointer is a CUDA device pointer owned by the
 *     caller, every `h_*` pointer is host memory owned by the caller;
 *   - the library keeps no reference to caller memory after a call returns, except that
 *     device work enqueued on `stream` may still be running (stage calls are asynchronous
 *     with respect to the host unless stated otherwise);
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - scratch memory is provided by the caller, sized by the matching *_workspace_bytes();
 *   - return value: 0 = OK, <0 = error; kmg_last_error() gives the thread-local message;
 *   - there is NO CPU fallback: without a CUDA device every compute call fails.
 *
 * Key format ("narrow" stream, windows made only of the four plain bases):
 *   k <= 32 : uint64, k <= 64 : 128-bit {lo, hi} little-endian limbs (16-byte aligned);
 *   value = sum(code[j] << 2*(k-1-j)), A<C<G<T(U) = 0,1,2,3 -- integer order == the
 *   reference's string order (batch.py:156-168) for equal-length upper-case strings.
 * Key format ("wide" stream, windows that pass the alphabet test but hold >= 1 other
 *   symbol, e.g. N): 4-bit ASCII-rank codes over "ABCDGHKMNRSTUVWY", MSB first,
 *   k <= 32 : 128-bit {lo, hi}; k <= 64 : 256-bit, four little-endian 64-bit limbs (key_bytes = 32).
 * Payload ("val") format: (global window start in the flat base buffer << 1) | strand
 *   (0 '+', 1 '-'), as uint32 (val_bytes 4) or uint64 (val_bytes 8).
 */
#ifndef KMG_H_
#define KMG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KMG_VERSION 100 /* 0.1.0 */

#define KMG_OK 0
#define KMG_ERR_ARG (-1)    /* invalid argument (the reference raises AssertionError) */
#define KMG_ERR_CUDA (-2)   /* CUDA runtime error */
#define KMG_ERR_WS (-3)     /* workspace too small */
#define KMG_ERR_RANGE (-4)  /* size beyond what this build supports */
#define KMG_ERR_STATE (-5)  /* device-side consistency check failed */

/* LUT byte layout (one entry per input byte value, see kmg_build_lut):
 *   bit 7    : symbol not in the alphabet -> every window touching it is skipped
 *              (seq.py:318-327)
 *   bit 6    : symbol in the alphabet but not one of the four plain bases
 *   bits 5:2 : 4-bit ASCII rank code (wide stream)
 *   bits 1:0 : 2-bit code (narrow stream)                                         */
#define KMG_LUT_INVALID 0x80u
#define KMG_LUT_NONPLAIN 0x40u

/* Bins of a multiplicity histogram (kmg_sort_histo and friends): d_hist[m] for m < KMG_HISTO_BINS,
 * larger multiplicities go to a list. */
#define KMG_HISTO_BINS 4096

int kmg_version(void);
const char* kmg_last_error(void);
/* number of CUDA devices visible, or <0 */
int kmg_device_count(void);

/* Host helper: fill lut[256] and comp4[16] from an alphabet given as the reference gives
 * it: `symbols` and `complement` are the two rows of oligo_melting.AB_NA[t]
 * (used at seq.py:318 and seq.py:279); case-folding per seq.py:313. */
int kmg_build_lut(const char* symbols, const char* complement, uint8_t* h_lut256, uint8_t* h_comp16);

/* Read back (and thereby wait for) the status word of a stage workspace after the stage's
 * kernels were enqueued on `stream`: KMG_OK, KMG_ERR_STATE (device-side look-back gave up)
 * or KMG_ERR_RANGE (a run length overflowed uint32).  Synchronises the stream. */
int kmg_ws_status(void* d_ws, void* stream);

/* ---- K1+K2: encode + rolling-window extraction (seq.py:284-328, rc :245-282) ----------
 * Emits, in position order ('+' then '-' per position when rc), the keys of all windows
 * whose start lies in [win_begin, win_end) of the flat buffer d_bases[0..n_bases) and that
 *   wide == 0 : consist only of plain bases (narrow stream, 2-bit codes)
 *   wide == 1 : pass the alphabet test and contain >= 1 non-plain symbol (4-bit codes)
 * Record separators are any byte the LUT marks invalid (the loader uses '\n').
 * d_vals_out may be NULL (val_bytes 0).  `pos_offset` is added to the window start before
 * it is stored in the payload (multi-GPU chunks).
 * d_counts[0] = number of keys emitted, d_counts[1] (narrow only) = number of windows
 * that belong to the wide stream.  Output capacity must be (win_end-win_begin)*(1+rc).
 * d_hist_out (optional, narrow stream, k >= 4): uint64[16][256] digit histograms of the emitted
 * keys for kmg_radix_sort's pass plan over bits [0, 2k), derived from one 4-mer histogram of
 * the bases; hand it to kmg_radix_sort(d_hist_in) to skip the sort's own histogram sweep.
 * For 8-byte keys and k >= 12, rows 13..15 additionally hold the histograms of the three top
 * key bytes (bits [2k-24, 2k)), which the hybrid sort's prefix passes use. */
size_t kmg_extract_workspace_bytes(uint64_t n_windows);
int kmg_extract(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k, int rc,
                int wide, const uint8_t* d_lut256, const uint8_t* d_comp16, void* d_keys_out, int key_bytes,
                void* d_vals_out, int val_bytes, uint64_t pos_offset, uint64_t* d_counts, uint64_t* d_hist_out,
                void* d_ws, size_t ws_bytes, void* stream);

/* ---- K1+K2 by key range: one pass of a sorted output that does not fit the device at once ----------
 * With n_parts = 2^b parts (b <= 8), the part of a narrow key is its top b bits, key >> (2k - b) (the
 * first bases; the same rule as kmg_range_partition and kmg_extract_dest_counts for power-of-two
 * n_parts).  The part of a wide key follows the merged string order: if its first 4 symbols s are plain
 * bases it is the narrow part of that 4-mer, otherwise the part of the largest plain 4-mer that sorts
 * below s.  So every wide key of part p sorts after all narrow keys of parts < p and before all narrow
 * keys of parts > p, and concatenating the per-part outputs in part order gives the whole sorted output.
 *
 * kmg_wide_part_table (host): h_table65536[x] = part of a wide key whose top 16 bits are x (its first
 * 4 symbols), for DNA (plain ACGT) or RNA (rna != 0, plain ACGU).  Copy it to the device for the calls
 * below. */
int kmg_wide_part_table(int rna, int n_parts, uint8_t* h_table65536);
/* kmg_extract restricted to the keys whose part lies in [part_lo, part_hi) (k >= 4): the kept keys in
 * the same position order ('+' before '-' per position), so equal keys keep their emission order.
 * Keys that are not kept are neither stored nor counted: d_counts[0] = keys stored, d_counts[1]
 * (narrow) = windows of the wide stream in the whole window range.  Output capacity = the exact number
 * of keys in the range (kmg_extract_dest_counts, kmg_extract_wide_part_counts).  d_wide_parts: device
 * copy of kmg_wide_part_table's table (required for wide = 1).  d_hist_out must be NULL (KMG_ERR_ARG):
 * the 4-mer-derived histograms describe every key, not the kept ones.  Workspace:
 * kmg_extract_workspace_bytes(win_end - win_begin). */
int kmg_extract_parts(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k, int rc,
                      int wide, const uint8_t* d_lut256, const uint8_t* d_comp16, int n_parts, int part_lo, int part_hi,
                      const uint8_t* d_wide_parts, void* d_keys_out, int key_bytes, void* d_vals_out, int val_bytes,
                      uint64_t pos_offset, uint64_t* d_counts, uint64_t* d_hist_out, void* d_ws, size_t ws_bytes,
                      void* stream);
/* Keys of the wide stream per part (count-only launch of the filtered wide extraction, k >= 4):
 * d_counts[0..n_parts).  d_comp16 is required with rc (the '-' key has its own part). */
int kmg_extract_wide_part_counts(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k,
                                 int rc, const uint8_t* d_lut256, const uint8_t* d_comp16, int n_parts,
                                 const uint8_t* d_wide_parts, uint64_t* d_counts, void* stream);

/* ---- K3: HBM-resident LSD radix sort (batch.py:156-168 + the merge of join.py:63-93) --
 * Stable, sorts on key bits [begin_bit, end_bit).  Ping-pongs between (keys, keys_alt)
 * [and (vals, vals_alt)]; *h_selector_out (host, written before return) is 0 if the
 * result is in keys/vals, 1 if in keys_alt/vals_alt.  d_hist_in (optional): the digit histograms
 * kmg_extract produced for exactly these keys (requires begin_bit 0, end_bit 2k).
 * Key-only sorts over bits [0, end_bit), end_bit >= 32, with 2^20 <= n <= 2^33 take the "hybrid
 * finish": 2-3 ordinary passes over the top 16/24 bits (the first of them without stable
 * ranking), then ONE shared-memory local sort per ~6000-key tile orders all remaining bits
 * (local_sort.cuh: local_sort_kernel).  Tiles the local scheme cannot hold (prefix buckets above
 * 8192 keys, 4096 for 16-byte keys: repeats) are gathered, sorted by the plain LSD passes and put back; above n/8 such
 * keys the plain passes sort everything.  The result is identical on every path.  The call
 * synchronises the stream in that mode (2 KB histogram read-back unless d_hist_in is given; one
 * 56-byte read-back of the status words after the local sort).
 * All keys must agree in the bits at and above end_bit in that mode (kmg_extract's keys do: those
 * bits are zero; after kmg_range_partition they are the rank's common prefix).
 * kmg_set_option("hybrid", 0) switches it off. */
size_t kmg_radix_sort_workspace_bytes(uint64_t n, int key_bytes, int val_bytes, int begin_bit, int end_bit);
int kmg_radix_sort(void* d_keys, void* d_keys_alt, void* d_vals, void* d_vals_alt, uint64_t n, int key_bytes,
                   int val_bytes, int begin_bit, int end_bit, const uint64_t* d_hist_in, int* h_selector_out,
                   void* d_ws, size_t ws_bytes, void* stream);

/* ---- K4: run-length / unique on sorted keys (join.py:95-130, :265-285, :243-263) ------
 * rle_count: distinct keys ascending + run lengths; *d_n_out = number of runs.
 * select_singletons: keys (and payload) of runs of length exactly 1. */
size_t kmg_rle_workspace_bytes(uint64_t n);
int kmg_rle_count(const void* d_sorted_keys, uint64_t n, int key_bytes, void* d_uniq_keys_out,
                  uint32_t* d_counts_out, uint64_t* d_n_out, void* d_ws, size_t ws_bytes, void* stream);
/* Keeps the rows of a count table (n 8-, 16- or 32-byte keys and their counts) with
 * min_count <= count <= max_count, in their order; *d_n_out (device) = their number.  May run in place
 * (d_keys_out == d_keys and d_counts_out == d_counts); other overlaps are undefined.  KMG_ERR_ARG unless
 * 1 <= min_count <= max_count.  Workspace: kmg_rle_workspace_bytes(n). */
int kmg_filter_counts(const void* d_keys, const uint32_t* d_counts, uint64_t n, int key_bytes, uint32_t min_count,
                      uint32_t max_count, void* d_keys_out, uint32_t* d_counts_out, uint64_t* d_n_out, void* d_ws,
                      size_t ws_bytes, void* stream);

/* sort + rle_count in one call (the count path: join.py:63-130 after batch.py:156-168).  Sorts
 * the n keys on bits [0, end_bit) and leaves the distinct keys ascending in d_keys
 * (*h_selector_out = 0) or d_keys_alt (1), their multiplicities in d_counts_out and their number
 * in *d_n_out (device); the other key buffer is scratch.  When the hybrid finish applies (see
 * kmg_radix_sort) its local sort emits the table directly and the sorted keys are never written
 * or re-read; otherwise this is kmg_radix_sort followed by kmg_rle_count.  Same result either way. */
size_t kmg_sort_count_workspace_bytes(uint64_t n, int key_bytes, int end_bit);
int kmg_sort_count(void* d_keys, void* d_keys_alt, uint64_t n, int key_bytes, int end_bit, const uint64_t* d_hist_in,
                   uint32_t* d_counts_out, uint64_t* d_n_out, int* h_selector_out, void* d_ws, size_t ws_bytes,
                   void* stream);
/* kmg_sort_count's table restricted to the rows with min_count <= count <= max_count (KMG_ERR_ARG unless
 * 1 <= min_count <= max_count), in the same order.  The full range [1, 2^32-1] is kmg_sort_count.  Otherwise
 * the hybrid finish's local sort writes only the kept rows; where it does not finish the table (plain
 * passes, tiles it cannot hold) kmg_sort_count's table is compacted in place with kmg_filter_counts.  A run
 * beyond uint32 is KMG_ERR_RANGE whatever the range.  Workspace: kmg_sort_count_workspace_bytes. */
int kmg_sort_count_range(void* d_keys, void* d_keys_alt, uint64_t n, int key_bytes, int end_bit, const uint64_t* d_hist_in,
                         uint32_t min_count, uint32_t max_count, uint32_t* d_counts_out, uint64_t* d_n_out,
                         int* h_selector_out, void* d_ws, size_t ws_bytes, void* stream);
/* sort + select_singletons in one call (the uniq path: join.py:63-130 + join_unique :243-263).
 * Leaves the keys that occur exactly once, ascending, with their payload in (d_keys, d_vals)
 * (*h_selector_out = 0) or (d_keys_alt, d_vals_alt) (1); *d_n_out (device) = their number.  Because
 * repeated keys are dropped, their relative order does not matter and the keys take the
 * hybrid finish with the payload following through a 16-bit index (tiles of 6144 8-byte / 4096
 * 16-byte keys); its local
 * sort emits the singletons itself unless irregular tiles force sort + kmg_select_singletons. */
size_t kmg_sort_uniq_workspace_bytes(uint64_t n, int key_bytes, int val_bytes, int end_bit);
int kmg_sort_uniq(void* d_keys, void* d_keys_alt, void* d_vals, void* d_vals_alt, uint64_t n, int key_bytes,
                  int val_bytes, int end_bit, const uint64_t* d_hist_in, uint64_t* d_n_out, int* h_selector_out,
                  void* d_ws, size_t ws_bytes, void* stream);
int kmg_select_singletons(const void* d_sorted_keys, const void* d_vals, uint64_t n, int key_bytes, int val_bytes,
                          void* d_keys_out, void* d_vals_out, uint64_t* d_n_out, void* d_ws, size_t ws_bytes,
                          void* stream);
/* The multiplicity spectrum of the keys (`kmer histo`: what a histogram of kmg_sort_count's counts
 * gives) without the table.  Output, ADDED to the caller's arrays (zero them once, then sum streams and
 * passes on the device):
 *   d_hist[KMG_HISTO_BINS]: d_hist[m] = distinct keys that occur exactly m times (m >= 1);
 *   d_big[] / *d_n_big: one entry per distinct key that occurs >= KMG_HISTO_BINS times, its multiplicity,
 *   in no particular order, appended at *d_n_big.  Capacity (total keys) / KMG_HISTO_BINS + 1 always holds.
 * kmg_sort_histo consumes both key buffers (sorts n 8- or 16-byte keys on bits [0, end_bit)).  When the
 * hybrid finish applies, its local sort adds every tile's run lengths to the histogram and writes no key
 * (no output order, no compaction); tiles it cannot hold (huge prefix buckets: repeats) are gathered,
 * sorted with the plain passes and histogrammed on the side ("hybrid_path" 2), above n/8 such keys all
 * keys are sorted and histogrammed ("hybrid_path" 3).  The status word (kmg_ws_status(d_ws)) becomes
 * KMG_ERR_RANGE for a multiplicity beyond uint32, as in the count path.
 * kmg_count_histogram: the same histogram of an existing count table (d_counts[0..n)); no workspace. */
size_t kmg_sort_histo_workspace_bytes(uint64_t n, int key_bytes, int end_bit);
int kmg_sort_histo(void* d_keys, void* d_keys_alt, uint64_t n, int key_bytes, int end_bit, const uint64_t* d_hist_in,
                   uint64_t* d_hist, uint32_t* d_big, uint64_t* d_n_big, void* d_ws, size_t ws_bytes, void* stream);
int kmg_count_histogram(const uint32_t* d_counts, uint64_t n, uint64_t* d_hist, uint32_t* d_big, uint64_t* d_n_big,
                        void* stream);

/* ---- K1-K4 in one call: the device path of `kmer count` / `kmer uniq` for the narrow stream -------
 * (FastaBatcher.do batcher.py:454-487 + KJoiner.join join.py:337-391 on one flat base buffer.)
 * Same results as kmg_extract followed by kmg_sort_count / kmg_sort_uniq, but when the hybrid sort
 * applies (>= 2^20 keys, k >= 16) the extraction kernel itself is the sort's
 * first prefix pass: a pre-pass over the BASES (the 16-bit prefix histogram of the valid windows)
 * yields the histograms of the top key bytes, then every key is written once, straight into the region
 * of its digit -- the keys are never stored in extraction order.  Two host synchronisations per call
 * (32 + 56 bytes read back).
 * d_keys / d_keys_alt (and d_vals / d_vals_alt): capacity (win_end-win_begin)*(1+rc) items each.
 * h_result[4] (host): [0] rows of the result ((k-mer, count) pairs / singletons), [1] keys that were
 * sorted, [2] windows that belong to the WIDE stream (the caller runs those through the stage
 * API), [3] selector: 0 = result keys in d_keys (payload in d_vals), 1 = in the alt buffers.
 * count: multiplicities in d_counts_out[0 .. h_result[0]). */
size_t kmg_pipeline_workspace_bytes(uint64_t n_windows, int k, int rc, int val_bytes);
int kmg_extract_sort_count(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k, int rc,
                           const uint8_t* d_lut256, void* d_keys, void* d_keys_alt, uint32_t* d_counts_out,
                           uint64_t* h_result, void* d_ws, size_t ws_bytes, void* stream);
/* kmg_extract_sort_count with kmg_sort_count_range's finish: only the rows with
 * min_count <= count <= max_count; h_result[0] counts them.  Workspace: kmg_pipeline_workspace_bytes(n, k, rc, 0). */
int kmg_extract_sort_count_range(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k,
                                 int rc, const uint8_t* d_lut256, void* d_keys, void* d_keys_alt, uint32_t min_count,
                                 uint32_t max_count, uint32_t* d_counts_out, uint64_t* h_result, void* d_ws,
                                 size_t ws_bytes, void* stream);
int kmg_extract_sort_uniq(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k, int rc,
                          const uint8_t* d_lut256, void* d_keys, void* d_keys_alt, void* d_vals, void* d_vals_alt,
                          int val_bytes, uint64_t pos_offset, uint64_t* h_result, void* d_ws, size_t ws_bytes,
                          void* stream);
/* The same front end with kmg_sort_histo's finish: the narrow stream's multiplicity histogram added to
 * d_hist / d_big / d_n_big (see kmg_sort_histo).  h_result as above, except that there is no table:
 * [0] and [3] are 0.  Three host synchronisations (the last one reads the status word). */
size_t kmg_pipeline_histo_workspace_bytes(uint64_t n_windows, int k, int rc);
int kmg_extract_sort_histo(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k, int rc,
                           const uint8_t* d_lut256, void* d_keys, void* d_keys_alt, uint64_t* d_hist, uint32_t* d_big,
                           uint64_t* d_n_big, uint64_t* h_result, void* d_ws, size_t ws_bytes, void* stream);

/* ---- K5: range partition for the multi-GPU exchange (no reference counterpart) --------
 * Stable split of keys into n_parts contiguous regions of the output by
 *   part = ((key >> (key_bits-16)) * n_parts) >> 16      (key_bits >= 16)
 * so that concatenating the parts' sorted contents in part order is globally sorted.
 * d_part_counts[n_parts] receives the region sizes. */
size_t kmg_partition_workspace_bytes(uint64_t n, int key_bytes, int val_bytes);
int kmg_range_partition(const void* d_keys, const void* d_vals, uint64_t n, int key_bytes, int val_bytes,
                        int key_bits, int n_parts, void* d_keys_out, void* d_vals_out, uint64_t* d_part_counts,
                        void* d_ws, size_t ws_bytes, void* stream);

/* ---- K5b: fused extraction + range partition + peer-memory exchange (multi-GPU) --------
 * Same extraction as kmg_extract (narrow stream), but every key is stored straight into the
 * receive buffer of the GPU that owns its key range (part as in kmg_range_partition, with
 * key_bits = 2k; needs k >= 8): d_dest_keys / d_dest_vals are DEVICE arrays of n_parts
 * pointers (peer-mapped, e.g. from kmg_ipc_open), d_cursors[n_parts] holds, per destination,
 * the first free element of THIS source's region and is advanced atomically.  With
 * count_only != 0 nothing is written: d_counts[0..n_parts) receives the number of keys per
 * destination and d_counts[n_parts] the number of windows that belong to the wide stream.
 * As in kmg_extract, val_bytes = 4 with ((pos_offset + n_bases) << 1) >= 2^32 is KMG_ERR_RANGE (the
 * payload would not hold the position); this holds for all three kmg_extract_scatter* calls. */
int kmg_extract_scatter(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k, int rc,
                        const uint8_t* d_lut256, int n_parts, void* const* d_dest_keys, void* const* d_dest_vals,
                        int key_bytes, int val_bytes, uint64_t pos_offset, uint64_t* d_cursors, uint64_t* d_counts,
                        int count_only, void* stream);
/* Single-launch variant: no count-only launch and no count matrix.  Every destination owns ONE
 * cursor word (d_cursor_ptrs[dst] points to it, peer-mapped, zeroed by its owner before the
 * exchange) that all sources advance with system-scope atomics over NVLink, so the regions of the
 * sources interleave tile by tile inside the receive buffer; afterwards the cursor is the number
 * of keys received.  `capacity` = elements every receive buffer holds: a reservation that would
 * pass it stores nothing and sets d_status[0] = 1 (the caller then repeats the exchange with exact
 * region sizes through kmg_extract_scatter); d_status[1] = 1 reports wide-stream windows. */
int kmg_extract_scatter_shared(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k,
                               int rc, const uint8_t* d_lut256, int n_parts, void* const* d_dest_keys,
                               void* const* d_dest_vals, int key_bytes, int val_bytes, uint64_t pos_offset,
                               uint64_t* const* d_cursor_ptrs, uint64_t capacity, uint32_t* d_status, void* stream);
/* kmg_extract_scatter with a guard for callers that launch before they know whether the receive
 * buffers still fit: a reservation that would pass `capacity` elements stores nothing and sets
 * d_status[0] = 1 (re-provision, repeat). */
int kmg_extract_scatter_checked(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k,
                                int rc, const uint8_t* d_lut256, int n_parts, void* const* d_dest_keys,
                                void* const* d_dest_vals, int key_bytes, int val_bytes, uint64_t pos_offset,
                                uint64_t* d_cursors, uint64_t capacity, uint32_t* d_status, void* stream);
/* What kmg_extract_scatter's count-only launch computes, from the 4-mer histogram of the BASES instead
 * of a second key-building pass (power-of-two n_parts <= 256, k >= 12): the top log2(n_parts) bits of a
 * key are its first bases.  d_counts[0..n_parts) keys per destination, d_counts[n_parts] windows of
 * the wide stream. */
size_t kmg_dest_counts_workspace_bytes(void);
int kmg_extract_dest_counts(const uint8_t* d_bases, uint64_t n_bases, uint64_t win_begin, uint64_t win_end, int k, int rc,
                            const uint8_t* d_lut256, int n_parts, uint64_t* d_counts, void* d_ws, size_t ws_bytes,
                            void* stream);
/* Device memory that other processes of the same box can map (CUDA IPC, 64-byte handle). */
int kmg_ipc_alloc(size_t bytes, void** d_ptr_out, uint8_t* h_handle64);
int kmg_ipc_open(const uint8_t* h_handle64, void** d_ptr_out);
int kmg_ipc_close(void* d_ptr);
int kmg_ipc_free(void* d_ptr);

/* ---- K6: text emission (join.py:262,284; seq.py:103-104,489-495) ----------------------
 * count lines "SEQ\tCOUNT\n"; *d_bytes_out = total bytes; d_text_out capacity must be
 * n*(k+12).  Symbols: narrow keys decode through "ACGT"/"ACGU" (rna != 0), wide keys
 * through the 16-letter table. */
size_t kmg_format_workspace_bytes(uint64_t n);
int kmg_format_counts(const void* d_keys, const uint32_t* d_counts, uint64_t n, int key_bytes, int k, int wide,
                      int rna, uint8_t* d_text_out, uint64_t* d_bytes_out, void* d_ws, size_t ws_bytes,
                      void* stream);
/* uniq records ">NAME:START-END:STRAND\nSEQ\n".  Record r spans
 * [d_rec_starts[r], d_rec_starts[r+1]-1) of the flat buffer (one separator byte after
 * each record); its name is d_names[d_name_offs[r] .. d_name_offs[r+1]).
 * d_text_out capacity must be n*(k+48+max_name_len). */
int kmg_format_uniq(const void* d_keys, const void* d_vals, uint64_t n, int key_bytes, int val_bytes, int k,
                    int wide, int rna, const uint64_t* d_rec_starts, uint32_t n_rec, const uint8_t* d_names,
                    const uint64_t* d_name_offs, uint8_t* d_text_out, uint64_t* d_bytes_out, void* d_ws,
                    size_t ws_bytes, void* stream);

/* ---- FASTA text -> flat base buffer (kmermaid/parsers.py:53-128; SURVEY.md §8f-2) --------------
 * d_raw holds the file's bytes.  Writes the flat layout the extraction expects (record bytes,
 * one '\n' after every record) to d_bases_out (capacity n_raw + 16), d_rec_starts[r] / [n_rec]
 * and d_hdr_begin[r] = raw offset of the first title character, for r < max_rec.
 * d_totals[0] = bytes written, [1] = number of records, [2] != 0 if the text holds bytes this
 * kernel does not implement (TAB/VT/FF/FS..US or non-ASCII: the host loader handles those). */
size_t kmg_fasta_workspace_bytes(uint64_t n_raw);
int kmg_fasta_flatten(const uint8_t* d_raw, uint64_t n_raw, uint8_t* d_bases_out, uint64_t* d_rec_starts,
                      uint64_t* d_hdr_begin, uint64_t max_rec, uint64_t* d_totals, void* d_ws, size_t ws_bytes,
                      void* stream);

/* ---- abundance vectors: `kmer count -m VEC_COUNT / VEC_COUNT_MASKED` (join.py:287-335, abundance.py:104-146)
 * Input: one stream's keys STABLY sorted with their payload (kmg_radix_sort / kmg_sort256 with vals), so that
 * equal keys are adjacent and their payloads ascend.  Every element writes, at out[strand][position - pos_base],
 * the size of its group of equal keys (masked = 0) or the number of group members that start in OTHER records
 * (masked = 1; elements of groups confined to one record write nothing).  The vectors are uint32 per flat
 * position, zeroed by the caller; positions nobody writes stay 0 like the reference's np.zeros.
 * d_rec_starts[n_rec + 1]: flat start of every record (the entry past the last one: one past the end).
 * *d_err (zeroed by the caller) becomes 2 if a count does not fit uint32. */
int kmg_abundance_scatter(const void* d_sorted_keys, const void* d_vals, uint64_t n, int key_bytes, int val_bytes,
                          const uint64_t* d_rec_starts, uint32_t n_rec, int masked, uint64_t pos_base,
                          uint32_t* d_out_plus, uint32_t* d_out_minus, uint32_t* d_err, void* stream);
/* Length of every record's vector (abundance.py:137-146: a vector ends at its last written entry), computed where
 * the vectors live.  d_plus / d_minus cover flat positions [0, n); record r covers [d_rec_starts[r],
 * d_rec_starts[r+1] - 1).  d_lengths_out[2r + s] (s = 0 '+', 1 '-') = last non-zero position of the record's
 * strand-s vector + 1 - d_rec_starts[r], or 0 if that vector is all zeros. */
int kmg_vector_extents(const uint32_t* d_plus, const uint32_t* d_minus, uint64_t n, const uint64_t* d_rec_starts,
                       uint32_t n_rec, uint64_t* d_lengths_out, void* stream);
/* The text of n vector entries, "%d\n" per entry (abundance.py:168-172; the "# k=K" header line is the caller's),
 * formatted with the tile prefix of kmg_format_counts.  *d_bytes_out = total bytes; d_text_out capacity must be
 * 11*n.  Workspace: kmg_format_workspace_bytes(n). */
int kmg_format_vector(const uint32_t* d_counts, uint64_t n, uint8_t* d_text_out, uint64_t* d_bytes_out, void* d_ws,
                      size_t ws_bytes, void* stream);

/* ---- merge ranks between the narrow and the wide stream -------------------------------
 * For two sorted, disjoint key lists, rank_of_wide[i] = number of narrow keys that sort
 * before wide key i in the reference's ASCII order (and vice versa), so that the merged
 * position of an element is its own index + its rank in the other list. */
int kmg_merge_ranks(const void* d_narrow_keys, uint64_t n_narrow, int narrow_key_bytes, const void* d_wide_keys,
                    uint64_t n_wide, int wide_key_bytes, int k, int rna, uint64_t* d_rank_of_narrow,
                    uint64_t* d_rank_of_wide, void* stream);
/* The same for 33 <= k <= 64: 16-byte narrow keys, 32-byte wide keys; d_tmp16 = n_wide 16-byte slots of scratch. */
int kmg_merge_ranks_wide(const void* d_narrow_keys, uint64_t n_narrow, const void* d_wide_keys, uint64_t n_wide, int k,
                         int rna, uint64_t* d_rank_of_narrow, uint64_t* d_rank_of_wide, void* d_tmp16, void* stream);

/* ---- the wide stream at 33 <= k <= 64: 256-bit keys (four little-endian 64-bit limbs, 4-bit codes) -----
 * kmermaid/seq.py:317-318 puts no bound on k for windows that hold N / IUPAC symbols.  kmg_extract
 * (wide = 1) emits them with key_bytes = 32; kmg_sort256 sorts them stably (batch.py:156-168) on bits
 * [0, end_bit) into d_keys_out / d_vals_out (two stable 128-bit sorts carrying the element index, then
 * one gather); kmg_rle_count, kmg_select_singletons, kmg_format_counts and kmg_format_uniq take
 * key_bytes = 32. */
size_t kmg_sort256_workspace_bytes(uint64_t n);
int kmg_sort256(const void* d_keys, void* d_keys_out, const void* d_vals, void* d_vals_out, uint64_t n, int val_bytes,
                int end_bit, void* d_ws, size_t ws_bytes, void* stream);


/* ---- whole-path calls with HOST buffers (what FastaBatcher.do + KJoiner.join do) ------
 * A context owns device scratch on one GPU and a private stream; calls are synchronous.
 * h_bases is the flat buffer (records joined by '\n'), narrow stream only: the call
 * fails with KMG_ERR_STATE if the input holds wide windows (use the stage API then).
 * count: h_keys_out/h_counts_out capacity `cap` entries; *h_n_out = number of distinct
 * k-mers.  uniq: singletons with payload. */
typedef struct kmg_ctx kmg_ctx;
int kmg_ctx_create(int device, kmg_ctx** out);
void kmg_ctx_destroy(kmg_ctx* ctx);
int kmg_count_host(kmg_ctx* ctx, const uint8_t* h_bases, uint64_t n_bases, int k, int rc, const uint8_t* h_lut256,
                   void* h_keys_out, uint32_t* h_counts_out, uint64_t cap, uint64_t* h_n_out);
int kmg_uniq_host(kmg_ctx* ctx, const uint8_t* h_bases, uint64_t n_bases, int k, int rc, const uint8_t* h_lut256,
                  void* h_keys_out, uint64_t* h_vals_out, uint64_t cap, uint64_t* h_n_out);

/* ---- tuning / introspection -----------------------------------------------------------
 * Options (process-wide; defaults in brackets):
 *   "hybrid" [1]           hybrid finish of key-only 8-byte sorts (0: plain LSD passes only)
 *   "hybrid_pb" [0]        force its prefix width to 16 or 24 bits (0: by n and key skew)
 *   "count_fused" [1]      kmg_sort_count: the local sort emits the (k-mer, count) table itself
 *   "local_tile" [7936]    target tile width of the local sort (positions)
 *   "time_passes" [0]      bracket every onesweep / local sort launch with CUDA events
 *   "count_limit" [0]      test hook: run lengths above it raise KMG_ERR_RANGE in the run-length stage
 *                          (0 = the real limit 2^32-1)
 * Stats of the calling thread's last call: "launches" (kernel launches since "reset_launches"),
 * "sort_passes", "hybrid_path" (0 plain passes, 1 hybrid, 2 hybrid + re-sorted ranges, 3 fell
 * back; kmg_sort_histo: 2 = fused histogram plus re-sorted ranges), "hybrid_irregular" (tiles), "hybrid_big_runs" (runs a whole block had to sort),
 * "n_out" / "ws_err" (result rows and status word the last kmg_sort_count / kmg_sort_uniq already
 * read back when its hybrid finish synchronised, -1 otherwise: a caller can then skip its own
 * read-back of *d_n_out and kmg_ws_status), and with time_passes: "sort_pass_ns" /
 * "sort_pass_count", "local_sort_ns" / "local_sort_count", "prepass_ns" / "prepass_count",
 * "scatter_ns" / "scatter_count" (device time of the timed launches: onesweep passes, the local
 * sort, and the fused pipeline's histogram pre-pass and extraction pass). */
int kmg_set_option(const char* name, int64_t value);
int64_t kmg_get_stat(const char* name);

#ifdef __cplusplus
}
#endif
#endif /* KMG_H_ */
