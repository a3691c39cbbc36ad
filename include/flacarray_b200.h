/*
 * flacarray_b200.h -- C ABI of the B200-native FLAC encode/decode hot path of flacarray.
 *
 * Two layers, both plain C (pointers and sizes, no torch / C++ types):
 *
 *  (1) Drop-in replacements for the ten functions the reference's Cython binding links against
 *      (reference: src/flacarray/libflacarray/flacarray.h:209-311, bound in libflacarray.pyx:21-110).
 *      Same names, same argument meaning, same ownership (encode_* returns a malloc()ed byte buffer
 *      the caller frees with free(), pyx:336-337), same ERROR_* bitmask (flacarray.h:20-40).  Buffers
 *      are HOST pointers; the library stages them through HBM.  The *_threaded variants and
 *      `use_threads` are accepted for signature compatibility and behave identically: the work is
 *      always parallel on the GPU (they replace the OpenMP loops compress.c:315-392 /
 *      decompress.c:227-310).
 *
 *  (2) Device-resident entry points (fab_*) for callers that keep arrays in HBM (the Python host
 *      layer flacarray_b200 uses these through ctypes with torch-owned device memory).  All bulk
 *      buffers are DEVICE pointers, `stream` is a cudaStream_t passed as void*.
 *
 * There is no CPU fallback: every function returns FAB_ERROR_CUDA when no usable sm_100 device exists.
 */
#ifndef FLACARRAY_B200_H
#define FLACARRAY_B200_H

#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Error bits: identical values to the reference's flacarray.h:20-40. */
#define ERROR_NONE 0
#define ERROR_ALLOC (1 << 0)
#define ERROR_INVALID_LEVEL (1 << 1)
#define ERROR_ZERO_NSTREAM (1 << 2)
#define ERROR_ZERO_STREAMSIZE (1 << 3)
#define ERROR_ENCODE_SET_COMP_LEVEL (1 << 4)
#define ERROR_ENCODE_SET_BLOCK_SIZE (1 << 5)
#define ERROR_ENCODE_SET_CHANNELS (1 << 6)
#define ERROR_ENCODE_SET_BPS (1 << 7)
#define ERROR_ENCODE_INIT (1 << 8)
#define ERROR_ENCODE_PROCESS (1 << 9)
#define ERROR_ENCODE_FINISH (1 << 10)
#define ERROR_ENCODE_COLLECT (1 << 11)
#define ERROR_DECODE_READ_ZEROBUF (1 << 12)
#define ERROR_DECODE_INIT (1 << 13)
#define ERROR_DECODE_PROCESS (1 << 14)
#define ERROR_DECODE_FINISH (1 << 15)
#define ERROR_DECODE_STREAMSIZE (1 << 16)
#define ERROR_DECODE_SAMPLE_RANGE (1 << 17)
#define ERROR_DECODE_SEEK (1 << 18)
#define ERROR_CONVERT_TYPE (1 << 19)
/* Extensions (bits the reference never sets). */
#define FAB_ERROR_CUDA (1 << 20)  /* CUDA runtime failure: no device, launch error, out of memory */
#define FAB_ERROR_NAN (1 << 21)   /* float input holds a NaN (reference raises in utils.py:268) */

/* ------------------------------------------------------------------------------------------------
 * (1) Reference-compatible host-buffer entry points
 *
 * Same signatures, ownership (`*bytes` is malloc()ed, the caller frees it) and return codes as the
 * reference.  Like the reference they are re-entrant: every call leases one of a few host slots (context +
 * staging buffers, FLACARRAY_B200_HOST_SLOTS, default 4), so concurrent callers run side by side on their own
 * CUDA streams; callers beyond the slot count wait for a slot.  Arrays of 64 MB or more move through
 * persistent pinned staging buffers in 128 MB chunks of whole streams (host copies on several threads,
 * H2D / kernels / D2H on three CUDA streams); FLACARRAY_B200_NO_PIPE=1 selects the plain
 * cudaMemcpy path, FLACARRAY_B200_PIPE_DEBUG=1 prints the phase times of the pipelined encode.
 * ---------------------------------------------------------------------------------------------- */

/* flacarray.h:209-217 (compress.c:440-459) */
int encode_i32(int32_t* const data, int64_t n_stream, int64_t stream_size, uint32_t level, int64_t* n_bytes,
               int64_t* starts, unsigned char** bytes);
/* flacarray.h:219-227 (compress.c:461-480) */
int encode_i32_threaded(int32_t* const data, int64_t n_stream, int64_t stream_size, uint32_t level,
                        int64_t* n_bytes, int64_t* starts, unsigned char** bytes);
/* flacarray.h:229-237 (compress.c:482-509): int64 as 2 channels, ch0 = low word, ch1 = high word */
int encode_i64(int64_t* const data, int64_t n_stream, int64_t stream_size, uint32_t level, int64_t* n_bytes,
               int64_t* starts, unsigned char** bytes);
/* flacarray.h:239-247 (compress.c:511-540) */
int encode_i64_threaded(int64_t* const data, int64_t n_stream, int64_t stream_size, uint32_t level,
                        int64_t* n_bytes, int64_t* starts, unsigned char** bytes);
/* flacarray.h:249-259 (decompress.c:318-341).  first/last < 0 => whole stream; else [first, last). */
int decode_i32(unsigned char* const bytes, int64_t* const starts, int64_t* const nbytes, int64_t n_stream,
               int64_t stream_size, int64_t first_sample, int64_t last_sample, int32_t* data, bool use_threads);
/* flacarray.h:261-271 (decompress.c:343-375) */
int decode_i64(unsigned char* const bytes, int64_t* const starts, int64_t* const nbytes, int64_t n_stream,
               int64_t stream_size, int64_t first_sample, int64_t last_sample, int64_t* data, bool use_threads);
/* flacarray.h:275-283 (utils.c:160-243).  quanta == NULL => derive from the data range. */
int float32_to_int32(float const* input, int64_t n_stream, int64_t stream_size, float const* quanta,
                     int32_t* output, float* offsets, float* gains);
/* flacarray.h:285-293 (utils.c:245-328) */
int float64_to_int64(double const* input, int64_t n_stream, int64_t stream_size, double const* quanta,
                     int64_t* output, double* offsets, double* gains);
/* flacarray.h:295-302 (utils.c:330-348) */
void int64_to_float64(int64_t const* input, int64_t n_stream, int64_t stream_size, double const* offsets,
                      double const* gains, double* output);
/* flacarray.h:304-311 (utils.c:350-368) */
void int32_to_float32(int32_t const* input, int64_t n_stream, int64_t stream_size, float const* offsets,
                      float const* gains, float* output);

/* ------------------------------------------------------------------------------------------------
 * (2) Device-resident entry points
 * ---------------------------------------------------------------------------------------------- */

typedef struct fab_ctx fab_ctx; /* per (thread, device) context: tables + grow-only scratch */

enum { FAB_I32 = 0, FAB_I64 = 1, FAB_F32 = 2, FAB_F64 = 3 };

/* Create / destroy a context on the CURRENT CUDA device.  Returns an ERROR_* mask. */
int fab_create(fab_ctx** ctx);
void fab_destroy(fab_ctx* ctx);
/* Text of the last CUDA error seen by this context (never NULL). */
const char* fab_last_error(const fab_ctx* ctx);
/* Number of kernels this context has launched so far (bench.py's gpu_launches). */
int64_t fab_launch_count(const fab_ctx* ctx);

/* Upper bound of the compressed size (bytes) for n_stream streams of stream_size samples. */
int64_t fab_encode_bound(int64_t n_stream, int64_t stream_size, int dtype, uint32_t level);

/*
 * Workspace.  fab_encode / fab_decode / fab_float_to_int / fab_stream_std keep their intermediates (per-frame
 * statistics and plans, frame slots, frame-offset tables, min/max partials) in one device block.  By default the
 * context owns a grow-only block; growing it waits for this context's own streams only.  A caller that wants no
 * allocation inside the calls sizes the block with fab_*_workspace_bytes (0 = invalid arguments) and hands it
 * over with fab_set_workspace (256-byte aligned device memory; NULL returns to the context-owned block).  With a
 * caller-supplied workspace a call that needs more than was supplied fails with ERROR_ALLOC and says how much in
 * fab_last_error -- it never allocates.  (The reference has no equivalent: libFLAC allocates per encoder object,
 * compress.c:184-200.)
 */
int64_t fab_encode_workspace_bytes(int64_t n_stream, int64_t stream_size, int dtype, uint32_t level);
int64_t fab_decode_workspace_bytes(int64_t n_stream, int64_t stream_size, int blocksize_hint);
int fab_set_workspace(fab_ctx* ctx, void* d_workspace, int64_t bytes);

/*
 * Encode (replaces compress.c:133-435 + the libFLAC encoder; for float input also utils.c:160-328
 * fused in front).  d_data: [n_stream][stream_size] of `dtype`.  For FAB_F32/FAB_F64, d_quanta is
 * NULL (auto) or [n_stream], and d_offsets/d_gains [n_stream] receive the per-stream conversion.
 * d_out (capacity out_capacity bytes) receives the concatenated streams; d_starts/d_nbytes
 * [n_stream] int64 the bookkeeping of compress.c:402-411 / pyx:331-332; d_total one int64.
 * Asynchronous on `stream`; call fab_finish() to synchronise and collect the error mask.
 */
int fab_encode(fab_ctx* ctx, const void* d_data, int dtype, int64_t n_stream, int64_t stream_size, uint32_t level,
               const void* d_quanta, void* d_offsets, void* d_gains, unsigned char* d_out, int64_t out_capacity,
               int64_t* d_starts, int64_t* d_nbytes, int64_t* d_total, void* stream);

/*
 * Decode (replaces decompress.c:194-313 + the libFLAC decoder; with d_offsets/d_gains != NULL also
 * the int->float restore utils.c:330-368 fused behind).  d_starts/d_nbytes: [n_stream] windows into
 * d_bytes (any order, e.g. after a keep mask).  first/last as in decode_i32.  d_out:
 * [n_stream][n_decode] of int32/int64 (is_int64) or float32/float64 when offsets/gains are given.
 * max_nbytes: max over d_nbytes (host knows it; <= 0 lets the library compute it with one sync).
 * blocksize_hint: nominal FLAC blocksize of the streams (0 = 4096); only sizes the frame table.
 */
int fab_decode(fab_ctx* ctx, const unsigned char* d_bytes, const int64_t* d_starts, const int64_t* d_nbytes,
               int64_t n_stream, int64_t stream_size, int is_int64, int64_t first_sample, int64_t last_sample,
               void* d_out, const void* d_offsets, const void* d_gains, int64_t max_nbytes, int blocksize_hint,
               void* stream);

/*
 * fab_decode with per-stream fault isolation (no reference equivalent: the reference fails the whole call).
 * d_status[n_stream] (int32, device) receives 0 or the ERROR_DECODE_INIT / ERROR_DECODE_PROCESS bit of each
 * stream; the output rows of failed streams are filled (0 for integer output, quiet NaN for float output);
 * the mask fab_finish returns carries only call-level errors (CUDA, ALLOC, SAMPLE_RANGE, ...).  Only frames
 * overlapping [first, last) are examined.  Same launches as fab_decode plus one fill kernel per 65535 streams.
 * A NULL d_status makes the call a plain fab_decode.  Workspace: fab_decode_workspace_bytes.
 */
int fab_decode_isolated(fab_ctx* ctx, const unsigned char* d_bytes, const int64_t* d_starts, const int64_t* d_nbytes,
                        int64_t n_stream, int64_t stream_size, int is_int64, int64_t first_sample, int64_t last_sample,
                        void* d_out, const void* d_offsets, const void* d_gains, int64_t max_nbytes, int blocksize_hint,
                        int32_t* d_status, void* stream);
/*
 * Decode every frame of every stream and check it (CRC-8/16, syntax, frame chain, sample count) without writing
 * samples; d_status as above.  A stream is accepted exactly when a full fab_decode of it succeeds (the same
 * decoder stages, with the tile decoder's stores and the restore left out), so an archive can be checked after a
 * transfer without room for its samples.  d_status must not be NULL (ERROR_ALLOC otherwise).
 * Workspace: fab_decode_workspace_bytes.
 */
int fab_verify(fab_ctx* ctx, const unsigned char* d_bytes, const int64_t* d_starts, const int64_t* d_nbytes, int64_t n_stream,
               int64_t stream_size, int is_int64, int64_t max_nbytes, int blocksize_hint, int32_t* d_status, void* stream);

/*
 * Decode many sample windows, each of its own stream and range, in one call (no reference equivalent).
 * Window w = (d_win_stream[w], d_win_first[w], d_win_last[w], d_win_out[w]) decodes samples [first, last)
 * of stream slot d_win_stream[w] in [0, n_stream) to d_out[d_win_out[w] ...] (counted in samples of the
 * output type: packed, a row pitch, ... -- output regions must not overlap).  Windows may be empty
 * (first == last), overlap, repeat and come in any order.  A record with the slot out of range, first < 0,
 * last > stream_size or first > last sets ERROR_DECODE_SAMPLE_RANGE in the error mask and is skipped.
 * Only the frames the windows touch are decoded; metadata, frame tables and the sync scan of foreign
 * streams run once per stream slot, so give each distinct stream one slot.  Offsets and gains are indexed
 * by slot and restore like fab_decode.  All window arrays are device memory (int64).  One host round trip
 * per call sizes the grids.  The workspace (fab_decode_windows_workspace_bytes; total_items, the number of
 * (window, frame) items, does not enter the present layout) grows with n_stream x frames + n_win.
 */
int fab_decode_windows(fab_ctx* ctx, const unsigned char* d_bytes, const int64_t* d_starts, const int64_t* d_nbytes,
                       int64_t n_stream, int64_t stream_size, int is_int64, const int64_t* d_win_stream,
                       const int64_t* d_win_first, const int64_t* d_win_last, const int64_t* d_win_out, int64_t n_win,
                       void* d_out, const void* d_offsets, const void* d_gains, int64_t max_nbytes, int blocksize_hint,
                       void* stream);
int64_t fab_decode_windows_workspace_bytes(int64_t n_stream, int64_t stream_size, int64_t n_win, int64_t total_items,
                                           int blocksize_hint);

/*
 * Per-row, per-bin statistics of decoded integer rows (no reference equivalent): the reduction behind
 * FlacArray.stats().  d_rows: [n_rows][n] int32 (is_int64 = 0) or int64, e.g. the output of fab_decode without
 * offsets / gains, aligned to its element size.  Each row is cut into bins of `bin` samples (bin = 0: one bin of n
 * samples; a bin longer than n is one bin; the last bin may be shorter), nbins = ceil(n / bin); a bin longer than
 * 2^32 - 1 samples is rejected.  Per (row, bin), row-major [n_rows][nbins]:
 *   d_count  int64   the number of samples;
 *   d_min    / d_max  the extreme values, in the array's type: int32 / int64, or float32 / float64 when d_offsets and
 *            d_gains ([n_rows] float32 / float64, as fab_decode takes them; both NULL for integer output) are given --
 *            then they are the restored extremes, bit-equal to the min / max of the restored samples;
 *   d_mean / d_std    double: the mean and population standard deviation (ddof = 0).  The sums S = sum x and
 *            Q = sum x^2 are exact integers; mean = dbl(S) / n and std = sqrt(dbl(n*Q - S^2)) / n with dbl() the
 *            round-to-nearest-even conversion and plain IEEE double operations after it, so results do not depend on how
 *            the rows were grouped into calls.  With offsets / gains: mean = off + coeff * mean, std = |coeff| * std, with
 *            the restore's coeff = 1 / gain in the storage type, widened to double.
 * d_status ([n_rows] int32, may be NULL): rows with a non-zero status get count 0, NaN mean / std and min / max NaN
 * (float output) or 0 (integer output).  Bad arguments return error bits (ERROR_ZERO_NSTREAM, ERROR_ZERO_STREAMSIZE,
 * ERROR_DECODE_SAMPLE_RANGE for a negative or too long bin, ERROR_CONVERT_TYPE for offsets without gains or a
 * misaligned d_rows, ERROR_ALLOC for NULL arrays) and launch nothing.  Workspace: fab_row_stats_workspace_bytes
 * (0 when none is needed, -1 for invalid arguments); a caller-supplied workspace that is too small fails with
 * ERROR_ALLOC.  One or two launches per 65535 rows.
 */
int fab_row_stats(fab_ctx* ctx, const void* d_rows, int is_int64, int64_t n_rows, int64_t n, int64_t bin,
                  const void* d_offsets, const void* d_gains, const int32_t* d_status, int64_t* d_count, void* d_min,
                  void* d_max, double* d_mean, double* d_std, void* stream);
int64_t fab_row_stats_workspace_bytes(int64_t n_rows, int64_t n, int64_t bin, int is_int64);

/*
 * Per-sample weighted sums across decoded integer rows (no reference equivalent): the reduction behind
 * FlacArray.combine() (common modes, pair differences, group averages).  d_rows: [n_rows][n] int32 (is_int64 = 0) or
 * int64, e.g. the output of fab_decode without offsets / gains, aligned to its element size.  Rows come as n_seg
 * segments: segment s is rows [d_seg[s], d_seg[s + 1]) and adds into row d_seg_out[s] of d_out ([n_out][n] double).
 * For every sample i of segment s, in plain IEEE double (multiply and add each rounded, never an FMA):
 *     acc = d_out[d_seg_out[s]][i]
 *     for k = d_seg[s] .. d_seg[s + 1] - 1 with d_status[k] == 0:   acc = acc + d_weights[k] * x_k[i]
 *     d_out[d_seg_out[s]][i] = acc
 * x_k[i] is the integer (int64 converts with round to nearest even) or, when d_offsets and d_gains ([n_rows] float32 /
 * float64, as fab_decode takes them; both NULL for integer rows) are given, the value fab_decode's restore produces in
 * the array's type, widened to double.  So a zero-filled d_out gives the fold +0.0 + w x + ... in row order, and a
 * segment continues from what an earlier call stored in its output row: a group of rows split over several calls gives
 * the same bits as one call.  d_weights: [n_rows] double.  d_status ([n_rows] int32, may be NULL): rows with a non-zero
 * status are skipped.  d_seg ([n_seg + 1]) and d_seg_out ([n_seg]) are device int64 and must satisfy
 * 0 <= d_seg[s] <= d_seg[s + 1] <= n_rows, 0 <= d_seg_out[s] < n_out and d_seg_out strictly increasing, so that no two
 * segments write the same output row; they are checked on the device, and a record that breaks a rule sets
 * ERROR_DECODE_SAMPLE_RANGE in the mask fab_finish returns and its segment writes nothing (the output of such a call
 * is not meaningful).  Bad arguments return error bits (ERROR_ZERO_NSTREAM for n_rows, n_seg or n_out <= 0,
 * ERROR_ZERO_STREAMSIZE for n <= 0, ERROR_ALLOC for NULL arrays, ERROR_CONVERT_TYPE for offsets without gains or a
 * misaligned array) and launch nothing.  No workspace.  One launch per 65535 segments.
 */
int fab_combine_rows(fab_ctx* ctx, const void* d_rows, int is_int64, int64_t n_rows, int64_t n, const void* d_offsets,
                     const void* d_gains, const int32_t* d_status, const double* d_weights, const int64_t* d_seg,
                     const int64_t* d_seg_out, int64_t n_seg, double* d_out, int64_t n_out, void* stream);

/*
 * Ranges of out-of-threshold samples of decoded integer rows (no reference equivalent): the search behind
 * FlacArray.flag_ranges() (glitches, samples at the ADC rails, excursions beyond N sigma).  d_rows: [n_rows][n] int32
 * (is_int64 = 0) or int64, e.g. the output of fab_decode without offsets / gains, aligned to its element size.  Sample i
 * of row k is flagged iff its value v is below the row's low threshold or above its high one (a value equal to a
 * threshold is not flagged):
 *   integer rows (d_offsets = d_gains = NULL): d_lo / d_hi are int64 [n_rows] bounds L / H, and x is flagged iff
 *            x < L or x > H (L > H flags every sample);
 *   float rows (d_offsets, d_gains [n_rows] float32 / float64, as fab_decode takes them): d_lo / d_hi are float64
 *            [n_rows] thresholds (-inf / +inf leave a side open), and v is fab_decode's restore of x, widened to double.
 *            The restore is monotone in x, so each row's kept samples are one integer interval, found once per row by
 *            binary search; offsets and coefficients must be finite.
 * Flagged samples j1 < j2 that follow each other are in one range iff j2 - j1 <= 2 * pad + 1 (pad >= 0; larger than n
 * is allowed); a range with first and last flagged samples js and je is [max(js - pad, 0), min(je + pad + 1, n)).
 *
 * Two calls on the same rows, status, pad and workspace, the second after the caller has read the counts:
 *   fab_flag_count  writes d_nflag[k] (int64: flagged samples of row k before widening, -1 for a row with a non-zero
 *                   d_status) and d_nrange[k] (int64: its ranges, 0 for such a row);
 *   fab_flag_write  writes the ranges of row k, in order, to slots d_base[k] .. d_base[k] + d_nrange[k] - 1 of
 *                   d_first_out / d_last_out (int64), as sample indices plus sample0 (the index of the rows' sample 0 in
 *                   their streams).  d_base: int64 [n_rows].
 * The workspace d_work (work_bytes >= fab_flag_ranges_workspace_bytes(n_rows, n, is_int64), 16-byte aligned) carries a
 * per-row bitmask of the flagged samples and per-piece summaries from the first call to the second, so it is supplied
 * by the caller and not taken from the context; fab_flag_ranges_workspace_bytes returns -1 for invalid arguments.
 * d_status ([n_rows] int32, may be NULL): rows with a non-zero status are skipped.  Bad arguments return error bits
 * (ERROR_ZERO_NSTREAM, ERROR_ZERO_STREAMSIZE, ERROR_DECODE_SAMPLE_RANGE for a negative pad, ERROR_CONVERT_TYPE for
 * offsets without gains or a misaligned array, ERROR_ALLOC for NULL arrays or a workspace that is too small) and launch
 * nothing.  fab_flag_count: one launch per 65535 rows and one more; fab_flag_write: one launch per 65535 rows.
 */
int64_t fab_flag_ranges_workspace_bytes(int64_t n_rows, int64_t n, int is_int64);
int fab_flag_count(fab_ctx* ctx, const void* d_rows, int is_int64, int64_t n_rows, int64_t n, const void* d_lo,
                   const void* d_hi, const void* d_offsets, const void* d_gains, const int32_t* d_status, int64_t pad,
                   void* d_work, int64_t work_bytes, int64_t* d_nflag, int64_t* d_nrange, void* stream);
int fab_flag_write(fab_ctx* ctx, const void* d_rows, int is_int64, int64_t n_rows, int64_t n, const int32_t* d_status,
                   int64_t pad, void* d_work, int64_t work_bytes, const int64_t* d_base, int64_t sample0,
                   int64_t* d_first_out, int64_t* d_last_out, void* stream);

/*
 * Projections of decoded integer rows onto templates (no reference equivalent): the reduction behind
 * FlacArray.project() (common-mode couplings, baseline coefficients, lock-in amplitudes).  d_rows: [n_rows][n] int32
 * (is_int64 = 0) or int64, e.g. the output of fab_decode without offsets / gains, aligned to its element size.
 * d_templates: [n_tmpl][n] double.  d_out: [n_rows][n_tmpl] double.  With v_k[i] the integer (int64 converts with round
 * to nearest even) or, when d_offsets and d_gains ([n_rows] float32 / float64, as fab_decode takes them; both NULL for
 * integer rows) are given, the value fab_decode's restore produces in the array's type, widened to double, the samples
 * are cut into pieces of FAB_PROJECT_PIECE counted from sample 0 (the last one may be shorter) and, in plain IEEE double
 * (multiply and add each rounded, never an FMA):
 *     for each piece j:  p_j = +0.0;  for i in piece j ascending:  p_j = p_j + d_templates[t][i] * v_k[i]
 *     d_out[k][t] = +0.0;  for j ascending:  d_out[k][t] = d_out[k][t] + p_j
 * so the result depends on the piece length only, not on how rows are grouped into calls.  d_status ([n_rows] int32,
 * may be NULL): rows with a non-zero status get NaN.  Bad arguments return error bits (ERROR_ZERO_NSTREAM for n_rows or
 * n_tmpl <= 0, ERROR_ZERO_STREAMSIZE for n <= 0, ERROR_ALLOC for NULL arrays, ERROR_CONVERT_TYPE for offsets without
 * gains or a misaligned array) and launch nothing.  Workspace: fab_project_rows_workspace_bytes (one double per row,
 * template and piece; -1 for invalid arguments); a caller-supplied workspace that is too small fails with ERROR_ALLOC.
 * One launch per 65535 pieces and one more.
 */
#define FAB_PROJECT_PIECE 4096
int64_t fab_project_rows_workspace_bytes(int64_t n_rows, int64_t n, int64_t n_tmpl);
int fab_project_rows(fab_ctx* ctx, const void* d_rows, int is_int64, int64_t n_rows, int64_t n, const void* d_offsets,
                     const void* d_gains, const int32_t* d_status, const double* d_templates, int64_t n_tmpl,
                     double* d_out, void* stream);

/*
 * Per-stream population standard deviation of float32 / float64 streams, in the input's type: the device side of
 * `precision` -> quanta (replaces np.std(data, axis=-1) in utils.py:282-296).  One read of the input, moments
 * accumulated in double precision; differs from numpy's pairwise single-precision sum by rounding only.
 * d_std: [n_stream] of `dtype`.
 */
int fab_stream_std(fab_ctx* ctx, const void* d_input, int dtype, int64_t n_stream, int64_t stream_size, void* d_std,
                   void* stream);

/* utils.c:160-328 on device buffers (dtype FAB_F32 -> int32, FAB_F64 -> int64). */
int fab_float_to_int(fab_ctx* ctx, const void* d_input, int dtype, int64_t n_stream, int64_t stream_size,
                     const void* d_quanta, void* d_output, void* d_offsets, void* d_gains, void* stream);
/* utils.c:330-368 on device buffers (dtype FAB_I32 -> float32, FAB_I64 -> float64). */
int fab_int_to_float(fab_ctx* ctx, const void* d_input, int dtype, int64_t n_stream, int64_t stream_size,
                     const void* d_offsets, const void* d_gains, void* d_output, void* stream);

/* Optional kernel timing for roofline reports: when enabled, CUDA events are recorded on the launching
 * stream around the encoder kernel sequence of one fab_encode call (which = 0: k_enc_analyze,
 * k_enc_design, k_encode, k_enc_scan, k_enc_compact over all batches) and around the decoder kernels of
 * one fab_decode call (which = 1: k_dec_tile, k_dec_crc).  fab_profile_ms returns the accumulated
 * milliseconds and (through *count) the number of calls. */
void fab_profile(fab_ctx* ctx, int enable);
double fab_profile_ms(fab_ctx* ctx, int which, int64_t* count);

/* Synchronise `stream`, return (and clear) the device-side error mask accumulated since the last call. */
int fab_finish(fab_ctx* ctx, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FLACARRAY_B200_H */
