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
