// fa_api.cu -- CUDA kernels (sm_100a) and the C ABI of libflacarray_b200.so.
//
// See include/flacarray_b200.h for the contract.  This translation unit is the whole product
// library: kernels are thin __global__ wrappers around the bodies in fa_encode.h / fa_decode.h /
// fa_quant.h.  No CPU fallback exists: without a CUDA device every entry point fails with
// FAB_ERROR_CUDA.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <thread>
#include <string>
#include <vector>

#include "../../include/flacarray_b200.h"
#include "fa_combine.h"
#include "fa_decode.h"
#include "fa_decode_tile.h"
#include "fa_encode.h"
#include "fa_encode_fixed.h"
#include "fa_quant.h"
#include "fa_stats.h"

using namespace fa;

// =================================================================================================
// Kernels
// =================================================================================================

// persistent CTAs: each loops over (stream, frame) units of the batch; H = predictor history kept in registers
#ifndef FAB_ENC_CTAS
#define FAB_ENC_CTAS 6
#endif
template <int H>
__global__ void __launch_bounds__(kEncThreads, FAB_ENC_CTAS) k_encode(const EncParams P) {
    extern __shared__ __align__(128) unsigned char smem[];
    encode_frames_cta<H, true>(P, smem);
}
// the frames that are not full 4096-sample frames (see k_enc_analyze_short)
template <int H>
__global__ void __launch_bounds__(kEncThreads, 4) k_encode_short(const EncParams P, uint32_t first, uint32_t stride) {
    extern __shared__ __align__(128) unsigned char smem[];
    encode_frames_cta<H, false>(P, smem, first, stride);
}

// sample statistics, fixed-predictor error sums and windowed autocorrelation of every (frame, channel)
// (persistent CTAs: the thread's slice of the tukey window is loaded into shared memory once)
#ifndef FAB_AN_CTAS
#define FAB_AN_CTAS 5     // (96 registers: no spills in the autocorrelation loop; 5 CTAs beat 6 with spills and 6 with 4-sample trips)
#endif
template <int H>
__global__ void __launch_bounds__(kEncThreads, FAB_AN_CTAS) k_enc_analyze(const EncParams P) {
    __shared__ AnShared sh;
    analyze_fill_window(P, &sh);
    __syncthreads();
    for (uint32_t g = P.g_begin + blockIdx.x; g < P.g_end; g += gridDim.x) {
#ifdef FAB_AN_PREFETCH    // (measured: pulling the next frame into the L2 costs 0.5 ms per 10^9 samples instead of saving any)
        if (threadIdx.x == 0 && (uint64_t)g + gridDim.x < P.g_end) analyze_prefetch(P, g + gridDim.x);
#endif
        analyze_frame_cta<H, true>(P, g, &sh);
    }
}
// ... and of the frames that are not full 4096-sample frames: the last frame of every stream (CTA i takes the
// i-th such frame of the batch), or every frame of a blocksize-1152 level
template <int H>
__global__ void __launch_bounds__(kEncThreads) k_enc_analyze_short(const EncParams P, uint32_t first, uint32_t stride) {
    __shared__ AnShared sh;
    for (uint64_t g = (uint64_t)first + (uint64_t)blockIdx.x * stride; g < P.g_end; g += (uint64_t)gridDim.x * stride)
        analyze_frame_cta<H, false>(P, (uint32_t)g, &sh);
}

// levels 0..2: full blocksize-1152 frames, one warp each (fa_encode_fixed.h); what it declines keeps fsize == 0
__global__ void __launch_bounds__(kFxWarps * 32, 7) k_enc_fixed(const EncParams P) {
    __shared__ FxShared ws[kFxWarps];
    const uint64_t g = (uint64_t)P.g_begin + (uint64_t)blockIdx.x * kFxWarps + (threadIdx.x >> 5);
    if (g >= P.g_end) return;
    fixed_frame_warp(P, (uint32_t)g, &ws[threadIdx.x >> 5]);
}

// predictor design: one thread per (frame, channel)
__global__ void __launch_bounds__(128) k_enc_design(const EncParams P, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) design_frame(P, i);
}

// frame sizes of a batch -> inclusive byte prefixes (one CTA)
__global__ void __launch_bounds__(kScanThreads) k_enc_scan(const EncParams P) {
    __shared__ unsigned long long part[kScanThreads / 32 + 1];
    scan_batch_cta(P, part);
}

// frames of a batch from their slots to their final byte offsets, CRC-16 appended (CTAs stride over the frames)
#ifndef FAB_COMPACT_MINB
#define FAB_COMPACT_MINB 16     // (32 registers: 16 CTAs = 64 warps per SM hide the row loads; 12 and 8 CTAs measured slower)
#endif
__global__ void __launch_bounds__(128, FAB_COMPACT_MINB) k_enc_compact(const EncParams P) {
    __shared__ CompactShared cs;
    const uint32_t n = P.g_end - P.g_begin;
    // (size and byte prefix of the CTA's next frame are loaded one frame ahead: the frame's first row would otherwise
    // wait for two dependent trips to HBM)
    uint32_t i = blockIdx.x;
    uint32_t len = 0;
    unsigned long long end = 0;
    if (i < n) { len = P.fsize[i]; end = P.desc[P.g_begin + i]; }
    while (i < n) {
        const uint32_t inext = i + gridDim.x;
        uint32_t len_n = 0;
        unsigned long long end_n = 0;
        if (inext < n) { len_n = P.fsize[inext]; end_n = P.desc[P.g_begin + inext]; }
        compact_frame_cta(P, i, &cs, len, end);
        __syncthreads();      // cs is reused by the next frame
        i = inext; len = len_n; end = end_n;
    }
}

// stream headers, frame-size tables, stream_starts / stream_nbytes / total from the byte prefixes
__global__ void k_enc_finalize(const EncParams P, long long* __restrict__ nbytes, long long* __restrict__ total) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < P.n_stream * P.nframes) finalize_entry(P, i / P.nframes, (int)(i % P.nframes), nbytes, total);
}

// ---- float -> int: per-stream min/max (utils.c:182-193 / :267-278), chunked over the stream ------
#ifndef FAB_ENC_BATCH_LOG2
#define FAB_ENC_BATCH_LOG2 30
#endif
constexpr int64_t kEncBatchBytes = 1ll << FAB_ENC_BATCH_LOG2;   // slot scratch of one batch of encoder launches (two such buffers alternate)
constexpr int kMmThreads = 256;
constexpr int kMmChunk = 32768;  // elements per CTA

template <typename T>
__global__ void __launch_bounds__(kMmThreads) k_minmax(const T* __restrict__ data, int64_t stream_size, int nchunk,
                                                       T* __restrict__ pmin, T* __restrict__ pmax, int* __restrict__ err) {
    const int64_t s = blockIdx.y;
    const int c = blockIdx.x;
    const int64_t lo = (int64_t)c * kMmChunk;
    const int64_t hi = lo + kMmChunk < stream_size ? lo + kMmChunk : stream_size;
    const T* p = data + s * stream_size;
    T mn = p[lo], mx = p[lo];
    bool nan = false;
    for (int64_t i = lo + threadIdx.x; i < hi; i += kMmThreads) {
        T v = p[i];
        nan |= (v != v);
        mn = v < mn ? v : mn;
        mx = v > mx ? v : mx;
    }
    __shared__ T smn[kMmThreads / 32], smx[kMmThreads / 32];
    for (int m = 16; m >= 1; m >>= 1) {
        T a = __shfl_xor_sync(0xffffffffu, mn, m), b = __shfl_xor_sync(0xffffffffu, mx, m);
        mn = a < mn ? a : mn;
        mx = b > mx ? b : mx;
    }
    if (__syncthreads_or(nan) && threadIdx.x == 0) atomicOr(err, FAB_ERROR_NAN);
    if ((threadIdx.x & 31) == 0) { smn[threadIdx.x >> 5] = mn; smx[threadIdx.x >> 5] = mx; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < kMmThreads / 32; ++w) {
            mn = smn[w] < mn ? smn[w] : mn;
            mx = smx[w] > mx ? smx[w] : mx;
        }
        pmin[s * nchunk + c] = mn;
        pmax[s * nchunk + c] = mx;
    }
}

template <typename T>
__global__ void k_quant_params(const T* __restrict__ pmin, const T* __restrict__ pmax, int nchunk, int64_t n_stream,
                               const T* __restrict__ quanta, T* __restrict__ offsets, T* __restrict__ gains) {
    int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_stream) return;
    T mn = pmin[s * nchunk], mx = pmax[s * nchunk];
    for (int c = 1; c < nchunk; ++c) {
        T a = pmin[s * nchunk + c], b = pmax[s * nchunk + c];
        mn = a < mn ? a : mn;
        mx = b > mx ? b : mx;
    }
    if constexpr (sizeof(T) == 4) quant_params_f32(mn, mx, quanta != nullptr, quanta ? quanta[s] : 0.f, &offsets[s], &gains[s]);
    else quant_params_f64(mn, mx, quanta != nullptr, quanta ? quanta[s] : 0., &offsets[s], &gains[s]);
}

// ---- `precision` -> quanta: per-stream population standard deviation (reference utils.py:282-296 calls
// np.std(data, axis=-1)).  One read of the input: every CTA reduces a chunk to (mean, M2 = sum (x - mean)^2) in
// double precision around a local shift (the chunk's first element), one thread per stream then merges the chunk
// moments in chunk order (Chan et al.) -> sqrt(M2 / n), rounded to the storage type.
template <typename T>
__global__ void __launch_bounds__(kMmThreads) k_moments(const T* __restrict__ data, int64_t stream_size, int nchunk,
                                                        double* __restrict__ pmean, double* __restrict__ pm2) {
    const int64_t s = blockIdx.y;
    const int c = blockIdx.x;
    const int64_t lo = (int64_t)c * kMmChunk;
    const int64_t hi = lo + kMmChunk < stream_size ? lo + kMmChunk : stream_size;
    const T* p = data + s * stream_size;
    const double K = (double)p[lo];
    double s1 = 0.0, s2 = 0.0;
    for (int64_t i = lo + threadIdx.x; i < hi; i += kMmThreads) {
        const double d = (double)p[i] - K;
        s1 += d;
        s2 = fma(d, d, s2);
    }
    __shared__ double sh1[kMmThreads / 32], sh2[kMmThreads / 32];
    for (int m = 16; m >= 1; m >>= 1) {
        s1 += __shfl_xor_sync(0xffffffffu, s1, m);
        s2 += __shfl_xor_sync(0xffffffffu, s2, m);
    }
    if ((threadIdx.x & 31) == 0) { sh1[threadIdx.x >> 5] = s1; sh2[threadIdx.x >> 5] = s2; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < kMmThreads / 32; ++w) { s1 += sh1[w]; s2 += sh2[w]; }
        const double n = (double)(hi - lo);
        pmean[s * nchunk + c] = K + s1 / n;
        pm2[s * nchunk + c] = s2 - s1 * s1 / n;
    }
}

template <typename T>
__global__ void k_std_final(const double* __restrict__ pmean, const double* __restrict__ pm2, int nchunk, int64_t stream_size,
                            int64_t n_stream, T* __restrict__ out) {
    int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_stream) return;
    double n = 0.0, mean = 0.0, m2 = 0.0;
    for (int c = 0; c < nchunk; ++c) {
        const int64_t lo = (int64_t)c * kMmChunk;
        const double nb = (double)((lo + kMmChunk < stream_size ? lo + kMmChunk : stream_size) - lo);
        const double mb = pmean[s * nchunk + c], qb = pm2[s * nchunk + c];
        const double d = mb - mean, nt = n + nb;
        mean += d * (nb / nt);
        m2 += qb + d * d * (n * nb / nt);
        n = nt;
    }
    out[s] = (T)sqrt(m2 > 0.0 ? m2 / n : 0.0);
}

template <typename T, typename I>
__global__ void __launch_bounds__(256) k_quantise(const T* __restrict__ data, int64_t stream_size, int64_t per_cta,
                                                  const T* __restrict__ offsets, const T* __restrict__ gains,
                                                  I* __restrict__ out) {
    const int64_t s = blockIdx.y;
    const T off = offsets[s], gain = gains[s];
    const int64_t lo = (int64_t)blockIdx.x * per_cta;
    const int64_t hi = lo + per_cta < stream_size ? lo + per_cta : stream_size;
    const T* p = data + s * stream_size;
    I* o = out + s * stream_size;
    for (int64_t i = lo + threadIdx.x; i < hi; i += 256) {
        if constexpr (sizeof(T) == 4) o[i] = quant_f32(p[i], off, gain);
        else o[i] = quant_f64(p[i], off, gain);
    }
}

// int -> float (utils.c:330-368).  `in` and `out` may alias (same element size).
template <typename I, typename T>
__global__ void __launch_bounds__(256) k_restore(const I* in, int64_t n_per_stream, int64_t per_cta,
                                                 const T* __restrict__ offsets, const T* __restrict__ gains, T* out) {
    const int64_t s = blockIdx.y;
    const T off = offsets[s];
    T coeff;
    if constexpr (sizeof(T) == 4) coeff = restore_coeff_f32(gains[s]);
    else coeff = restore_coeff_f64(gains[s]);
    const int64_t lo = (int64_t)blockIdx.x * per_cta;
    const int64_t hi = lo + per_cta < n_per_stream ? lo + per_cta : n_per_stream;
    const I* p = in + s * n_per_stream;
    T* o = out + s * n_per_stream;
    for (int64_t i = lo + threadIdx.x; i < hi; i += 256) {
        I v = p[i];
        if constexpr (sizeof(T) == 4) o[i] = restore_f32(v, off, coeff);
        else o[i] = restore_f64(v, off, coeff);
    }
}

// ---- decode stages ---------------------------------------------------------------------------------
// one warp per stream: metadata + frame offsets (meta_warp)
__global__ void __launch_bounds__(128) k_dec_meta(const DecParams P) {
    const int64_t k = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    if (k >= P.n_sel) return;
    meta_warp(P, k);
}

constexpr int kSyncThreads = 256;
constexpr int kSyncBytesPerThread = 64;      // grid sizing: bytes of a stream per thread and grid pass

// frame-sync scan of the streams without a frame-size table: grid (x, stream), the warps of a stream's CTAs stride
// over its 512-byte rows (sync_scan_warp)
__global__ void __launch_bounds__(kSyncThreads) k_dec_sync(const DecParams P) {
    const int64_t k = blockIdx.y;
    sync_scan_warp(P, k, (int64_t)blockIdx.x * (kSyncThreads / 32) + (threadIdx.x >> 5), (int64_t)gridDim.x * (kSyncThreads / 32));
}

constexpr int kDecThreads = 128;

template <bool WIN>
__global__ void __launch_bounds__(kDecThreads) k_dec_frames(const DecParams P, const WinParams W, int64_t nwin) {
    // one thread per work item (stream, frame index inside the sample window), see resolve_item
    frames_item<WIN>(P, W, nwin, (int64_t)blockIdx.x * kDecThreads + threadIdx.x);
}

// throughput path: one warp = 32 (stream, frame) items, see fa_decode_tile.h.
// 20 resident one-warp CTAs per SM at 96 registers: no spills in the sample loop (21 would cap the kernel at 80).  The
// figures below were taken with two-warp CTAs.  Measured on cfg2-shaped decodes of
// 350 / 600 / 1000 streams (k_dec_tile + k_dec_crc, ms; residency below the build's limit forced with unused shared
// memory): 12 CTAs at 80 registers 1.58 / 2.59 / 3.74, 11: 1.55 / 2.63 / 3.82, 10 CTAs at 96 registers 1.33 / 2.34 / 3.41,
// 9: 1.72 / 2.44 / 3.50, 8: 1.83 / 2.35 / 3.74, 13 CTAs at 72 registers 4.70 at 1000 streams (spills).  A work item is a
// warp of 32 whole frames (~1 ms, a third of the kernel at cfg2), so the fill of the last wave shows in every column
// (1340 CTAs on 1480 slots at 350 streams); a per-call choice of the residency from a wave model was tried and bought
// nothing over the fixed 10.
#ifndef FAB_DEC_CTAS
#define FAB_DEC_CTAS (20 / FAB_TILE_WARPS)
#endif
// (WIN: the item space of fab_decode_windows, `total` items; STORE = false: fab_verify, decode and check only)
template <bool WIN, bool STORE = true>
__global__ void __launch_bounds__(kTileWarps * 32, FAB_DEC_CTAS) k_dec_tile(const TileParams P, int64_t total) {
    __shared__ TileShared ws[kTileWarps];
    int64_t item0 = ((int64_t)blockIdx.x * kTileWarps + (threadIdx.x >> 5)) * 32;
    if (item0 >= total) return;
    tile_warp_body<WIN, STORE>(P, item0, &ws[threadIdx.x >> 5]);
}

// frame CRC-16 of every (stream, frame) item: one warp per item, see crc_frame_warp
template <bool WIN>
__global__ void __launch_bounds__(128) k_dec_crc(const TileParams P, int64_t total) {
    int64_t idx = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    if (idx >= total) return;
    crc_frame_warp<WIN>(P, idx);
}

// int32 -> float32 for the sample ranges that were NOT written by the fused tile path (frames left to
// the general decoder, streams left to the walker).  grid = (nwin, n_sel)
__global__ void __launch_bounds__(256) k_restore_fixup(const TileParams P) {
    const DecParams& D = P.D;
    const int64_t k = blockIdx.y;
    const int sflag = D.stream_flag[k];
    if (sflag == 4) return;
    const int bs = D.meta[k].blocksize > 0 ? D.meta[k].blocksize : 4096;
    int64_t j0 = D.first / bs, j1 = (D.first + D.n_decode - 1) / bs;
    int64_t nfr = j1 - j0 + 1;
    float* out = (float*)D.data + k * D.n_decode;
    const int32_t* in = D.data + k * D.n_decode;
    const float off = P.offsets[k], coeff = restore_coeff_f32(P.gains[k]);
    if (sflag != 0) {
        // whole window of this stream was (re)written as integers by the walker
        for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < D.n_decode; i += (int64_t)gridDim.x * 256)
            out[i] = restore_f32(in[i], off, coeff);
        return;
    }
    __shared__ unsigned char fl[256];
    for (int64_t base = (int64_t)blockIdx.x * 256; base < nfr; base += (int64_t)gridDim.x * 256) {
        const int64_t jt = j0 + base + threadIdx.x;
        const bool mine = base + threadIdx.x < nfr && jt < D.nframes_cap && P.frame_flag[k * (int64_t)D.nframes_cap + jt];
        if (!__syncthreads_or(mine)) continue;     // the usual case: the tile path wrote floats everywhere
        fl[threadIdx.x] = mine;
        __syncthreads();
        for (int q = 0; q < 256; ++q) {
            if (!fl[q]) continue;
            const int64_t j = j0 + base + q;
            int64_t lo = j * bs - D.first, hi = lo + bs;
            if (lo < 0) lo = 0;
            if (hi > D.n_decode) hi = D.n_decode;
            for (int64_t i = lo + threadIdx.x; i < hi; i += 256) out[i] = restore_f32(in[i], off, coeff);
        }
        __syncthreads();
    }
}

__global__ void k_dec_walker(const DecParams P) {
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < P.n_sel) walker_body(P, k);
}

// fab_decode_isolated / fab_verify: failures go to P.status, P.data null = discard mode
__global__ void k_dec_walker_iso(const DecParams P) {
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < P.n_sel) walker_body<true>(P, k);
}

// fab_decode_isolated: overwrite the whole output row of every stream whose status is not 0 with `fill` (0 for integer
// output, a quiet NaN for float output), after the walker and the restore.  grid = (x, streams of one slab).
template <typename W>
__global__ void __launch_bounds__(256) k_dec_fill_failed(const int* __restrict__ status, W* out, int64_t n_per_stream, W fill) {
    fill_failed<W>(status, out, n_per_stream, fill, blockIdx.y, (int64_t)blockIdx.x * 256 + threadIdx.x, (int64_t)gridDim.x * 256);
}

// ---- fab_row_stats (fa_stats.h): grid = (pieces / kStatsWarps, rows of one slab); one warp per piece / per bin -------
template <bool I64>
__global__ void __launch_bounds__(kStatsWarps * 32) k_row_stats(const StatsParams P, int64_t row0) {
    const int64_t idx = (int64_t)blockIdx.x * kStatsWarps + (threadIdx.x >> 5);
    if (idx < P.nbins * P.ppb) stats_piece_warp<I64>(P, row0 + blockIdx.y, idx);
}

__global__ void __launch_bounds__(kStatsWarps * 32) k_row_stats_merge(const StatsParams P, int64_t row0) {
    const int64_t b = (int64_t)blockIdx.x * kStatsWarps + (threadIdx.x >> 5);
    if (b < P.nbins) stats_merge_warp(P, row0 + blockIdx.y, b);
}

// ---- fab_combine_rows (fa_combine.h): grid = (column chunks, segments of one slab); one CTA per (segment, chunk) ----
template <bool I64, bool FLT>
__global__ void __launch_bounds__(kCombineThreads) k_combine_rows(const CombineParams P, int64_t s0) {
    __shared__ CombineRow sh[kCombineThreads];
    combine_segment_cta<I64, FLT, kCombineThreads>(P, s0 + blockIdx.y,
                                                   (int64_t)blockIdx.x * (kCombineThreads * kCombineCols), sh);
}

// ---- fab_decode_windows ------------------------------------------------------------------------------
// window records -> item space (win_prep_cta), one CTA
constexpr int kWinScanThreads = 1024;
__global__ void __launch_bounds__(kWinScanThreads) k_win_prep(const WinParams W, int64_t n_sel, int64_t stream_size, int* err) {
    __shared__ long long wpre[kWinScanThreads / 32];
    __shared__ long long ctot;
    win_prep_cta<kWinScanThreads>(W, n_sel, stream_size, err, wpre, &ctot);
}

// fab_decode_windows: the walker, one thread per window (walker_win)
__global__ void k_dec_walker_win(const DecParams P, const WinParams W) {
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w < W.n_win) walker_win(P, W, w);
}

// Windowed int -> float, one warp per work item over the item's samples.  F64: every sample (the decoders wrote int64
// everywhere).  float32: only what the fused tile path did not restore -- frames flagged for the general decoder, and the
// whole window of a stream left to the walker (there the items cover the window in hinted-blocksize pieces).
template <bool F64>
__global__ void __launch_bounds__(128) k_restore_win(const TileParams P, int64_t total) {
    const int64_t idx = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    if (idx >= total) return;
    const DecParams& D = P.D;
    const WorkItem it = resolve_item<true>(D, P.W, P.nwin, idx);
    const int64_t k = it.k;
    if (k < 0) return;
    const int sflag = D.stream_flag[k];
    const bool whole = F64 || sflag != 0;
    if (!whole && D.meta[k].blocksize <= 0) return;
    if (!F64 && sflag == 4) return;
    const int64_t bs = whole ? P.W.bsh : D.meta[k].blocksize;
    const int64_t j = it.first / bs + it.jrel;
    if (!whole && (j >= D.nframes_cap || !P.frame_flag[k * (int64_t)D.nframes_cap + j])) return;
    int64_t lo = j * bs - it.first, hi = lo + bs;
    if (lo < 0) lo = 0;
    if (hi > it.n) hi = it.n;
    const int ln = threadIdx.x & 31;
    if constexpr (F64) {
        const double off = ((const double*)P.offsets)[k], coeff = restore_coeff_f64(((const double*)P.gains)[k]);
        const long long* in = (const long long*)D.data + it.out;
        double* out = (double*)D.data + it.out;
        for (int64_t i = lo + ln; i < hi; i += 32) out[i] = restore_f64(in[i], off, coeff);
    } else {
        const float off = P.offsets[k], coeff = restore_coeff_f32(P.gains[k]);
        const int32_t* in = D.data + it.out;
        float* out = (float*)D.data + it.out;
        for (int64_t i = lo + ln; i < hi; i += 32) out[i] = restore_f32(in[i], off, coeff);
    }
}

__global__ void k_max_i64(const long long* __restrict__ v, int64_t n, long long* __restrict__ out) {
    long long m = 0;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) m = v[i] > m ? v[i] : m;
    __shared__ long long sm[256];
    sm[threadIdx.x] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < blockDim.x; ++i) m = sm[i] > m ? sm[i] : m;
        *out = m;
    }
}

// =================================================================================================
// Context
// =================================================================================================
struct fab_ctx {
    int device = -1;
    CrcTables* d_crc = nullptr;
    EncTables* d_tab = nullptr;
    int n_sm = 0;
    int enc_ctas_per_sm[2][2] = {{0, 0}, {0, 0}};   // [H == 12][nch - 1]
    int compact_ctas_per_sm = 0;
    float* d_window[3] = {nullptr, nullptr, nullptr};  // [0] 1152, [1] 4096 (both zero-padded to 4096 floats), [2] 4096 in [quad][thread][4] order
    int* d_err = nullptr;
    int* h_err = nullptr;  // pinned
    unsigned char* scratch = nullptr;      // grow-only block owned by the context ...
    size_t scratch_bytes = 0;
    unsigned char* ws_user = nullptr;      // ... unless the caller supplied a workspace (fab_set_workspace)
    size_t ws_user_bytes = 0;
    cudaStream_t last_stream = nullptr;    // stream of the most recent call that used the scratch block
    int64_t launches = 0;
    std::string last_error = "";
    bool smem_configured = false;
    // second stream for work that only fills idle SMs (CRC pass behind the tile decoder's last wave,
    // compaction of batch b under the analysis of batch b + 1); fork / join with events
    cudaStream_t aux = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_join2 = nullptr;
    // third stream: the few frames that are not full (last frame of every stream) are analysed / encoded by their own
    // small kernels next to the full-frame kernels of the same batch instead of behind them
    cudaStream_t aux2 = nullptr;
    cudaEvent_t ev_sfork = nullptr, ev_sjoin = nullptr;
    // optional per-kernel timing (bench.py's roofline): CUDA events on the launching stream
    bool prof = false;
    struct Pending { cudaEvent_t a, b; int which; };
    std::vector<Pending> pending;
    double prof_ms[3] = {0.0, 0.0, 0.0};   // [0] k_encode, [1] k_dec_tile, [2] k_enc_analyze
    int64_t prof_n[3] = {0, 0, 0};
};

static void prof_begin(fab_ctx* ctx, int which, cudaStream_t st) {
    if (!ctx->prof) return;
    fab_ctx::Pending p;
    p.which = which;
    if (cudaEventCreate(&p.a) != cudaSuccess || cudaEventCreate(&p.b) != cudaSuccess) return;
    cudaEventRecord(p.a, st);
    ctx->pending.push_back(p);
}
static void prof_end(fab_ctx* ctx, cudaStream_t st) {
    if (!ctx->prof || ctx->pending.empty()) return;
    cudaEventRecord(ctx->pending.back().b, st);
}
static void prof_collect(fab_ctx* ctx) {
    for (auto& p : ctx->pending) {
        float ms = 0.f;
        if (cudaEventSynchronize(p.b) == cudaSuccess && cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) {
            ctx->prof_ms[p.which] += ms;
            ctx->prof_n[p.which]++;
        }
        cudaEventDestroy(p.a);
        cudaEventDestroy(p.b);
    }
    ctx->pending.clear();
}

#define FAB_CUDA(ctx, call)                                                                   \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess) {                                                              \
            if (ctx) (ctx)->last_error = std::string(#call) + ": " + cudaGetErrorString(e_);  \
            return FAB_ERROR_CUDA;                                                            \
        }                                                                                     \
    } while (0)

static int ctx_scratch(fab_ctx* ctx, size_t bytes, unsigned char** out, cudaStream_t st) {
    if (ctx->ws_user) {
        // caller-supplied workspace (fab_set_workspace): never allocate behind the caller's back
        if (bytes > ctx->ws_user_bytes) {
            ctx->last_error = "workspace too small: " + std::to_string(bytes) + " bytes needed, " +
                              std::to_string(ctx->ws_user_bytes) + " supplied (see fab_encode_workspace_bytes / fab_decode_workspace_bytes)";
            return ERROR_ALLOC;
        }
        ctx->last_stream = st;
        *out = ctx->ws_user;
        return 0;
    }
    if (bytes > ctx->scratch_bytes) {
        if (ctx->scratch) {
            // only this context's own work can still be reading the old block: the stream of its previous call and the
            // helper streams (not the whole device -- other contexts and the caller's other streams keep running)
            FAB_CUDA(ctx, cudaStreamSynchronize(ctx->last_stream));
            FAB_CUDA(ctx, cudaStreamSynchronize(ctx->aux));
            FAB_CUDA(ctx, cudaStreamSynchronize(ctx->aux2));
            cudaFree(ctx->scratch);
            ctx->scratch = nullptr;
            ctx->scratch_bytes = 0;
        }
        size_t want = bytes + (bytes >> 2) + (1 << 20);
        cudaError_t e = cudaMalloc((void**)&ctx->scratch, want);
        if (e != cudaSuccess) {
            ctx->last_error = std::string("cudaMalloc(scratch): ") + cudaGetErrorString(e);
            cudaGetLastError();
            return ERROR_ALLOC | FAB_ERROR_CUDA;
        }
        ctx->scratch_bytes = want;
    }
    ctx->last_stream = st;
    *out = ctx->scratch;
    return 0;
}

static size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

extern "C" int fab_create(fab_ctx** out) {
    *out = nullptr;
    int dev = -1;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) { cudaGetLastError(); return FAB_ERROR_CUDA; }
    fab_ctx* ctx = new fab_ctx();
    ctx->device = dev;
    CrcTables* h = new CrcTables();
    crc_tables_init(h);
    EncTables* ht = new EncTables();
    enc_tables_init(ht);
    cudaDeviceGetAttribute(&ctx->n_sm, cudaDevAttrMultiProcessorCount, dev);
    std::vector<float> w0(4096, 0.f), w1(4096), w2(4096);
    make_tukey_window(w0.data(), 1152);
    make_tukey_window(w1.data(), 4096);
    permute_window_qt(w1.data(), w2.data());
    bool ok = cudaMalloc((void**)&ctx->d_crc, sizeof(CrcTables)) == cudaSuccess &&
              cudaMemcpy(ctx->d_crc, h, sizeof(CrcTables), cudaMemcpyHostToDevice) == cudaSuccess &&
              cudaMalloc((void**)&ctx->d_tab, sizeof(EncTables)) == cudaSuccess &&
              cudaMemcpy(ctx->d_tab, ht, sizeof(EncTables), cudaMemcpyHostToDevice) == cudaSuccess &&
              cudaMalloc((void**)&ctx->d_window[0], 4096 * 4) == cudaSuccess &&
              cudaMemcpy(ctx->d_window[0], w0.data(), 4096 * 4, cudaMemcpyHostToDevice) == cudaSuccess &&
              cudaMalloc((void**)&ctx->d_window[2], 4096 * 4) == cudaSuccess &&
              cudaMemcpy(ctx->d_window[2], w2.data(), 4096 * 4, cudaMemcpyHostToDevice) == cudaSuccess &&
              cudaMalloc((void**)&ctx->d_window[1], 4096 * 4) == cudaSuccess &&
              cudaMemcpy(ctx->d_window[1], w1.data(), 4096 * 4, cudaMemcpyHostToDevice) == cudaSuccess &&
              cudaMalloc((void**)&ctx->d_err, 4) == cudaSuccess && cudaMemset(ctx->d_err, 0, 4) == cudaSuccess &&
              cudaMallocHost((void**)&ctx->h_err, 4) == cudaSuccess &&
              cudaStreamCreateWithFlags(&ctx->aux, cudaStreamNonBlocking) == cudaSuccess &&
              cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) == cudaSuccess &&
              cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming) == cudaSuccess &&
              cudaEventCreateWithFlags(&ctx->ev_join2, cudaEventDisableTiming) == cudaSuccess &&
              cudaStreamCreateWithFlags(&ctx->aux2, cudaStreamNonBlocking) == cudaSuccess &&
              cudaEventCreateWithFlags(&ctx->ev_sfork, cudaEventDisableTiming) == cudaSuccess &&
              cudaEventCreateWithFlags(&ctx->ev_sjoin, cudaEventDisableTiming) == cudaSuccess;
    delete h;
    delete ht;
    if (!ok) {
        cudaGetLastError();
        fab_destroy(ctx);
        return FAB_ERROR_CUDA;
    }
    *out = ctx;
    return 0;
}

extern "C" void fab_destroy(fab_ctx* ctx) {
    if (!ctx) return;
    if (ctx->d_crc) cudaFree(ctx->d_crc);
    if (ctx->d_tab) cudaFree(ctx->d_tab);
    if (ctx->d_window[0]) cudaFree(ctx->d_window[0]);
    if (ctx->d_window[1]) cudaFree(ctx->d_window[1]);
    if (ctx->d_window[2]) cudaFree(ctx->d_window[2]);
    if (ctx->d_err) cudaFree(ctx->d_err);
    if (ctx->h_err) cudaFreeHost(ctx->h_err);
    if (ctx->scratch) cudaFree(ctx->scratch);
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    if (ctx->ev_join2) cudaEventDestroy(ctx->ev_join2);
    if (ctx->aux) cudaStreamDestroy(ctx->aux);
    if (ctx->ev_sfork) cudaEventDestroy(ctx->ev_sfork);
    if (ctx->ev_sjoin) cudaEventDestroy(ctx->ev_sjoin);
    if (ctx->aux2) cudaStreamDestroy(ctx->aux2);
    delete ctx;
}

extern "C" int fab_set_workspace(fab_ctx* ctx, void* d_workspace, int64_t bytes) {
    if (!ctx) return FAB_ERROR_CUDA;
    if (d_workspace && (bytes <= 0 || ((uintptr_t)d_workspace & 255) != 0)) {
        ctx->last_error = "fab_set_workspace: the block must be 256-byte aligned and not empty";
        return ERROR_ALLOC;
    }
    // work queued by earlier calls may still use the block that is being replaced
    FAB_CUDA(ctx, cudaStreamSynchronize(ctx->last_stream));
    FAB_CUDA(ctx, cudaStreamSynchronize(ctx->aux));
    FAB_CUDA(ctx, cudaStreamSynchronize(ctx->aux2));
    ctx->ws_user = (unsigned char*)d_workspace;
    ctx->ws_user_bytes = d_workspace ? (size_t)bytes : 0;
    if (d_workspace && ctx->scratch) {
        cudaFree(ctx->scratch);
        ctx->scratch = nullptr;
        ctx->scratch_bytes = 0;
    }
    return 0;
}

extern "C" const char* fab_last_error(const fab_ctx* ctx) { return ctx ? ctx->last_error.c_str() : "no context"; }
extern "C" int64_t fab_launch_count(const fab_ctx* ctx) { return ctx ? ctx->launches : 0; }

extern "C" void fab_profile(fab_ctx* ctx, int enable) {
    if (!ctx) return;
    prof_collect(ctx);
    ctx->prof = enable != 0;
    ctx->prof_ms[0] = ctx->prof_ms[1] = ctx->prof_ms[2] = 0.0;
    ctx->prof_n[0] = ctx->prof_n[1] = ctx->prof_n[2] = 0;
}
extern "C" double fab_profile_ms(fab_ctx* ctx, int which, int64_t* count) {
    if (!ctx || which < 0 || which > 2) return 0.0;
    prof_collect(ctx);
    if (count) *count = ctx->prof_n[which];
    return ctx->prof_ms[which];
}

extern "C" int fab_finish(fab_ctx* ctx, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    FAB_CUDA(ctx, cudaMemcpyAsync(ctx->h_err, ctx->d_err, 4, cudaMemcpyDeviceToHost, st));
    FAB_CUDA(ctx, cudaMemsetAsync(ctx->d_err, 0, 4, st));
    FAB_CUDA(ctx, cudaStreamSynchronize(st));
    FAB_CUDA(ctx, cudaGetLastError());
    return *ctx->h_err;
}

// =================================================================================================
// Encode
// =================================================================================================
static int dtype_channels(int dtype) { return (dtype == FAB_I64 || dtype == FAB_F64) ? 2 : 1; }

extern "C" int64_t fab_encode_bound(int64_t n_stream, int64_t stream_size, int dtype, uint32_t level) {
    if (level > 8 || n_stream <= 0 || stream_size <= 0) return 0;
    LevelPreset lp = level_preset((int)level);
    int nch = dtype_channels(dtype);
    int64_t nf = (stream_size + lp.blocksize - 1) / lp.blocksize;
    return n_stream * (stream_header_bytes((int)nf) + nf * (16 + 2 + (int64_t)nch * (lp.blocksize * 4 + 8)));
}

// Workspace of one fab_encode call: [min/max partials of the quantise pre-pass] | byte prefixes | ends | work counters |
// per-batch statistics, plans, frame sizes, slots.  Sized once up front so that the pre-pass (queued first on the same
// stream) and the encoder never share bytes.
struct EncWorkspace {
    size_t pre, desc_b, ends_b, stats_b, plans_b, tick_b, fsize_b, slots_b, total;
    int64_t total_frames, slot_bytes, batch, nbatch;
    int nbuf;
};
static EncWorkspace enc_workspace(int64_t n_stream, int64_t stream_size, int dtype, const LevelPreset& lp) {
    EncWorkspace W;
    const int nch = dtype_channels(dtype);
    const int64_t nf = (stream_size + lp.blocksize - 1) / lp.blocksize;
    W.pre = 0;
    if (dtype >= FAB_F32) {
        int nchunk = (int)((stream_size + kMmChunk - 1) / kMmChunk);
        W.pre = 2 * align256((size_t)n_stream * nchunk * (dtype == FAB_F32 ? 4 : 8));
    }
    W.desc_b = align256((size_t)(n_stream * nf) * 8);
    W.ends_b = align256((size_t)n_stream * 8);
    // the encoder kernels run over batches of (stream, frame) units so that the per-frame records and the
    // slot buffers between them stay bounded (2 x 1 GB); one work counter per batch
    W.total_frames = n_stream * nf;
    W.slot_bytes = (int64_t)((16 + 2 + (int64_t)nch * (lp.blocksize * 4 + 8) + 15) & ~15ll);
    W.batch = std::min<int64_t>(W.total_frames, std::max<int64_t>(1024, kEncBatchBytes / W.slot_bytes));
    W.nbatch = (W.total_frames + W.batch - 1) / W.batch;
    W.nbuf = W.nbatch > 1 ? 2 : 1;     // slot / frame-size buffers alternate between consecutive batches
    W.stats_b = align256((size_t)W.batch * nch * sizeof(FrameStats));
    W.plans_b = align256((size_t)W.batch * nch * sizeof(FramePlan)) + align256((size_t)W.batch * nch * sizeof(PlanHeader));
    W.tick_b = align256((size_t)W.nbatch * 4 + 16);
    W.fsize_b = align256((size_t)W.batch * 4);
    W.slots_b = align256((size_t)W.batch * (size_t)W.slot_bytes);
    W.total = W.pre + W.desc_b + W.ends_b + W.tick_b + W.stats_b + W.plans_b + W.nbuf * (W.fsize_b + W.slots_b) + 256;
    return W;
}

extern "C" int64_t fab_encode_workspace_bytes(int64_t n_stream, int64_t stream_size, int dtype, uint32_t level) {
    if (level > 8 || n_stream <= 0 || stream_size <= 0 || dtype < 0 || dtype > 3) return 0;
    return (int64_t)enc_workspace(n_stream, stream_size, dtype, level_preset((int)level)).total;
}

template <typename T>
static int launch_quant_params(fab_ctx* ctx, const T* d_in, int64_t n_stream, int64_t stream_size, const T* d_quanta,
                               T* d_off, T* d_gain, cudaStream_t st) {
    int nchunk = (int)((stream_size + kMmChunk - 1) / kMmChunk);
    unsigned char* scr;
    size_t need = 2 * align256((size_t)n_stream * nchunk * sizeof(T));
    int rc = ctx_scratch(ctx, need, &scr, st);
    if (rc) return rc;
    T* pmin = (T*)scr;
    T* pmax = (T*)(scr + align256((size_t)n_stream * nchunk * sizeof(T)));
    // gridDim.y is limited to 65535: loop over slabs of streams
    for (int64_t s0 = 0; s0 < n_stream; s0 += 65535) {
        int64_t ns = std::min<int64_t>(65535, n_stream - s0);
        dim3 grid((unsigned)nchunk, (unsigned)ns);
        k_minmax<T><<<grid, kMmThreads, 0, st>>>(d_in + s0 * stream_size, stream_size, nchunk, pmin + s0 * nchunk,
                                                 pmax + s0 * nchunk, ctx->d_err);
        ctx->launches++;
    }
    k_quant_params<T><<<(unsigned)((n_stream + 127) / 128), 128, 0, st>>>(pmin, pmax, nchunk, n_stream, d_quanta, d_off, d_gain);
    ctx->launches++;
    FAB_CUDA(ctx, cudaGetLastError());
    return 0;
}

extern "C" int fab_encode(fab_ctx* ctx, const void* d_data, int dtype, int64_t n_stream, int64_t stream_size,
                          uint32_t level, const void* d_quanta, void* d_offsets, void* d_gains, unsigned char* d_out,
                          int64_t out_capacity, int64_t* d_starts, int64_t* d_nbytes, int64_t* d_total, void* stream) {
    if (!ctx) return FAB_ERROR_CUDA;
    // argument checks: compress.c:143-152
    if (level > 8) return ERROR_INVALID_LEVEL;
    if (n_stream == 0) return ERROR_ZERO_NSTREAM;
    if (stream_size == 0) return ERROR_ZERO_STREAMSIZE;
    if (dtype < 0 || dtype > 3) return ERROR_CONVERT_TYPE;
    cudaStream_t st = (cudaStream_t)stream;
    LevelPreset lp = level_preset((int)level);
    const int nch = dtype_channels(dtype);
    const int64_t nf = (stream_size + lp.blocksize - 1) / lp.blocksize;
    if (n_stream * nf > 0x7fffffffLL) return ERROR_ALLOC;  // frame indices are 32 bit
    if (8 + 3 * nf > 0xFFFFFFLL) {
        // the per-stream frame-size table (APPLICATION block "faB2") carries a 24-bit length: a stream of more than
        // ~5.59 M frames (6.4e9 samples at blocksize 1152, 22.9e9 at 4096) cannot be described
        ctx->last_error = "stream too long for the frame-size table (more than 5592402 frames)";
        return ERROR_ENCODE_INIT;
    }

    const EncWorkspace W = enc_workspace(n_stream, stream_size, dtype, lp);
    const size_t pre = W.pre, desc_b = W.desc_b, ends_b = W.ends_b, stats_b = W.stats_b, plans_b = W.plans_b, tick_b = W.tick_b,
                 fsize_b = W.fsize_b, slots_b = W.slots_b;
    const int64_t total_frames = W.total_frames, slot_bytes = W.slot_bytes, batch = W.batch, nbatch = W.nbatch;
    const int nbuf = W.nbuf;
    unsigned char* scr;
    int rc = ctx_scratch(ctx, W.total, &scr, st);
    if (rc) return rc;

    prof_begin(ctx, 0, st);     // slot 0: every kernel of this call: min/max pre-pass, all encoder batches
    if (dtype == FAB_F32) {
        rc = launch_quant_params<float>(ctx, (const float*)d_data, n_stream, stream_size, (const float*)d_quanta,
                                        (float*)d_offsets, (float*)d_gains, st);
        if (rc) return rc;
    } else if (dtype == FAB_F64) {
        rc = launch_quant_params<double>(ctx, (const double*)d_data, n_stream, stream_size, (const double*)d_quanta,
                                         (double*)d_offsets, (double*)d_gains, st);
        if (rc) return rc;
    }
    unsigned long long* desc = (unsigned long long*)(scr + pre);
    long long* ends = (long long*)(scr + pre + desc_b);
    uint32_t* ticket = (uint32_t*)(scr + pre + desc_b + ends_b);
    FrameStats* stats = (FrameStats*)(scr + pre + desc_b + ends_b + tick_b);
    FramePlan* plans = (FramePlan*)(scr + pre + desc_b + ends_b + tick_b + stats_b);
    unsigned char* fs0 = scr + pre + desc_b + ends_b + tick_b + stats_b + plans_b;
    unsigned char* sl0 = fs0 + nbuf * fsize_b;
    FAB_CUDA(ctx, cudaMemsetAsync(desc, 0, desc_b + ends_b + tick_b, st));

    EncParams P;
    P.data = d_data; P.dtype = dtype; P.offsets = d_offsets; P.gains = d_gains;
    P.n_stream = n_stream; P.stream_size = stream_size; P.nch = nch;
    P.blocksize = lp.blocksize; P.nframes = (int)nf;
    P.max_lpc_order = lp.max_lpc_order; P.max_porder = lp.max_porder;
    P.qlp_precision = lp.blocksize <= 384 ? 13 : (lp.blocksize <= 1152 ? 14 : 15);
    P.window = ctx->d_window[lp.blocksize == 1152 ? 0 : 1];
    P.window_qt = ctx->d_window[2];
    P.crc = ctx->d_crc; P.tab = ctx->d_tab;
    P.out = d_out; P.out_capacity = out_capacity;
    P.starts = (long long*)d_starts; P.ends = ends; P.desc = desc; P.ticket = ticket; P.err = ctx->d_err;
    P.hdr_bytes = stream_header_bytes((int)nf);

#ifndef FAB_SMEM_PAD
#define FAB_SMEM_PAD 0
#endif
    size_t smem = enc_smem_bytes(nch) + FAB_SMEM_PAD;   // (FAB_SMEM_PAD: experiment knob, shrinks the L1)
    if (!ctx->smem_configured) {
        FAB_CUDA(ctx, cudaFuncSetAttribute(k_encode<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)enc_smem_bytes(2) + FAB_SMEM_PAD));
        FAB_CUDA(ctx, cudaFuncSetAttribute(k_encode<12>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)enc_smem_bytes(2)));
        FAB_CUDA(ctx, cudaFuncSetAttribute(k_encode_short<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)enc_smem_bytes(2)));
        FAB_CUDA(ctx, cudaFuncSetAttribute(k_encode_short<12>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)enc_smem_bytes(2)));
        for (int c = 0; c < 2; ++c) {
            FAB_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->enc_ctas_per_sm[0][c], k_encode<8>, kEncThreads, enc_smem_bytes(c + 1) + FAB_SMEM_PAD));
            FAB_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->enc_ctas_per_sm[1][c], k_encode<12>, kEncThreads, enc_smem_bytes(c + 1)));
        }
        FAB_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->compact_ctas_per_sm, k_enc_compact, 128, 0));
        ctx->smem_configured = true;
    }
    P.stats = stats; P.plans = plans;
    P.hdrs = (PlanHeader*)((unsigned char*)plans + align256((size_t)batch * nch * sizeof(FramePlan)));
    P.slot_bytes = slot_bytes;
    P.base = (unsigned long long*)(ticket + ((nbatch + 3) & ~3ll));   // zeroed with the tickets (8-byte aligned)
    const int h12 = lp.max_lpc_order > 8 ? 1 : 0;
    int64_t resident = (int64_t)ctx->n_sm * std::max(1, ctx->enc_ctas_per_sm[h12][nch - 1]);
    cudaEvent_t joins[2] = {ctx->ev_join, ctx->ev_join2};
    for (int64_t bi = 0; bi < nbatch; ++bi) {
        P.g_begin = (uint32_t)(bi * batch);
        P.g_end = (uint32_t)std::min<int64_t>(total_frames, (bi + 1) * batch);
        P.ticket = ticket + bi;
        P.fsize = (uint32_t*)(fs0 + (bi & 1) * fsize_b);
        P.slots = sl0 + (bi & 1) * slots_b;
        const int64_t nfr = (int64_t)P.g_end - (int64_t)P.g_begin;
        // The size scan and the compaction of batch b (memory-bound, plus the frame CRCs) run on the second stream
        // under the kernels of batch b + 1, which use the other slot / frame-size buffers; k_enc_analyze of batch
        // b + 2 parks samples in the slots batch b compacts from, so it waits for that compaction.
        if (bi >= 2) FAB_CUDA(ctx, cudaStreamWaitEvent(st, joins[bi & 1], 0));
        if (lp.blocksize == kFxBs) {
            // levels 0..2: the warp-per-frame encoder first; the kernels below then only see what it left (fsize == 0)
            FAB_CUDA(ctx, cudaMemsetAsync(P.fsize, 0, (size_t)nfr * 4, st));
            k_enc_fixed<<<(unsigned)((nfr + kFxWarps - 1) / kFxWarps), kFxWarps * 32, 0, st>>>(P);
            ctx->launches++;
        }
        // frames that are not full: every frame (blocksize 1152), or the last frame of each stream when the stream
        // length is not a multiple of the blocksize
        uint32_t first = P.g_begin, stride = 1;
        int64_t cnt = nfr;
        if (lp.blocksize == kMaxBs) {
            cnt = 0;
            if (stream_size % lp.blocksize != 0) {
                stride = (uint32_t)nf;
                const int64_t g_last = ((int64_t)P.g_begin / nf) * nf + (nf - 1);     // last frame of the batch's first stream
                first = (uint32_t)g_last;
                cnt = g_last < (int64_t)P.g_end ? ((int64_t)P.g_end - 1 - g_last) / nf + 1 : 0;
            }
        }
        // (with full frames around, the short-frame kernels go to the third stream: latency-bound, a CTA per SM)
#ifdef FAB_NO_SIDE
        const bool side = false;
#else
        const bool side = lp.blocksize == kMaxBs && cnt > 0;
#endif
        cudaStream_t sst = side ? ctx->aux2 : st;
        if (side) {
            FAB_CUDA(ctx, cudaEventRecord(ctx->ev_sfork, st));
            FAB_CUDA(ctx, cudaStreamWaitEvent(sst, ctx->ev_sfork, 0));
        }
        if (cnt > 0) {
            const unsigned sgrid = (unsigned)std::min<int64_t>(cnt, (int64_t)ctx->n_sm * 8);
            if (h12) k_enc_analyze_short<12><<<sgrid, kEncThreads, 0, sst>>>(P, first, stride);
            else k_enc_analyze_short<8><<<sgrid, kEncThreads, 0, sst>>>(P, first, stride);
            ctx->launches++;
        }
        if (lp.blocksize == kMaxBs) {
            const unsigned agrid = (unsigned)std::min<int64_t>(nfr, (int64_t)ctx->n_sm * FAB_AN_CTAS);
            if (h12) k_enc_analyze<12><<<agrid, kEncThreads, 0, st>>>(P);
            else k_enc_analyze<8><<<agrid, kEncThreads, 0, st>>>(P);
            ctx->launches++;
        }
        if (side) {
            FAB_CUDA(ctx, cudaEventRecord(ctx->ev_sjoin, sst));
            FAB_CUDA(ctx, cudaStreamWaitEvent(st, ctx->ev_sjoin, 0));
        }
        k_enc_design<<<(unsigned)((nfr * nch + 127) / 128), 128, 0, st>>>(P, nfr * nch);
        if (side) {
            FAB_CUDA(ctx, cudaEventRecord(ctx->ev_sfork, st));
            FAB_CUDA(ctx, cudaStreamWaitEvent(sst, ctx->ev_sfork, 0));
        }
        if (cnt > 0) {
            const unsigned sgrid = (unsigned)std::min<int64_t>(cnt, (int64_t)ctx->n_sm * 4);
            if (h12) k_encode_short<12><<<sgrid, kEncThreads, smem, sst>>>(P, first, stride);
            else k_encode_short<8><<<sgrid, kEncThreads, smem, sst>>>(P, first, stride);
            ctx->launches++;
        }
        if (lp.blocksize == kMaxBs) {
            unsigned grid = (unsigned)std::min<int64_t>(nfr, resident);
            if (h12) k_encode<12><<<grid, kEncThreads, smem, st>>>(P);
            else k_encode<8><<<grid, kEncThreads, smem, st>>>(P);
            ctx->launches++;
        }
        if (side) {
            FAB_CUDA(ctx, cudaEventRecord(ctx->ev_sjoin, sst));
            FAB_CUDA(ctx, cudaStreamWaitEvent(st, ctx->ev_sjoin, 0));
        }
        FAB_CUDA(ctx, cudaEventRecord(ctx->ev_fork, st));
        FAB_CUDA(ctx, cudaStreamWaitEvent(ctx->aux, ctx->ev_fork, 0));
        k_enc_scan<<<1, kScanThreads, 0, ctx->aux>>>(P);      // (the running byte total is carried from scan to scan: all on aux)
        // (CTAs stride over the frames: exactly one resident wave, or the CTAs of a partial second wave run their whole
        // share of the frames after everybody else has finished)
#ifndef FAB_COMPACT_CTAS
#define FAB_COMPACT_CTAS std::max(1, ctx->compact_ctas_per_sm)
#endif
        k_enc_compact<<<(unsigned)std::min<int64_t>(nfr, (int64_t)ctx->n_sm * (FAB_COMPACT_CTAS)), 128, 0, ctx->aux>>>(P);
        FAB_CUDA(ctx, cudaEventRecord(joins[bi & 1], ctx->aux));
        ctx->launches += 3;
    }
    FAB_CUDA(ctx, cudaStreamWaitEvent(st, joins[(nbatch - 1) & 1], 0));
    if (nbatch > 1) FAB_CUDA(ctx, cudaStreamWaitEvent(st, joins[nbatch & 1], 0));
    P.g_begin = 0; P.g_end = (uint32_t)total_frames;
    k_enc_finalize<<<(unsigned)((n_stream * nf + 255) / 256), 256, 0, st>>>(P, (long long*)d_nbytes, (long long*)d_total);
    ctx->launches++;
    prof_end(ctx, st);
    FAB_CUDA(ctx, cudaGetLastError());
    return 0;
}

// =================================================================================================
// Decode
// =================================================================================================
// Workspace of one fab_decode call: stream metadata | frame offsets | stream flags | frame flags | one int64
struct DecWorkspace { size_t meta_b, fo_b, flag_b, fflag_b, total; };
static DecWorkspace dec_workspace(int64_t n_stream, int nframes_cap) {
    DecWorkspace W;
    W.meta_b = align256((size_t)n_stream * sizeof(StreamMeta));
    W.fo_b = align256((size_t)n_stream * (size_t)(nframes_cap + 1) * 8);
    W.flag_b = align256((size_t)n_stream * 4);
    W.fflag_b = align256((size_t)n_stream * (size_t)nframes_cap);
    W.total = W.meta_b + W.fo_b + W.flag_b + W.fflag_b + 256;
    return W;
}
extern "C" int64_t fab_decode_workspace_bytes(int64_t n_stream, int64_t stream_size, int blocksize_hint) {
    int bsh = 0, cap = 0;
    if (n_stream <= 0 || stream_size <= 0 || dec_frames_cap(stream_size, blocksize_hint, &bsh, &cap)) return 0;
    return (int64_t)dec_workspace(n_stream, cap).total;
}

// Stages 1 and 2 of a decode, once per stream slot: metadata + frame offsets (k_dec_meta), then the sync scan of the
// streams without a frame-size table (k_dec_sync, grid.y split at 65535 streams).
static void dec_index_streams(fab_ctx* ctx, const DecParams& P, int64_t max_nbytes, cudaStream_t st) {
    const int64_t n_stream = P.n_sel;
    k_dec_meta<<<(unsigned)((n_stream + 3) / 4), 128, 0, st>>>(P);
    ctx->launches++;
    int64_t per_cta = (int64_t)kSyncThreads * kSyncBytesPerThread;
    int64_t gx = (max_nbytes + per_cta - 1) / per_cta;
    // streams carrying a frame-size table leave at once: keep the grid near one wave-set of CTAs and
    // let the CTAs of a foreign stream stride over its chunks
    gx = std::max<int64_t>(1, std::min<int64_t>(gx, (148 * 32 + n_stream - 1) / n_stream));
    for (int64_t s0 = 0; s0 < n_stream; s0 += 65535) {
        int64_t ns = std::min<int64_t>(65535, n_stream - s0);
        DecParams Q = P;
        Q.starts += s0; Q.nbytes += s0; Q.meta += s0; Q.frame_off += s0 * (int64_t)(P.nframes_cap + 1); Q.stream_flag += s0;
        Q.n_sel = ns;
        dim3 grid((unsigned)gx, (unsigned)ns);
        k_dec_sync<<<grid, kSyncThreads, 0, st>>>(Q);
        ctx->launches++;
    }
}

// Stage 3 over `total` work items (resolve_item): warp-tile decoder, its CRC pass next to it on the second stream, then
// the general per-thread decoder on the frames the tile path flagged.  TP.frame_flag must be cleared.  STORE = false
// (fab_verify, TP.D.data null): the same stages, no samples written.
template <bool WIN, bool STORE = true>
static int dec_items(fab_ctx* ctx, const TileParams& TP, int64_t total, cudaStream_t st) {
    int64_t per_cta = (int64_t)kTileWarps * 32;
    prof_begin(ctx, 1, st);
    FAB_CUDA(ctx, cudaEventRecord(ctx->ev_fork, st));
    k_dec_tile<WIN, STORE><<<(unsigned)((total + per_cta - 1) / per_cta), kTileWarps * 32, 0, st>>>(TP, total);
    // the CRC pass only needs the frame table: it runs on the second stream, queued behind the tile
    // kernel's launch so that its CTAs fill the SMs the decoder's last partial wave leaves idle
    FAB_CUDA(ctx, cudaStreamWaitEvent(ctx->aux, ctx->ev_fork, 0));
    k_dec_crc<WIN><<<(unsigned)((total + 3) / 4), 128, 0, ctx->aux>>>(TP, total);
    FAB_CUDA(ctx, cudaEventRecord(ctx->ev_join, ctx->aux));
    FAB_CUDA(ctx, cudaStreamWaitEvent(st, ctx->ev_join, 0));
    prof_end(ctx, st);
    ctx->launches += 2;
    // general per-thread decoder: only the frames the tile path flagged
    DecParams P = TP.D;
    P.frame_flag = TP.frame_flag;
    k_dec_frames<WIN><<<(unsigned)((total + kDecThreads - 1) / kDecThreads), kDecThreads, 0, st>>>(P, TP.W, TP.nwin);
    ctx->launches++;
    return 0;
}

// fab_decode, fab_decode_isolated and fab_verify.  d_status null (fab_decode): a stream-fatal error goes to the call's
// error mask.
// d_status set: every stream reports its own (k_dec_meta, walker), and the rows of failed streams are filled once the
// walker and the restore are done.  store = false (fab_verify): d_out, d_offsets and d_gains are null and the tile
// decoder runs its no-store instantiation.
static int dec_uniform(fab_ctx* ctx, const unsigned char* d_bytes, const int64_t* d_starts, const int64_t* d_nbytes,
                       int64_t n_stream, int64_t stream_size, int is_int64, int64_t first_sample, int64_t last_sample,
                       void* d_out, const void* d_offsets, const void* d_gains, int64_t max_nbytes, int blocksize_hint,
                       int32_t* d_status, bool store, void* stream) {
    if (!ctx) return FAB_ERROR_CUDA;
    if (n_stream <= 0) return ERROR_ZERO_NSTREAM;
    if (stream_size <= 0) return ERROR_ZERO_STREAMSIZE;
    // decompress.c:207-222
    int64_t first_decode = 0, n_decode = stream_size;
    if (first_sample >= 0 && last_sample >= 0) {
        if (last_sample > stream_size) return ERROR_DECODE_SAMPLE_RANGE;
        if (first_sample > stream_size - 1) return ERROR_DECODE_SAMPLE_RANGE;
        if (first_sample >= last_sample) return ERROR_DECODE_SAMPLE_RANGE;
        first_decode = first_sample;
        n_decode = last_sample - first_sample;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int nch = is_int64 ? 2 : 1;
    int bsh = 0, nframes_cap = 0;
    if (dec_frames_cap(stream_size, blocksize_hint, &bsh, &nframes_cap)) return ERROR_ALLOC;

    const DecWorkspace W = dec_workspace(n_stream, nframes_cap);
    const size_t meta_b = W.meta_b, fo_b = W.fo_b, flag_b = W.flag_b, fflag_b = W.fflag_b;
    unsigned char* scr;
    int rc = ctx_scratch(ctx, W.total, &scr, st);
    if (rc) return rc;
    unsigned char* frame_flag = scr + meta_b + fo_b + flag_b;

    if (max_nbytes <= 0) {
        long long* d_max = (long long*)(scr + meta_b + fo_b + flag_b + fflag_b);
        k_max_i64<<<1, 256, 0, st>>>((const long long*)d_nbytes, n_stream, d_max);
        ctx->launches++;
        long long h = 0;
        FAB_CUDA(ctx, cudaMemcpyAsync(&h, d_max, 8, cudaMemcpyDeviceToHost, st));
        FAB_CUDA(ctx, cudaStreamSynchronize(st));
        max_nbytes = h;
    }

    DecParams P;
    P.bytes = d_bytes; P.starts = (const long long*)d_starts; P.nbytes = (const long long*)d_nbytes;
    P.n_sel = n_stream; P.stream_size = stream_size; P.nch = nch;
    P.first = first_decode; P.n_decode = n_decode; P.data = (int32_t*)d_out; P.crc = ctx->d_crc;
    P.meta = (StreamMeta*)scr; P.frame_off = (long long*)(scr + meta_b); P.nframes_cap = nframes_cap;
    P.stream_flag = (int*)(scr + meta_b + fo_b); P.err = ctx->d_err; P.verify_crc16 = 1; P.frame_flag = frame_flag;
    P.status = d_status;

    dec_index_streams(ctx, P, max_nbytes, st);
    const bool fuse_restore = d_offsets && d_gains && !is_int64;
    TileParams TP;
    {
        // frames overlapping the window, for the hinted blocksize (a stream whose real blocksize needs
        // more frames than that is handed to the walker by the kernels)
        int64_t nwin = (first_decode + n_decode - 1) / bsh - first_decode / bsh + 1;
        int64_t total = n_stream * nwin;
        FAB_CUDA(ctx, cudaMemsetAsync(frame_flag, 0, fflag_b, st));
        TP.D = P; TP.j0 = first_decode / bsh; TP.nwin = nwin; TP.frame_flag = frame_flag;
        TP.restore = fuse_restore ? 1 : 0; TP.offsets = (const float*)d_offsets; TP.gains = (const float*)d_gains;
        TP.W = WinParams{};
        int rc2 = store ? dec_items<false>(ctx, TP, total, st) : dec_items<false, false>(ctx, TP, total, st);
        if (rc2) return rc2;
    }
    if (d_status) k_dec_walker_iso<<<(unsigned)((n_stream + 31) / 32), 32, 0, st>>>(P);
    else k_dec_walker<<<(unsigned)((n_stream + 31) / 32), 32, 0, st>>>(P);
    ctx->launches++;

    if (fuse_restore) {
        for (int64_t s0 = 0; s0 < n_stream; s0 += 65535) {
            int64_t ns = std::min<int64_t>(65535, n_stream - s0);
            TileParams Q = TP;
            Q.D.starts += s0; Q.D.nbytes += s0; Q.D.meta += s0; Q.D.frame_off += s0 * (int64_t)(nframes_cap + 1);
            Q.D.stream_flag += s0; Q.D.data += s0 * n_decode; Q.D.n_sel = ns;
            Q.frame_flag += s0 * (int64_t)nframes_cap; Q.offsets += s0; Q.gains += s0;
            // x: 256 frames per CTA pass; walker-decoded streams (rare) spread their samples over x too
            dim3 grid((unsigned)std::min<int64_t>((TP.nwin + 255) / 256 + 3, 64), (unsigned)ns);
            k_restore_fixup<<<grid, 256, 0, st>>>(Q);
            ctx->launches++;
        }
    } else if (d_offsets && d_gains) {
        int64_t per_cta = 256 * 16;
        int64_t gx = (n_decode + per_cta - 1) / per_cta;
        for (int64_t s0 = 0; s0 < n_stream; s0 += 65535) {
            int64_t ns = std::min<int64_t>(65535, n_stream - s0);
            dim3 grid((unsigned)gx, (unsigned)ns);
            k_restore<long long, double><<<grid, 256, 0, st>>>((const long long*)d_out + s0 * n_decode, n_decode, per_cta,
                                                               (const double*)d_offsets + s0, (const double*)d_gains + s0,
                                                               (double*)d_out + s0 * n_decode);
            ctx->launches++;
        }
    }
    if (d_status && store) {
        // a few CTAs per stream: those of good streams leave at once, the rare failed row is strided over
        const bool flt = d_offsets && d_gains;
        const int64_t gx = std::min<int64_t>((n_decode + 2047) / 2048, 16);
        for (int64_t s0 = 0; s0 < n_stream; s0 += 65535) {
            int64_t ns = std::min<int64_t>(65535, n_stream - s0);
            dim3 grid((unsigned)gx, (unsigned)ns);
            if (is_int64)
                k_dec_fill_failed<unsigned long long><<<grid, 256, 0, st>>>(
                    d_status + s0, (unsigned long long*)d_out + s0 * n_decode, n_decode, flt ? 0x7FF8000000000000ull : 0ull);
            else
                k_dec_fill_failed<uint32_t><<<grid, 256, 0, st>>>(d_status + s0, (uint32_t*)d_out + s0 * n_decode, n_decode,
                                                                  flt ? 0x7FC00000u : 0u);
            ctx->launches++;
        }
    }
    FAB_CUDA(ctx, cudaGetLastError());
    return 0;
}

extern "C" int fab_decode(fab_ctx* ctx, const unsigned char* d_bytes, const int64_t* d_starts, const int64_t* d_nbytes,
                          int64_t n_stream, int64_t stream_size, int is_int64, int64_t first_sample, int64_t last_sample,
                          void* d_out, const void* d_offsets, const void* d_gains, int64_t max_nbytes,
                          int blocksize_hint, void* stream) {
    return dec_uniform(ctx, d_bytes, d_starts, d_nbytes, n_stream, stream_size, is_int64, first_sample, last_sample, d_out,
                       d_offsets, d_gains, max_nbytes, blocksize_hint, nullptr, true, stream);
}

extern "C" int fab_decode_isolated(fab_ctx* ctx, const unsigned char* d_bytes, const int64_t* d_starts,
                                   const int64_t* d_nbytes, int64_t n_stream, int64_t stream_size, int is_int64,
                                   int64_t first_sample, int64_t last_sample, void* d_out, const void* d_offsets,
                                   const void* d_gains, int64_t max_nbytes, int blocksize_hint, int32_t* d_status,
                                   void* stream) {
    return dec_uniform(ctx, d_bytes, d_starts, d_nbytes, n_stream, stream_size, is_int64, first_sample, last_sample, d_out,
                       d_offsets, d_gains, max_nbytes, blocksize_hint, d_status, true, stream);
}

extern "C" int fab_verify(fab_ctx* ctx, const unsigned char* d_bytes, const int64_t* d_starts, const int64_t* d_nbytes,
                          int64_t n_stream, int64_t stream_size, int is_int64, int64_t max_nbytes, int blocksize_hint,
                          int32_t* d_status, void* stream) {
    if (!ctx) return FAB_ERROR_CUDA;
    if (!d_status) {            // (the walker's discard mode reports through the status array only)
        ctx->last_error = "fab_verify: d_status must not be NULL";
        return ERROR_ALLOC;
    }
    return dec_uniform(ctx, d_bytes, d_starts, d_nbytes, n_stream, stream_size, is_int64, -1, -1, nullptr, nullptr, nullptr,
                       max_nbytes, blocksize_hint, d_status, false, stream);
}

// Workspace of one fab_decode_windows call: fab_decode's layout for the stream slots | item0 of the windows.  The item
// space itself needs no storage (frame flags are kept per stream slot and frame), so total_items does not change it.
static size_t win_item0_bytes(int64_t n_win) { return align256((size_t)(n_win + 1) * 8); }
extern "C" int64_t fab_decode_windows_workspace_bytes(int64_t n_stream, int64_t stream_size, int64_t n_win,
                                                      int64_t total_items, int blocksize_hint) {
    int bsh = 0, cap = 0;
    if (n_stream <= 0 || stream_size <= 0 || n_win < 0 || total_items < 0 ||
        dec_frames_cap(stream_size, blocksize_hint, &bsh, &cap))
        return 0;
    return (int64_t)(dec_workspace(n_stream, cap).total + win_item0_bytes(n_win));
}

extern "C" int fab_decode_windows(fab_ctx* ctx, const unsigned char* d_bytes, const int64_t* d_starts, const int64_t* d_nbytes,
                                  int64_t n_stream, int64_t stream_size, int is_int64, const int64_t* d_win_stream,
                                  const int64_t* d_win_first, const int64_t* d_win_last, const int64_t* d_win_out,
                                  int64_t n_win, void* d_out, const void* d_offsets, const void* d_gains, int64_t max_nbytes,
                                  int blocksize_hint, void* stream) {
    if (!ctx) return FAB_ERROR_CUDA;
    if (n_win < 0) return ERROR_DECODE_SAMPLE_RANGE;
    if (n_win == 0) return 0;
    if (n_stream <= 0) return ERROR_ZERO_NSTREAM;
    if (stream_size <= 0) return ERROR_ZERO_STREAMSIZE;
    cudaStream_t st = (cudaStream_t)stream;
    const int nch = is_int64 ? 2 : 1;
    int bsh = 0, nframes_cap = 0;
    if (dec_frames_cap(stream_size, blocksize_hint, &bsh, &nframes_cap)) return ERROR_ALLOC;

    const DecWorkspace DW = dec_workspace(n_stream, nframes_cap);
    unsigned char* scr;
    int rc = ctx_scratch(ctx, DW.total + win_item0_bytes(n_win), &scr, st);
    if (rc) return rc;
    unsigned char* frame_flag = scr + DW.meta_b + DW.fo_b + DW.flag_b;
    long long* d_max = (long long*)(frame_flag + DW.fflag_b);

    WinParams W;
    W.stream = (const long long*)d_win_stream; W.first = (const long long*)d_win_first; W.last = (const long long*)d_win_last;
    W.out = (const long long*)d_win_out; W.item0 = (const long long*)(scr + DW.total); W.n_win = n_win; W.bsh = bsh;
    k_win_prep<<<1, kWinScanThreads, 0, st>>>(W, n_stream, stream_size, ctx->d_err);
    ctx->launches++;
    // the grids are sized by the number of items: one round trip for it (and for the longest stream when not given)
    long long h_total = 0, h_max = 0;
    if (max_nbytes <= 0) {
        k_max_i64<<<1, 256, 0, st>>>((const long long*)d_nbytes, n_stream, d_max);
        ctx->launches++;
        FAB_CUDA(ctx, cudaMemcpyAsync(&h_max, d_max, 8, cudaMemcpyDeviceToHost, st));
    }
    FAB_CUDA(ctx, cudaMemcpyAsync(&h_total, W.item0 + n_win, 8, cudaMemcpyDeviceToHost, st));
    FAB_CUDA(ctx, cudaStreamSynchronize(st));
    if (max_nbytes <= 0) max_nbytes = h_max;
    const int64_t total = h_total;
    if (total == 0) {           // every window empty (or rejected: the error mask says so)
        FAB_CUDA(ctx, cudaGetLastError());
        return 0;
    }

    DecParams P;
    P.bytes = d_bytes; P.starts = (const long long*)d_starts; P.nbytes = (const long long*)d_nbytes;
    P.n_sel = n_stream; P.stream_size = stream_size; P.nch = nch;
    P.first = 0; P.n_decode = 0; P.data = (int32_t*)d_out; P.crc = ctx->d_crc;      // (windows carry their own ranges)
    P.meta = (StreamMeta*)scr; P.frame_off = (long long*)(scr + DW.meta_b); P.nframes_cap = nframes_cap;
    P.stream_flag = (int*)(scr + DW.meta_b + DW.fo_b); P.err = ctx->d_err; P.verify_crc16 = 1; P.frame_flag = frame_flag;
    dec_index_streams(ctx, P, max_nbytes, st);

    const bool fuse_restore = d_offsets && d_gains && !is_int64;
    TileParams TP;
    FAB_CUDA(ctx, cudaMemsetAsync(frame_flag, 0, DW.fflag_b, st));
    TP.D = P; TP.j0 = 0; TP.nwin = 0; TP.frame_flag = frame_flag;
    TP.restore = fuse_restore ? 1 : 0; TP.offsets = (const float*)d_offsets; TP.gains = (const float*)d_gains;
    TP.W = W;
    rc = dec_items<true>(ctx, TP, total, st);
    if (rc) return rc;
    k_dec_walker_win<<<(unsigned)((n_win + 127) / 128), 128, 0, st>>>(P, W);
    ctx->launches++;
    if (d_offsets && d_gains) {
        if (fuse_restore) k_restore_win<false><<<(unsigned)((total + 3) / 4), 128, 0, st>>>(TP, total);
        else k_restore_win<true><<<(unsigned)((total + 3) / 4), 128, 0, st>>>(TP, total);
        ctx->launches++;
    }
    FAB_CUDA(ctx, cudaGetLastError());
    return 0;
}

// =================================================================================================
// Per-row, per-bin statistics of decoded integer rows
// =================================================================================================
static size_t stats_workspace(const StatsParams& P) {
    return P.ppb > 1 ? align256((size_t)P.n_rows * (size_t)P.nbins * (size_t)P.ppb * sizeof(StatPart)) : 0;
}

extern "C" int64_t fab_row_stats_workspace_bytes(int64_t n_rows, int64_t n, int64_t bin, int is_int64) {
    StatsParams P{};
    if (stats_geometry(n_rows, n, bin, is_int64, &P)) return -1;
    return (int64_t)stats_workspace(P);
}

extern "C" int fab_row_stats(fab_ctx* ctx, const void* d_rows, int is_int64, int64_t n_rows, int64_t n, int64_t bin,
                             const void* d_offsets, const void* d_gains, const int32_t* d_status, int64_t* d_count,
                             void* d_min, void* d_max, double* d_mean, double* d_std, void* stream) {
    if (!ctx) return FAB_ERROR_CUDA;
    StatsParams P{};
    int rc = stats_geometry(n_rows, n, bin, is_int64, &P);
    if (rc) return rc;
    if ((d_offsets == nullptr) != (d_gains == nullptr) || ((uintptr_t)d_rows & (is_int64 ? 7 : 3)) != 0) {
        ctx->last_error = "fab_row_stats: offsets and gains go together, and d_rows must be aligned to its element size";
        return ERROR_CONVERT_TYPE;
    }
    if (!d_rows || !d_count || !d_min || !d_max || !d_mean || !d_std) {
        ctx->last_error = "fab_row_stats: d_rows and the five result arrays must not be NULL";
        return ERROR_ALLOC;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const size_t ws = stats_workspace(P);
    if (ws) {
        unsigned char* scr;
        rc = ctx_scratch(ctx, ws, &scr, st);
        if (rc) return rc;
        P.part = (StatPart*)scr;
    }
    P.rows = d_rows; P.offsets = d_offsets; P.gains = d_gains; P.status = d_status;
    P.count = (long long*)d_count; P.mn = d_min; P.mx = d_max; P.mean = d_mean; P.std = d_std;
    const unsigned gx = (unsigned)((P.nbins * P.ppb + kStatsWarps - 1) / kStatsWarps);
    const unsigned gm = (unsigned)((P.nbins + kStatsWarps - 1) / kStatsWarps);
    for (int64_t r0 = 0; r0 < n_rows; r0 += 65535) {
        const dim3 grid(gx, (unsigned)std::min<int64_t>(65535, n_rows - r0));
        if (is_int64) k_row_stats<true><<<grid, kStatsWarps * 32, 0, st>>>(P, r0);
        else k_row_stats<false><<<grid, kStatsWarps * 32, 0, st>>>(P, r0);
        ctx->launches++;
        if (P.ppb > 1) {
            k_row_stats_merge<<<dim3(gm, grid.y), kStatsWarps * 32, 0, st>>>(P, r0);
            ctx->launches++;
        }
    }
    FAB_CUDA(ctx, cudaGetLastError());
    return 0;
}

// =================================================================================================
// Per-sample weighted sums across decoded integer rows
// =================================================================================================
extern "C" int fab_combine_rows(fab_ctx* ctx, const void* d_rows, int is_int64, int64_t n_rows, int64_t n,
                                const void* d_offsets, const void* d_gains, const int32_t* d_status,
                                const double* d_weights, const int64_t* d_seg, const int64_t* d_seg_out, int64_t n_seg,
                                double* d_out, int64_t n_out, void* stream) {
    if (!ctx) return FAB_ERROR_CUDA;
    if (n_rows <= 0 || n_seg <= 0 || n_out <= 0) return ERROR_ZERO_NSTREAM;
    if (n <= 0) return ERROR_ZERO_STREAMSIZE;
    if (!d_rows || !d_weights || !d_seg || !d_seg_out || !d_out) {
        ctx->last_error = "fab_combine_rows: d_rows, d_weights, d_seg, d_seg_out and d_out must not be NULL";
        return ERROR_ALLOC;
    }
    if ((d_offsets == nullptr) != (d_gains == nullptr) || ((uintptr_t)d_rows & (is_int64 ? 7 : 3)) != 0 ||
        (((uintptr_t)d_weights | (uintptr_t)d_seg | (uintptr_t)d_seg_out | (uintptr_t)d_out) & 7) != 0) {
        ctx->last_error = "fab_combine_rows: offsets and gains go together, and every array must be aligned to its "
                          "element size";
        return ERROR_CONVERT_TYPE;
    }
    const int64_t gx = (n + kCombineThreads * kCombineCols - 1) / (kCombineThreads * kCombineCols);
    if (gx > 0x7FFFFFFFll) return ERROR_ALLOC;
    CombineParams P{};
    P.rows = d_rows; P.n_rows = n_rows; P.n = n;
    P.offsets = d_offsets; P.gains = d_gains; P.status = d_status; P.weights = d_weights;
    P.seg = (const int64_t*)d_seg; P.seg_out = (const int64_t*)d_seg_out; P.n_seg = n_seg;
    P.out = d_out; P.n_out = n_out; P.err = ctx->d_err;
    cudaStream_t st = (cudaStream_t)stream;
    const bool flt = d_offsets != nullptr;
    for (int64_t s0 = 0; s0 < n_seg; s0 += 65535) {
        const dim3 grid((unsigned)gx, (unsigned)std::min<int64_t>(65535, n_seg - s0));
        if (is_int64) {
            if (flt) k_combine_rows<true, true><<<grid, kCombineThreads, 0, st>>>(P, s0);
            else k_combine_rows<true, false><<<grid, kCombineThreads, 0, st>>>(P, s0);
        } else {
            if (flt) k_combine_rows<false, true><<<grid, kCombineThreads, 0, st>>>(P, s0);
            else k_combine_rows<false, false><<<grid, kCombineThreads, 0, st>>>(P, s0);
        }
        ctx->launches++;
    }
    FAB_CUDA(ctx, cudaGetLastError());
    return 0;
}

// =================================================================================================
// Converters
// =================================================================================================
template <typename T>
static int launch_stream_std(fab_ctx* ctx, const T* d_in, int64_t n_stream, int64_t stream_size, T* d_std, cudaStream_t st) {
    int nchunk = (int)((stream_size + kMmChunk - 1) / kMmChunk);
    unsigned char* scr;
    const size_t part = align256((size_t)n_stream * nchunk * sizeof(double));
    int rc = ctx_scratch(ctx, 2 * part, &scr, st);
    if (rc) return rc;
    double* pmean = (double*)scr;
    double* pm2 = (double*)(scr + part);
    for (int64_t s0 = 0; s0 < n_stream; s0 += 65535) {
        int64_t ns = std::min<int64_t>(65535, n_stream - s0);
        dim3 grid((unsigned)nchunk, (unsigned)ns);
        k_moments<T><<<grid, kMmThreads, 0, st>>>(d_in + s0 * stream_size, stream_size, nchunk, pmean + s0 * nchunk, pm2 + s0 * nchunk);
        ctx->launches++;
    }
    k_std_final<T><<<(unsigned)((n_stream + 127) / 128), 128, 0, st>>>(pmean, pm2, nchunk, stream_size, n_stream, d_std);
    ctx->launches++;
    FAB_CUDA(ctx, cudaGetLastError());
    return 0;
}

extern "C" int fab_stream_std(fab_ctx* ctx, const void* d_input, int dtype, int64_t n_stream, int64_t stream_size,
                              void* d_std, void* stream) {
    if (!ctx) return FAB_ERROR_CUDA;
    if (n_stream == 0) return ERROR_ZERO_NSTREAM;
    if (stream_size == 0) return ERROR_ZERO_STREAMSIZE;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == FAB_F32) return launch_stream_std<float>(ctx, (const float*)d_input, n_stream, stream_size, (float*)d_std, st);
    if (dtype == FAB_F64) return launch_stream_std<double>(ctx, (const double*)d_input, n_stream, stream_size, (double*)d_std, st);
    return ERROR_CONVERT_TYPE;
}

extern "C" int fab_float_to_int(fab_ctx* ctx, const void* d_input, int dtype, int64_t n_stream, int64_t stream_size,
                                const void* d_quanta, void* d_output, void* d_offsets, void* d_gains, void* stream) {
    if (!ctx) return FAB_ERROR_CUDA;
    if (n_stream <= 0) return ERROR_ZERO_NSTREAM;
    if (stream_size <= 0) return ERROR_ZERO_STREAMSIZE;
    cudaStream_t st = (cudaStream_t)stream;
    int64_t per_cta = 256 * 16;
    int64_t gx = (stream_size + per_cta - 1) / per_cta;
    if (dtype == FAB_F32) {
        int rc = launch_quant_params<float>(ctx, (const float*)d_input, n_stream, stream_size, (const float*)d_quanta,
                                            (float*)d_offsets, (float*)d_gains, st);
        if (rc) return rc;
        for (int64_t s0 = 0; s0 < n_stream; s0 += 65535) {
            dim3 grid((unsigned)gx, (unsigned)std::min<int64_t>(65535, n_stream - s0));
            k_quantise<float, int32_t><<<grid, 256, 0, st>>>((const float*)d_input + s0 * stream_size, stream_size, per_cta,
                                                             (const float*)d_offsets + s0, (const float*)d_gains + s0,
                                                             (int32_t*)d_output + s0 * stream_size);
            ctx->launches++;
        }
    } else if (dtype == FAB_F64) {
        int rc = launch_quant_params<double>(ctx, (const double*)d_input, n_stream, stream_size, (const double*)d_quanta,
                                             (double*)d_offsets, (double*)d_gains, st);
        if (rc) return rc;
        for (int64_t s0 = 0; s0 < n_stream; s0 += 65535) {
            dim3 grid((unsigned)gx, (unsigned)std::min<int64_t>(65535, n_stream - s0));
            k_quantise<double, long long><<<grid, 256, 0, st>>>((const double*)d_input + s0 * stream_size, stream_size, per_cta,
                                                                (const double*)d_offsets + s0, (const double*)d_gains + s0,
                                                                (long long*)d_output + s0 * stream_size);
            ctx->launches++;
        }
    } else {
        return ERROR_CONVERT_TYPE;
    }
    FAB_CUDA(ctx, cudaGetLastError());
    return 0;
}

extern "C" int fab_int_to_float(fab_ctx* ctx, const void* d_input, int dtype, int64_t n_stream, int64_t stream_size,
                                const void* d_offsets, const void* d_gains, void* d_output, void* stream) {
    if (!ctx) return FAB_ERROR_CUDA;
    if (n_stream <= 0) return ERROR_ZERO_NSTREAM;
    if (stream_size <= 0) return ERROR_ZERO_STREAMSIZE;
    cudaStream_t st = (cudaStream_t)stream;
    int64_t per_cta = 256 * 16;
    int64_t gx = (stream_size + per_cta - 1) / per_cta;
    for (int64_t s0 = 0; s0 < n_stream; s0 += 65535) {
        dim3 grid((unsigned)gx, (unsigned)std::min<int64_t>(65535, n_stream - s0));
        if (dtype == FAB_I32)
            k_restore<int32_t, float><<<grid, 256, 0, st>>>((const int32_t*)d_input + s0 * stream_size, stream_size, per_cta,
                                                            (const float*)d_offsets + s0, (const float*)d_gains + s0,
                                                            (float*)d_output + s0 * stream_size);
        else if (dtype == FAB_I64)
            k_restore<long long, double><<<grid, 256, 0, st>>>((const long long*)d_input + s0 * stream_size, stream_size, per_cta,
                                                               (const double*)d_offsets + s0, (const double*)d_gains + s0,
                                                               (double*)d_output + s0 * stream_size);
        else
            return ERROR_CONVERT_TYPE;
        ctx->launches++;
    }
    FAB_CUDA(ctx, cudaGetLastError());
    return 0;
}

// =================================================================================================
// Reference-compatible host-buffer entry points (flacarray.h:209-311)
// =================================================================================================
namespace {

struct DevBuf {
    void* p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
    bool alloc(size_t n) { return cudaMalloc(&p, n ? n : 1) == cudaSuccess; }
};

// ---- large host buffers: chunks of whole streams through pinned staging buffers -------------------------
// The caller's arrays are pageable (malloc / numpy): a cudaMemcpy straight from them runs at a fraction of
// the link rate.  Chunk c+1 is copied into pinned memory by a few host threads and uploaded while the
// kernels work on chunk c and chunk c-1 is copied out.  Buffers, streams and events persist between calls.
constexpr size_t kPipeChunk = (size_t)128 << 20;   // raw bytes per chunk
constexpr size_t kPipeMin = (size_t)64 << 20;      // smaller calls take the plain path below

struct HostPipe {
    bool ready = false;
    void* pin_in[2] = {nullptr, nullptr};
    void* pin_out[2] = {nullptr, nullptr};
    size_t pin_in_b = 0, pin_out_b = 0;
    cudaStream_t s_in = nullptr, s_k = nullptr, s_out = nullptr;
    cudaEvent_t ev_in[2], ev_k[2], ev_out[2];

    bool init() {
        if (ready) return true;
        if (cudaStreamCreateWithFlags(&s_in, cudaStreamNonBlocking) != cudaSuccess) return false;
        if (cudaStreamCreateWithFlags(&s_k, cudaStreamNonBlocking) != cudaSuccess) return false;
        if (cudaStreamCreateWithFlags(&s_out, cudaStreamNonBlocking) != cudaSuccess) return false;
        for (int i = 0; i < 2; ++i) {
            if (cudaEventCreateWithFlags(&ev_in[i], cudaEventDisableTiming) != cudaSuccess) return false;
            if (cudaEventCreateWithFlags(&ev_k[i], cudaEventDisableTiming) != cudaSuccess) return false;
            if (cudaEventCreateWithFlags(&ev_out[i], cudaEventDisableTiming) != cudaSuccess) return false;
        }
        ready = true;
        return true;
    }
    static bool grow(void* buf[2], size_t& have, size_t want) {
        if (want <= have) return true;
        for (int i = 0; i < 2; ++i) {
            if (buf[i]) cudaFreeHost(buf[i]);
            buf[i] = nullptr;
        }
        have = 0;
        for (int i = 0; i < 2; ++i)
            if (cudaHostAlloc(&buf[i], want, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return false; }
        have = want;
        return true;
    }
    // device-side chunk buffers (input side, output side, per-stream tables), grow-only like the pinned ones
    void* dev_in[2] = {nullptr, nullptr};
    void* dev_out[2] = {nullptr, nullptr};
    void* dev_aux[2] = {nullptr, nullptr};
    size_t dev_in_b = 0, dev_out_b = 0, dev_aux_b = 0;
    static bool grow_dev(void* buf[2], size_t& have, size_t want) {
        if (want <= have) return true;
        for (int i = 0; i < 2; ++i) {
            if (buf[i]) cudaFree(buf[i]);
            buf[i] = nullptr;
        }
        have = 0;
        for (int i = 0; i < 2; ++i)
            if (cudaMalloc(&buf[i], want) != cudaSuccess) { cudaGetLastError(); return false; }
        have = want;
        return true;
    }
    bool reserve(size_t in_b, size_t out_b, size_t aux_b) {
        return init() && grow(pin_in, pin_in_b, in_b) && grow(pin_out, pin_out_b, out_b) && grow_dev(dev_in, dev_in_b, in_b) &&
               grow_dev(dev_out, dev_out_b, out_b) && grow_dev(dev_aux, dev_aux_b, aux_b);
    }
    void drain() { cudaStreamSynchronize(s_in); cudaStreamSynchronize(s_k); cudaStreamSynchronize(s_out); }
};

// The reference's entry points are re-entrant (each call owns its libFLAC encoder / decoder objects).  Here a call
// leases one of a few host slots -- a context (streams, scratch, size history) plus the pinned / device staging
// buffers of the chunked pipeline -- so concurrent callers run side by side on separate CUDA streams instead of
// queueing on one lock.  Slots are created on demand up to kHostSlots (FLACARRAY_B200_HOST_SLOTS, 1..16); callers
// beyond that wait for a slot to come back.
struct HostSlot {
    fab_ctx* ctx = nullptr;
    HostPipe pipe;
    bool busy = false;
};
std::mutex g_slot_mu;
std::condition_variable g_slot_cv;
std::vector<HostSlot*> g_slots;
int host_slot_limit() {
    static const int lim = [] {
        const char* e = getenv("FLACARRAY_B200_HOST_SLOTS");
        int v = e ? atoi(e) : 4;
        return v < 1 ? 1 : (v > 16 ? 16 : v);
    }();
    return lim;
}
class SlotLease {
    HostSlot* s_ = nullptr;
public:
    SlotLease() {
        std::unique_lock<std::mutex> lk(g_slot_mu);
        for (;;) {
            for (HostSlot* c : g_slots)
                if (!c->busy) { s_ = c; break; }
            if (s_) break;
            if ((int)g_slots.size() < host_slot_limit()) {
                HostSlot* c = new HostSlot();
                if (fab_create(&c->ctx) != 0) { delete c; return; }     // no CUDA device: the caller reports FAB_ERROR_CUDA
                g_slots.push_back(c);
                s_ = c;
                break;
            }
            g_slot_cv.wait(lk);
        }
        s_->busy = true;
    }
    ~SlotLease() {
        if (!s_) return;
        {
            std::lock_guard<std::mutex> lk(g_slot_mu);
            s_->busy = false;
        }
        g_slot_cv.notify_one();
    }
    SlotLease(const SlotLease&) = delete;
    SlotLease& operator=(const SlotLease&) = delete;
    fab_ctx* ctx() const { return s_ ? s_->ctx : nullptr; }
    HostPipe& pipe() const { return s_->pipe; }
};
// measurement switch: FLACARRAY_B200_NO_PIPE=1 sends every call down the plain (unpipelined) path
bool pipe_enabled() {
    static const bool off = [] { const char* e = getenv("FLACARRAY_B200_NO_PIPE"); return e && e[0] == '1'; }();
    return !off;
}

// memcpy split over a few threads (one core moves ~10 GB/s, the PCIe link 55)
void par_memcpy(void* dst, const void* src, size_t n) {
    const unsigned hw = std::thread::hardware_concurrency();
    const size_t nt = std::min<size_t>(std::max(1u, std::min(hw, 16u)), n / ((size_t)4 << 20) + 1);
    if (nt <= 1) { memcpy(dst, src, n); return; }
    const size_t step = (((n + nt - 1) / nt) + 4095) & ~(size_t)4095;
    std::vector<std::thread> th;
    for (size_t o = step; o < n; o += step)
        th.emplace_back([=] { memcpy((char*)dst + o, (const char*)src + o, std::min(step, n - o)); });
    memcpy(dst, src, std::min(step, n));
    for (auto& t : th) t.join();
}

struct PipeClock {   // FLACARRAY_B200_PIPE_DEBUG=1: phase times of the pipelined entry points on stderr
    bool on;
    double acc[6] = {0, 0, 0, 0, 0, 0};
    std::chrono::steady_clock::time_point t0;
    PipeClock() : on(getenv("FLACARRAY_B200_PIPE_DEBUG") != nullptr), t0(std::chrono::steady_clock::now()) {}
    void lap(int k) {
        if (!on) return;
        auto t = std::chrono::steady_clock::now();
        acc[k] += std::chrono::duration<double, std::milli>(t - t0).count();
        t0 = t;
    }
    void report(const char* what) {
        if (on) fprintf(stderr, "%s: setup %.1f ms, stage-in %.1f, launch+finish %.1f, copy-out %.1f, tail %.1f\n", what, acc[0], acc[1], acc[2], acc[3], acc[4]);
    }
};

#define PIPE_CUDA(expr)                                    \
    do {                                                   \
        if ((expr) != cudaSuccess) {                       \
            cudaGetLastError();                            \
            rc = FAB_ERROR_CUDA;                           \
            goto done;                                     \
        }                                                  \
    } while (0)

int host_encode_pipelined(fab_ctx* ctx, HostPipe& hp, const void* data, int dtype, int64_t n_stream, int64_t stream_size, uint32_t level,
                          int64_t* n_bytes, int64_t* starts, unsigned char** bytes) {
    PipeClock clk;
    const size_t stream_b = (size_t)stream_size * (dtype == FAB_I64 ? 8 : 4);
    const int64_t per = std::max<int64_t>(1, (int64_t)(kPipeChunk / stream_b));
    const int64_t nchunk = (n_stream + per - 1) / per;
    const int64_t bound_c = fab_encode_bound(per, stream_size, dtype, level);
    const int64_t bound_all = fab_encode_bound(n_stream, stream_size, dtype, level);
    if (!hp.reserve((size_t)per * stream_b, (size_t)bound_c, (size_t)per * 16 + 64)) return ERROR_ALLOC | FAB_ERROR_CUDA;
    struct { void* p; } d_in[2] = {{hp.dev_in[0]}, {hp.dev_in[1]}}, d_out[2] = {{hp.dev_out[0]}, {hp.dev_out[1]}},
                        d_aux[2] = {{hp.dev_aux[0]}, {hp.dev_aux[1]}};
    std::thread drainer;                 // copies chunk c-2 out of pinned memory while chunk c is staged
    std::atomic<int> drain_err{0};
    // worst-case size, untouched pages cost nothing; shrunk to the real size at the end
    unsigned char* hb = (unsigned char*)malloc((size_t)bound_all);
    if (!hb) return ERROR_ALLOC;
    std::vector<int64_t> tot((size_t)nchunk, 0), pos((size_t)nchunk + 1, 0);
    int rc = 0;
    clk.lap(0);
    for (int64_t c = 0; c < nchunk + 2; ++c) {
        if (c >= 2) {                                       // chunk c-2: pinned -> caller's buffer, on a helper thread
            const int64_t e = c - 2;
            const int b = (int)(e & 1);
            unsigned char* dst = hb + pos[(size_t)e];
            const size_t nb_e = (size_t)tot[(size_t)e];
            cudaEvent_t ev = hp.ev_out[b];
            const void* src = hp.pin_out[b];
            drainer = std::thread([=, &drain_err] {
                if (cudaEventSynchronize(ev) != cudaSuccess) { drain_err = 1; return; }
                par_memcpy(dst, src, nb_e);
            });
        }
        if (c < nchunk) {                                   // stage and upload chunk c
            const int b = (int)(c & 1);
            const int64_t s0 = c * per, ns = std::min(per, n_stream - s0);
            if (c >= 2) PIPE_CUDA(cudaEventSynchronize(hp.ev_in[b]));           // pinned buffer b is free again
            par_memcpy(hp.pin_in[b], (const char*)data + (size_t)s0 * stream_b, (size_t)ns * stream_b);
            if (c >= 2) PIPE_CUDA(cudaStreamWaitEvent(hp.s_in, hp.ev_k[b], 0));  // encode c-2 has read d_in[b]
            PIPE_CUDA(cudaMemcpyAsync(d_in[b].p, hp.pin_in[b], (size_t)ns * stream_b, cudaMemcpyHostToDevice, hp.s_in));
            PIPE_CUDA(cudaEventRecord(hp.ev_in[b], hp.s_in));
            clk.lap(1);
        }
        if (c >= 1 && c - 1 < nchunk) {                     // encode chunk c-1, start its download
            const int64_t e = c - 1;
            const int b = (int)(e & 1);
            const int64_t s0 = e * per, ns = std::min(per, n_stream - s0);
            int64_t* d_starts = (int64_t*)d_aux[b].p;
            int64_t* d_nb = d_starts + per;
            int64_t* d_total = d_nb + per;
            PIPE_CUDA(cudaStreamWaitEvent(hp.s_k, hp.ev_in[b], 0));
            if (e >= 2) PIPE_CUDA(cudaStreamWaitEvent(hp.s_k, hp.ev_out[b], 0));  // download e-2 has read d_out[b]
            rc = fab_encode(ctx, d_in[b].p, dtype, ns, stream_size, level, nullptr, nullptr, nullptr,
                            (unsigned char*)d_out[b].p, bound_c, d_starts, d_nb, d_total, hp.s_k);
            if (rc) goto done;
            PIPE_CUDA(cudaEventRecord(hp.ev_k[b], hp.s_k));
            rc = fab_finish(ctx, hp.s_k);
            if (rc) goto done;
            int64_t total = 0;
            PIPE_CUDA(cudaMemcpyAsync(&total, d_total, 8, cudaMemcpyDeviceToHost, hp.s_k));
            PIPE_CUDA(cudaMemcpyAsync(starts + s0, d_starts, (size_t)ns * 8, cudaMemcpyDeviceToHost, hp.s_k));
            PIPE_CUDA(cudaStreamSynchronize(hp.s_k));
            tot[(size_t)e] = total;
            pos[(size_t)e + 1] = pos[(size_t)e] + total;
            for (int64_t i = 0; i < ns; ++i) starts[s0 + i] += pos[(size_t)e];
            // pinned buffer b was emptied by the helper thread of the previous iteration (joined below)
            PIPE_CUDA(cudaMemcpyAsync(hp.pin_out[b], d_out[b].p, (size_t)total, cudaMemcpyDeviceToHost, hp.s_out));
            PIPE_CUDA(cudaEventRecord(hp.ev_out[b], hp.s_out));
            clk.lap(2);
        }
        if (drainer.joinable()) drainer.join();
        if (drain_err) { rc = FAB_ERROR_CUDA; goto done; }
        clk.lap(3);
    }
done:
    if (drainer.joinable()) drainer.join();
    if (rc) {
        hp.drain();
        free(hb);
        return rc;
    }
    {
        const int64_t total = pos[(size_t)nchunk];
        unsigned char* shrunk = (unsigned char*)realloc(hb, (size_t)std::max<int64_t>(total, 1));
        *bytes = shrunk ? shrunk : hb;
        *n_bytes = total;
    }
    clk.lap(4);
    clk.report("host_encode_pipelined");
    return ERROR_NONE;
}

int host_decode_pipelined(fab_ctx* ctx, HostPipe& hp, const unsigned char* bytes, const int64_t* starts, const int64_t* nbytes,
                          int64_t n_stream, int64_t stream_size, int is_int64, int64_t first, int64_t last, int64_t n_decode,
                          void* data, bool* handled) {
    *handled = false;
    const size_t row_b = (size_t)n_decode * (is_int64 ? 8 : 4);
    const int64_t per = std::max<int64_t>(1, (int64_t)(kPipeChunk / row_b));
    const int64_t nchunk = (n_stream + per - 1) / per;
    // byte range covering each chunk's streams (they may be scattered when the caller selected streams)
    std::vector<int64_t> lo((size_t)nchunk), hi((size_t)nchunk), mx((size_t)nchunk);
    int64_t max_in = 0;
    for (int64_t c = 0; c < nchunk; ++c) {
        int64_t l = INT64_MAX, h = 0, m = 0;
        for (int64_t i = c * per; i < std::min(n_stream, (c + 1) * per); ++i) {
            l = std::min(l, starts[i]);
            h = std::max(h, starts[i] + nbytes[i]);
            m = std::max(m, nbytes[i]);
        }
        lo[(size_t)c] = l; hi[(size_t)c] = h; mx[(size_t)c] = m;
        max_in = std::max(max_in, h - l);
    }
    if ((size_t)max_in > 2 * kPipeChunk) return 0;          // widely scattered selection: plain path
    *handled = true;
    if (!hp.reserve((size_t)std::max<int64_t>(max_in, 1), (size_t)per * row_b, (size_t)per * 16)) return ERROR_ALLOC | FAB_ERROR_CUDA;
    struct { void* p; } d_b[2] = {{hp.dev_in[0]}, {hp.dev_in[1]}}, d_o[2] = {{hp.dev_out[0]}, {hp.dev_out[1]}},
                        d_aux[2] = {{hp.dev_aux[0]}, {hp.dev_aux[1]}};
    std::thread drainer;                 // copies chunk c-2 out of pinned memory while chunk c is staged
    std::atomic<int> drain_err{0};
    const int bs_hint = stream_blocksize_hint(bytes + starts[0], nbytes[0]);
    std::vector<int64_t> rel[2];
    int rc = 0;
    for (int64_t c = 0; c < nchunk + 2; ++c) {
        if (c >= 2) {                                       // chunk c-2: pinned -> caller's buffer, on a helper thread
            const int64_t e = c - 2;
            const int b = (int)(e & 1);
            const int64_t s0 = e * per, ns = std::min(per, n_stream - s0);
            char* dst = (char*)data + (size_t)s0 * row_b;
            const size_t nb_e = (size_t)ns * row_b;
            cudaEvent_t ev = hp.ev_out[b];
            const void* src = hp.pin_out[b];
            drainer = std::thread([=, &drain_err] {
                if (cudaEventSynchronize(ev) != cudaSuccess) { drain_err = 1; return; }
                par_memcpy(dst, src, nb_e);
            });
        }
        if (c < nchunk) {                                   // stage and upload chunk c
            const int b = (int)(c & 1);
            const int64_t s0 = c * per, ns = std::min(per, n_stream - s0);
            const size_t in_b = (size_t)(hi[(size_t)c] - lo[(size_t)c]);
            if (c >= 2) PIPE_CUDA(cudaEventSynchronize(hp.ev_in[b]));
            par_memcpy(hp.pin_in[b], bytes + lo[(size_t)c], in_b);
            rel[b].resize((size_t)ns);
            for (int64_t i = 0; i < ns; ++i) rel[b][(size_t)i] = starts[s0 + i] - lo[(size_t)c];
            if (c >= 2) PIPE_CUDA(cudaStreamWaitEvent(hp.s_in, hp.ev_k[b], 0));  // decode c-2 has read d_b[b] / d_aux[b]
            // the two small pageable copies go first: the runtime waits for the stream before staging them,
            // and behind the large upload that wait would stall this thread for the whole transfer
            PIPE_CUDA(cudaMemcpyAsync(d_aux[b].p, rel[b].data(), (size_t)ns * 8, cudaMemcpyHostToDevice, hp.s_in));
            PIPE_CUDA(cudaMemcpyAsync((int64_t*)d_aux[b].p + per, nbytes + s0, (size_t)ns * 8, cudaMemcpyHostToDevice, hp.s_in));
            PIPE_CUDA(cudaMemcpyAsync(d_b[b].p, hp.pin_in[b], in_b, cudaMemcpyHostToDevice, hp.s_in));
            PIPE_CUDA(cudaEventRecord(hp.ev_in[b], hp.s_in));
        }
        if (c >= 1 && c - 1 < nchunk) {                     // decode chunk c-1, start its download
            const int64_t e = c - 1;
            const int b = (int)(e & 1);
            const int64_t s0 = e * per, ns = std::min(per, n_stream - s0);
            PIPE_CUDA(cudaStreamWaitEvent(hp.s_k, hp.ev_in[b], 0));
            if (e >= 2) PIPE_CUDA(cudaStreamWaitEvent(hp.s_k, hp.ev_out[b], 0));  // download e-2 has read d_o[b]
            rc = fab_decode(ctx, (const unsigned char*)d_b[b].p, (const int64_t*)d_aux[b].p, (const int64_t*)d_aux[b].p + per, ns,
                            stream_size, is_int64, first, last, d_o[b].p, nullptr, nullptr, mx[(size_t)e], bs_hint, hp.s_k);
            if (rc) goto done;
            PIPE_CUDA(cudaEventRecord(hp.ev_k[b], hp.s_k));
            PIPE_CUDA(cudaStreamWaitEvent(hp.s_out, hp.ev_k[b], 0));
            // pinned buffer b was emptied by the helper thread of the previous iteration (joined below)
            PIPE_CUDA(cudaMemcpyAsync(hp.pin_out[b], d_o[b].p, (size_t)ns * row_b, cudaMemcpyDeviceToHost, hp.s_out));
            PIPE_CUDA(cudaEventRecord(hp.ev_out[b], hp.s_out));
        }
        if (drainer.joinable()) drainer.join();
        if (drain_err) { rc = FAB_ERROR_CUDA; goto done; }
    }
    rc = fab_finish(ctx, hp.s_k);
done:
    if (drainer.joinable()) drainer.join();
    if (rc) hp.drain();
    return rc;
}
#undef PIPE_CUDA

int host_encode(const void* data, int dtype, int64_t n_stream, int64_t stream_size, uint32_t level, int64_t* n_bytes,
                int64_t* starts, unsigned char** bytes) {
    if (level > 8) return ERROR_INVALID_LEVEL;
    if (n_stream == 0) return ERROR_ZERO_NSTREAM;
    if (stream_size == 0) return ERROR_ZERO_STREAMSIZE;
    *n_bytes = 0;
    *bytes = nullptr;
    SlotLease lease;
    fab_ctx* ctx = lease.ctx();
    if (!ctx) return FAB_ERROR_CUDA;
    size_t in_b = (size_t)n_stream * stream_size * (dtype == FAB_I64 ? 8 : 4);
    if (in_b >= kPipeMin && n_stream >= 2 && pipe_enabled())
        return host_encode_pipelined(ctx, lease.pipe(), data, dtype, n_stream, stream_size, level, n_bytes, starts, bytes);
    int64_t bound = fab_encode_bound(n_stream, stream_size, dtype, level);
    DevBuf d_in, d_out, d_aux;
    if (!d_in.alloc(in_b) || !d_out.alloc((size_t)bound) || !d_aux.alloc((size_t)n_stream * 16 + 64)) {
        cudaGetLastError();
        return ERROR_ALLOC | FAB_ERROR_CUDA;
    }
    int64_t* d_starts = (int64_t*)d_aux.p;
    int64_t* d_nb = d_starts + n_stream;
    int64_t* d_total = d_nb + n_stream;
    if (cudaMemcpy(d_in.p, data, in_b, cudaMemcpyHostToDevice) != cudaSuccess) return FAB_ERROR_CUDA;
    int rc = fab_encode(ctx, d_in.p, dtype, n_stream, stream_size, level, nullptr, nullptr, nullptr,
                        (unsigned char*)d_out.p, bound, d_starts, d_nb, d_total, nullptr);
    if (rc) return rc;
    rc = fab_finish(ctx, nullptr);
    if (rc) return rc;
    int64_t total = 0;
    if (cudaMemcpy(&total, d_total, 8, cudaMemcpyDeviceToHost) != cudaSuccess) return FAB_ERROR_CUDA;
    if (cudaMemcpy(starts, d_starts, (size_t)n_stream * 8, cudaMemcpyDeviceToHost) != cudaSuccess) return FAB_ERROR_CUDA;
    unsigned char* hb = (unsigned char*)malloc((size_t)total);
    if (!hb) return ERROR_ALLOC;
    if (cudaMemcpy(hb, d_out.p, (size_t)total, cudaMemcpyDeviceToHost) != cudaSuccess) { free(hb); return FAB_ERROR_CUDA; }
    *n_bytes = total;
    *bytes = hb;
    return ERROR_NONE;
}

int host_decode(const unsigned char* bytes, const int64_t* starts, const int64_t* nbytes, int64_t n_stream,
                int64_t stream_size, int is_int64, int64_t first, int64_t last, void* data) {
    if (n_stream <= 0) return ERROR_ZERO_NSTREAM;
    int64_t n_decode = stream_size;
    if (first >= 0 && last >= 0) {
        if (last > stream_size || first > stream_size - 1 || first >= last) return ERROR_DECODE_SAMPLE_RANGE;
        n_decode = last - first;
    }
    SlotLease lease;
    fab_ctx* ctx = lease.ctx();
    if (!ctx) return FAB_ERROR_CUDA;
    // the selected windows may be scattered (keep mask): upload the covering byte range only
    int64_t lo = INT64_MAX, hi = 0, mx = 0;
    for (int64_t i = 0; i < n_stream; ++i) {
        lo = std::min(lo, starts[i]);
        hi = std::max(hi, starts[i] + nbytes[i]);
        mx = std::max(mx, nbytes[i]);
    }
    size_t out_b = (size_t)n_stream * n_decode * (is_int64 ? 8 : 4);
    if (out_b >= kPipeMin && n_stream >= 2 && pipe_enabled()) {
        bool handled = false;
        int prc = host_decode_pipelined(ctx, lease.pipe(), bytes, starts, nbytes, n_stream, stream_size, is_int64, first, last, n_decode,
                                        data, &handled);
        if (handled) return prc;
    }
    std::vector<int64_t> rel((size_t)n_stream);
    for (int64_t i = 0; i < n_stream; ++i) rel[(size_t)i] = starts[i] - lo;
    DevBuf d_b, d_aux, d_o;
    if (!d_b.alloc((size_t)(hi - lo)) || !d_aux.alloc((size_t)n_stream * 16) || !d_o.alloc(out_b)) {
        cudaGetLastError();
        return ERROR_ALLOC | FAB_ERROR_CUDA;
    }
    int64_t* d_starts = (int64_t*)d_aux.p;
    int64_t* d_nb = d_starts + n_stream;
    if (cudaMemcpy(d_b.p, bytes + lo, (size_t)(hi - lo), cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemcpy(d_starts, rel.data(), (size_t)n_stream * 8, cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemcpy(d_nb, nbytes, (size_t)n_stream * 8, cudaMemcpyHostToDevice) != cudaSuccess)
        return FAB_ERROR_CUDA;
    const int bs_hint = stream_blocksize_hint(bytes + starts[0], nbytes[0]);
    int rc = fab_decode(ctx, (const unsigned char*)d_b.p, d_starts, d_nb, n_stream, stream_size, is_int64, first, last,
                        d_o.p, nullptr, nullptr, mx, bs_hint, nullptr);
    if (rc) return rc;
    rc = fab_finish(ctx, nullptr);
    if (rc) return rc;
    if (cudaMemcpy(data, d_o.p, out_b, cudaMemcpyDeviceToHost) != cudaSuccess) return FAB_ERROR_CUDA;
    return ERROR_NONE;
}

template <typename T, typename I>
int host_float_to_int(const T* input, int64_t n_stream, int64_t stream_size, const T* quanta, I* output, T* offsets,
                      T* gains) {
    SlotLease lease;
    fab_ctx* ctx = lease.ctx();
    if (!ctx) return FAB_ERROR_CUDA;
    size_t n = (size_t)n_stream * stream_size;
    DevBuf d_in, d_out, d_aux;
    if (!d_in.alloc(n * sizeof(T)) || !d_out.alloc(n * sizeof(I)) || !d_aux.alloc((size_t)n_stream * 3 * sizeof(T))) {
        cudaGetLastError();
        return ERROR_ALLOC | FAB_ERROR_CUDA;
    }
    T* d_off = (T*)d_aux.p;
    T* d_gain = d_off + n_stream;
    T* d_q = d_gain + n_stream;
    if (cudaMemcpy(d_in.p, input, n * sizeof(T), cudaMemcpyHostToDevice) != cudaSuccess) return FAB_ERROR_CUDA;
    if (quanta && cudaMemcpy(d_q, quanta, (size_t)n_stream * sizeof(T), cudaMemcpyHostToDevice) != cudaSuccess) return FAB_ERROR_CUDA;
    int rc = fab_float_to_int(ctx, d_in.p, sizeof(T) == 4 ? FAB_F32 : FAB_F64, n_stream, stream_size, quanta ? d_q : nullptr,
                              d_out.p, d_off, d_gain, nullptr);
    if (rc) return rc;
    rc = fab_finish(ctx, nullptr);
    rc &= ~FAB_ERROR_NAN;  // the reference's C function does not look for NaNs (utils.py:268 does, before calling)
    if (rc) return rc;
    if (cudaMemcpy(output, d_out.p, n * sizeof(I), cudaMemcpyDeviceToHost) != cudaSuccess ||
        cudaMemcpy(offsets, d_off, (size_t)n_stream * sizeof(T), cudaMemcpyDeviceToHost) != cudaSuccess ||
        cudaMemcpy(gains, d_gain, (size_t)n_stream * sizeof(T), cudaMemcpyDeviceToHost) != cudaSuccess)
        return FAB_ERROR_CUDA;
    return ERROR_NONE;
}

template <typename I, typename T>
void host_int_to_float(const I* input, int64_t n_stream, int64_t stream_size, const T* offsets, const T* gains, T* output) {
    SlotLease lease;
    fab_ctx* ctx = lease.ctx();
    size_t n = (size_t)n_stream * stream_size;
    DevBuf d_in, d_out, d_aux;
    if (!ctx || !d_in.alloc(n * sizeof(I)) || !d_out.alloc(n * sizeof(T)) || !d_aux.alloc((size_t)n_stream * 2 * sizeof(T))) {
        fprintf(stderr, "flacarray_b200: int_to_float failed: no CUDA device or out of memory\n");
        abort();  // the reference signature returns void: fail loudly rather than return garbage
    }
    T* d_off = (T*)d_aux.p;
    T* d_gain = d_off + n_stream;
    cudaMemcpy(d_in.p, input, n * sizeof(I), cudaMemcpyHostToDevice);
    cudaMemcpy(d_off, offsets, (size_t)n_stream * sizeof(T), cudaMemcpyHostToDevice);
    cudaMemcpy(d_gain, gains, (size_t)n_stream * sizeof(T), cudaMemcpyHostToDevice);
    int rc = fab_int_to_float(ctx, d_in.p, sizeof(I) == 4 ? FAB_I32 : FAB_I64, n_stream, stream_size, d_off, d_gain, d_out.p, nullptr);
    if (!rc) rc = fab_finish(ctx, nullptr);
    if (rc || cudaMemcpy(output, d_out.p, n * sizeof(T), cudaMemcpyDeviceToHost) != cudaSuccess) {
        fprintf(stderr, "flacarray_b200: int_to_float failed (code %d): %s\n", rc, fab_last_error(ctx));
        abort();
    }
}
}  // namespace

extern "C" {
int encode_i32(int32_t* const data, int64_t n_stream, int64_t stream_size, uint32_t level, int64_t* n_bytes,
               int64_t* starts, unsigned char** bytes) {
    return host_encode(data, FAB_I32, n_stream, stream_size, level, n_bytes, starts, bytes);
}
int encode_i32_threaded(int32_t* const data, int64_t n_stream, int64_t stream_size, uint32_t level, int64_t* n_bytes,
                        int64_t* starts, unsigned char** bytes) {
    return host_encode(data, FAB_I32, n_stream, stream_size, level, n_bytes, starts, bytes);
}
int encode_i64(int64_t* const data, int64_t n_stream, int64_t stream_size, uint32_t level, int64_t* n_bytes,
               int64_t* starts, unsigned char** bytes) {
    return host_encode(data, FAB_I64, n_stream, stream_size, level, n_bytes, starts, bytes);
}
int encode_i64_threaded(int64_t* const data, int64_t n_stream, int64_t stream_size, uint32_t level, int64_t* n_bytes,
                        int64_t* starts, unsigned char** bytes) {
    return host_encode(data, FAB_I64, n_stream, stream_size, level, n_bytes, starts, bytes);
}
int decode_i32(unsigned char* const bytes, int64_t* const starts, int64_t* const nbytes, int64_t n_stream,
               int64_t stream_size, int64_t first_sample, int64_t last_sample, int32_t* data, bool) {
    return host_decode(bytes, starts, nbytes, n_stream, stream_size, 0, first_sample, last_sample, data);
}
int decode_i64(unsigned char* const bytes, int64_t* const starts, int64_t* const nbytes, int64_t n_stream,
               int64_t stream_size, int64_t first_sample, int64_t last_sample, int64_t* data, bool) {
    return host_decode(bytes, starts, nbytes, n_stream, stream_size, 1, first_sample, last_sample, data);
}
int float32_to_int32(float const* input, int64_t n_stream, int64_t stream_size, float const* quanta, int32_t* output,
                     float* offsets, float* gains) {
    return host_float_to_int<float, int32_t>(input, n_stream, stream_size, quanta, output, offsets, gains);
}
int float64_to_int64(double const* input, int64_t n_stream, int64_t stream_size, double const* quanta, int64_t* output,
                     double* offsets, double* gains) {
    return host_float_to_int<double, long long>(input, n_stream, stream_size, quanta, (long long*)output, offsets, gains);
}
void int64_to_float64(int64_t const* input, int64_t n_stream, int64_t stream_size, double const* offsets,
                      double const* gains, double* output) {
    host_int_to_float<long long, double>((const long long*)input, n_stream, stream_size, offsets, gains, output);
}
void int32_to_float32(int32_t const* input, int64_t n_stream, int64_t stream_size, float const* offsets,
                      float const* gains, float* output) {
    host_int_to_float<int32_t, float>(input, n_stream, stream_size, offsets, gains, output);
}
}
