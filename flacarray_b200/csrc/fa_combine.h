// fa_combine.h -- per-sample weighted sums across decoded integer rows: out[g][i] += sum over the rows k of group g of
// w_k * x_k[i], folded in row order in plain IEEE double.
//
// Input: rows [n_rows][n] of int32 (1-channel streams) or int64 (2-channel streams), the decoder's output layout, with
// per-row weight, optional offset / gain (the float restore) and optional status.  Rows come as segments: segment s is
// the contiguous rows [seg[s], seg[s + 1]) and adds into output row seg_out[s] of out[n_out][n] (double).  For each
// sample i of a segment the fold is
//     acc = out[seg_out[s]][i]
//     for k in [seg[s], seg[s + 1]) with status[k] == 0:   acc = acc + w_k * double(x_k[i])
//     out[seg_out[s]][i] = acc
// with separately rounded multiply and add (explicit _rn intrinsics: never contracted into an FMA).  x_k is the integer
// (int64 -> double rounds to nearest even), or the float the decode's restore returns (restore_f32 / restore_f64 of
// fa_quant.h, in the array's type; float32 then widens exactly).  A zero-filled out makes the first term +0.0 + w x,
// and a group split over several calls continues from the value the previous call stored, so the result is the fold
// over the whole group whatever the grouping into calls.
//
// One CTA of NT threads takes one segment and NT * kCombineCols consecutive columns; a thread keeps the running sums of
// its kCombineCols columns (stride NT, so every row load of a warp is one coalesced 128- or 256-byte piece of the row) in
// registers, with the loads of kCombineUnroll rows issued ahead of the dependent add chain.  Only elements inside the
// rows are read, so rows need no alignment beyond their element size.  The per-row weight, restore coefficient and
// status go through shared memory, one tile of NT rows at a time, so each row's coefficient (a division) is
// computed once per CTA.
//
// Segment records live in device memory and are checked here: 0 <= seg[s] <= seg[s + 1] <= n_rows, 0 <= seg_out[s] <
// n_out and seg_out[s - 1] < seg_out[s].  A record that breaks a rule sets ERROR_DECODE_SAMPLE_RANGE in *err and its
// segment writes nothing.  The same bodies are compiled by nvcc (fab_combine_rows) and by the host emulator of fa_simt.h
// (tests/hostsim/hostsim_combine.cpp).
#pragma once
#include <type_traits>

#include "fa_quant.h"
#include "fa_simt.h"

namespace fa {

constexpr int kCombineThreads = 256;        // threads per CTA of k_combine_rows
constexpr int kCombineCols = 2;             // columns per thread
constexpr int kCombineUnroll = 8;           // rows whose loads are in flight ahead of the adds
constexpr int kCombineBadSegment = 1 << 17; // ERROR_DECODE_SAMPLE_RANGE

struct CombineParams {
    const void* rows;        // [n_rows][n] int32 or int64
    int64_t n_rows, n;
    const void* offsets;     // [n_rows] float32 / float64, or null (integer rows); gains likewise
    const void* gains;
    const int* status;       // [n_rows] or null: rows with a non-zero status are skipped
    const double* weights;   // [n_rows]
    const int64_t* seg;      // [n_seg + 1] row bounds of the segments
    const int64_t* seg_out;  // [n_seg] output row of each segment
    int64_t n_seg;
    double* out;             // [n_out][n]
    int64_t n_out;
    int* err;
};

// per-row values of one tile: the weight, the restore's offset and coefficient (widened for float32 rows) and whether
// the row takes part
struct CombineRow {
    double w, off, coeff;
    int ok;
};

// w * x_k[i] with x_k[i] as to_array returns it, widened to double
template <bool I64, bool FLT>
FA_D double combine_term(typename std::conditional<I64, long long, int32_t>::type x, const CombineRow& r) {
    double v;
    if constexpr (!FLT) v = (double)x;
    else if constexpr (I64) v = restore_f64(x, r.off, r.coeff);
    else v = (double)restore_f32(x, (float)r.off, (float)r.coeff);
    return dmul(r.w, v);
}

// One CTA of NT threads: segment s, columns [c0, c0 + NT * kCombineCols).  `sh` holds NT CombineRow.
template <bool I64, bool FLT, int NT>
FA_D void combine_segment_cta(const CombineParams& P, int64_t s, int64_t c0, CombineRow* sh) {
    typedef typename std::conditional<I64, long long, int32_t>::type T;
    constexpr int C = kCombineCols, U = kCombineUnroll;
    static_assert(NT % U == 0, "a tile is a whole number of unrolled steps");
    const int64_t lo = P.seg[s], hi = P.seg[s + 1], o = P.seg_out[s];
    if (lo < 0 || hi < lo || hi > P.n_rows || o < 0 || o >= P.n_out || (s > 0 && P.seg_out[s - 1] >= o)) {
        if (tid() == 0 && c0 == 0) atom_or_global(P.err, kCombineBadSegment);
        return;                                    // the same decision in every thread of the CTA
    }
    const int64_t n = P.n, c = c0 + tid();
    const T* rows = (const T*)P.rows + c;
    double* orow = P.out + o * n + c;
    bool in[C];
    double acc[C];
#pragma unroll
    for (int j = 0; j < C; ++j) {
        in[j] = c + j * NT < n;
        acc[j] = in[j] ? orow[j * NT] : 0.0;
    }
    for (int64_t t0 = lo; t0 < hi; t0 += NT) {
        const int m = (int)(hi - t0 < NT ? hi - t0 : NT);
        sync();                                    // every thread has finished with the previous tile
        if (tid() < m) {
            const int64_t k = t0 + tid();
            CombineRow r;
            r.w = P.weights[k];
            r.ok = P.status == nullptr || P.status[k] == 0;
            r.off = 0.0;
            r.coeff = 0.0;
            if constexpr (FLT) {
                if constexpr (I64) {
                    r.off = ((const double*)P.offsets)[k];
                    r.coeff = restore_coeff_f64(((const double*)P.gains)[k]);
                } else {
                    r.off = (double)((const float*)P.offsets)[k];
                    r.coeff = (double)restore_coeff_f32(((const float*)P.gains)[k]);
                }
            }
            sh[tid()] = r;
        }
        sync();
        // U rows at a time: all U * C loads are issued before the first add that needs one
        for (int i = 0; i < m; i += U) {
            const T* rp = rows + (t0 + i) * n;
            T v[U][C];
#pragma unroll
            for (int u = 0; u < U; ++u)
#pragma unroll
                for (int j = 0; j < C; ++j) v[u][j] = (i + u < m && in[j]) ? rp[u * n + j * NT] : (T)0;
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (i + u >= m) break;
                const CombineRow r = sh[i + u];
                if (!r.ok) continue;
#pragma unroll
                for (int j = 0; j < C; ++j) acc[j] = dadd(acc[j], combine_term<I64, FLT>(v[u][j], r));
            }
        }
    }
#pragma unroll
    for (int j = 0; j < C; ++j)
        if (in[j]) orow[j * NT] = acc[j];
}

}  // namespace fa
