// fa_project.h -- per-row projections onto templates: out[k][t] = sum_i T[t][i] * v_k[i] of decoded integer rows,
// folded in a fixed order in plain IEEE double.
//
// Input: rows [n_rows][n] of int32 (1-channel streams) or int64 (2-channel streams), the decoder's output layout, with
// optional per-row offset / gain (the float restore) and status, and templates [n_tmpl][n] of double.  v_k[i] is the
// integer (int64 -> double rounds to nearest even), or the float the decode's restore returns (restore_f32 /
// restore_f64 of fa_quant.h, in the array's type; float32 then widens exactly).  The samples are cut into pieces of
// kProjectPiece counted from sample 0 (the last one may be shorter), and with separately rounded multiply and add
// (explicit _rn intrinsics: never contracted into an FMA)
//     for each piece j:  p_j = +0.0;  for i in piece j ascending:  p_j = p_j + T[t][i] * v_k[i]
//     out[k][t] = +0.0;  for j ascending:  out[k][t] = out[k][t] + p_j
// so the result is defined by the piece length alone, whatever the grid, the grouping of rows into calls or the
// residency of the bytes.
//
// Pass 1 (project_piece_cta): one CTA of NT threads takes one piece and NT consecutive rows; thread t owns row r0 + t.
// The piece goes through shared memory in sub-tiles of kProjectSub samples: the rows with coalesced loads (a warp reads
// 32 consecutive samples of one row) into a pitch of kProjectSub + 1 elements, so that the 32 threads of a warp reading
// sample i of their own rows hit 32 different banks, and CH templates in [sample][template] order, which every thread
// reads at the same address (a broadcast).  Each thread keeps the CH partials of its row in registers, so each sample
// is converted and restored once per chunk of CH templates; more than CH templates take several chunks, each a pass over
// the piece.  Only elements inside the rows are read, so rows need no alignment beyond their element size.  The partial
// of (row, template, piece) goes to part[n_rows][n_tmpl][npieces].
// Pass 2 (project_fold): one thread per (row, template) folds the partials in piece order and writes out[n_rows][n_tmpl];
// a row with a non-zero status gets NaN.
//
// The same bodies are compiled by nvcc (fab_project_rows) and by the host emulator of fa_simt.h
// (tests/hostsim/hostsim_project.cpp).
#pragma once
#include <type_traits>

#include "fa_bits.h"
#include "fa_quant.h"
#include "fa_simt.h"
#include "fa_stats.h"

namespace fa {

constexpr int kProjectPiece = 4096;         // samples per partial (FAB_PROJECT_PIECE): part of the result's definition
constexpr int kProjectThreads = 128;        // threads (rows) per CTA of k_project_piece
constexpr int kProjectSub = 32;             // samples per staged sub-tile
constexpr int kProjectMaxChunk = 16;        // templates whose partials one thread keeps in registers
constexpr int kProjectLoads = 16;           // row loads a thread has in flight while staging a sub-tile
constexpr int kProjectFoldThreads = 256;    // threads per CTA of k_project_fold

struct ProjectParams {
    const void* rows;        // [n_rows][n] int32 or int64
    int64_t n_rows, n;
    const void* offsets;     // [n_rows] float32 / float64, or null (integer rows); gains likewise
    const void* gains;
    const int* status;       // [n_rows] or null: rows with a non-zero status get NaN
    const double* tmpl;      // [n_tmpl][n]
    int64_t n_tmpl;
    int64_t npieces;         // ceil(n / kProjectPiece)
    double* part;            // [n_rows][n_tmpl][npieces] partials of pass 1
    double* out;             // [n_rows][n_tmpl]
};

// Geometry of a call: returns 0 and fills *P's sizes, or the error bits of bad arguments (kErrAlloc when the partials
// would not be addressable).
inline int project_geometry(int64_t n_rows, int64_t n, int64_t n_tmpl, ProjectParams* P) {
    if (n_rows <= 0 || n_tmpl <= 0) return kErrZeroNstream;
    if (n <= 0) return kErrZeroStreamsize;
    P->n_rows = n_rows; P->n = n; P->n_tmpl = n_tmpl;
    P->npieces = (n + kProjectPiece - 1) / kProjectPiece;
    if (n_tmpl > (int64_t)0x7FFFFFFFFFFFFFFFll / 8 / n_rows / P->npieces) return kErrAlloc;
    return 0;
}

// number of partials of pass 1
inline int64_t project_partials(const ProjectParams& P) { return P.n_rows * P.n_tmpl * P.npieces; }

// templates per chunk of pass 1: the smallest power of two >= n_tmpl, at most kProjectMaxChunk
inline int project_chunk(int64_t n_tmpl) {
    int c = 1;
    while (c < n_tmpl && c < kProjectMaxChunk) c *= 2;
    return c;
}

// v_k[i] as to_array returns it, widened to double
template <bool I64, bool FLT>
FA_D double project_value(typename std::conditional<I64, long long, int32_t>::type x, double off, double coeff) {
    if constexpr (!FLT) return (double)x;
    else if constexpr (I64) return restore_f64(x, off, coeff);
    else return (double)restore_f32(x, (float)off, (float)coeff);
}

// Pass 1, one CTA of NT threads: piece j of rows [r0, r0 + NT).  rs: NT * (kProjectSub + 1) elements of the row type,
// ts: kProjectSub * CH doubles, both in shared memory.
template <bool I64, bool FLT, int NT, int CH>
FA_D void project_piece_cta(const ProjectParams& P, int64_t r0, int64_t j,
                            typename std::conditional<I64, long long, int32_t>::type* rs, double* ts) {
    typedef typename std::conditional<I64, long long, int32_t>::type T;
    constexpr int S = kProjectSub, W = kProjectSub + 1;
    static_assert(S % kProjectLoads == 0, "whole load batches per sub-tile");
    const int64_t n = P.n, e0 = j * kProjectPiece, e1 = e0 + kProjectPiece < n ? e0 + kProjectPiece : n;
    const int64_t row = r0 + tid();
    const bool live = row < P.n_rows;
    const int nrows = (int)(P.n_rows - r0 < NT ? P.n_rows - r0 : NT);
    double off = 0.0, coeff = 0.0;
    if constexpr (FLT) {
        if (live) {
            if constexpr (I64) {
                off = ((const double*)P.offsets)[row];
                coeff = restore_coeff_f64(((const double*)P.gains)[row]);
            } else {
                off = (double)((const float*)P.offsets)[row];
                coeff = (double)restore_coeff_f32(((const float*)P.gains)[row]);
            }
        }
    }
    const T* rows = (const T*)P.rows + r0 * n;
    const T* mine = rs + tid() * W;
    for (int64_t c0 = 0; c0 < P.n_tmpl; c0 += CH) {
        const int nc = (int)(P.n_tmpl - c0 < CH ? P.n_tmpl - c0 : CH);
        double acc[CH];
#pragma unroll
        for (int c = 0; c < CH; ++c) acc[c] = 0.0;
        for (int64_t s0 = e0; s0 < e1; s0 += S) {
            const int m = (int)(e1 - s0 < S ? e1 - s0 : S);
            sync();                                // every thread has finished with the previous sub-tile
            // a thread issues kProjectLoads row loads into registers before it stores them to shared memory, so that
            // they are in flight together rather than one load / store pair at a time
#pragma unroll
            for (int k0 = 0; k0 < NT * S; k0 += NT * kProjectLoads) {
                T v[kProjectLoads];
#pragma unroll
                for (int u = 0; u < kProjectLoads; ++u) {
                    const int e = k0 + u * NT + tid(), r = e / S, i = e % S;
                    v[u] = (r < nrows && i < m) ? rows[r * n + s0 + i] : (T)0;
                }
#pragma unroll
                for (int u = 0; u < kProjectLoads; ++u) {
                    const int e = k0 + u * NT + tid();
                    rs[(e / S) * W + e % S] = v[u];
                }
            }
#pragma unroll
            for (int k = 0; k < CH * S; k += NT) {
                const int e = k + tid(), c = e / S, i = e % S;
                if (e < CH * S) ts[i * CH + c] = (c < nc && i < m) ? P.tmpl[(c0 + c) * n + s0 + i] : 0.0;
            }
            sync();
            if (live) {
                if (m == S) {
#pragma unroll 8
                    for (int i = 0; i < S; ++i) {
                        const double v = project_value<I64, FLT>(mine[i], off, coeff);
#pragma unroll
                        for (int c = 0; c < CH; ++c) acc[c] = dadd(acc[c], dmul(ts[i * CH + c], v));
                    }
                } else {
                    for (int i = 0; i < m; ++i) {
                        const double v = project_value<I64, FLT>(mine[i], off, coeff);
#pragma unroll
                        for (int c = 0; c < CH; ++c) acc[c] = dadd(acc[c], dmul(ts[i * CH + c], v));
                    }
                }
            }
        }
        if (live) {
            double* dst = P.part + (row * P.n_tmpl + c0) * P.npieces + j;
#pragma unroll
            for (int c = 0; c < CH; ++c)
                if (c < nc) dst[c * P.npieces] = acc[c];
        }
    }
}

// Pass 2: (row, template) idx = row * n_tmpl + t folds its partials in piece order.
FA_D void project_fold(const ProjectParams& P, int64_t idx) {
    const int64_t row = idx / P.n_tmpl;
    if (P.status && P.status[row] != 0) {
        P.out[idx] = bits_to_double(0x7FF8000000000000ull);
        return;
    }
    const double* src = P.part + idx * P.npieces;
    double acc = 0.0;
    for (int64_t j = 0; j < P.npieces; ++j) acc = dadd(acc, src[j]);
    P.out[idx] = acc;
}

}  // namespace fa
