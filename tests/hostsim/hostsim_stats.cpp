// hostsim_stats.cpp -- TEST HARNESS ONLY.  Host build of fab_row_stats with the OS-thread SIMT emulator of fa_simt.h:
// the kernel bodies of flacarray_b200/csrc/fa_stats.h (chunk reducer, per-bin merge, finisher) driven the way
// fab_row_stats drives them, so that their results can be compared bit for bit with a Python-integer reference without a
// GPU.  Never linked into libflacarray_b200.so and never loaded by the Python package.
#include <cstdint>

#include "../../flacarray_b200/csrc/fa_stats.h"

namespace fasim {
thread_local ThreadCtx tls;
}

using namespace fa;

extern "C" {

// fab_row_stats with the piece length as a parameter (piece <= 0: the library's kStatsPieceBytes), so that small rows
// exercise bins spanning many pieces.  bin == 0: one bin per row.  Returns 0 or -1 for arguments fab_row_stats rejects.
// *n_pieces receives nbins * ppb (the reducer's warps per row), *ppb_out the pieces per bin.
int hs_row_stats(const void* rows, int is_int64, int64_t n_rows, int64_t n, int64_t bin, int64_t piece, const void* offsets,
                 const void* gains, const int* status, long long* count, void* mn, void* mx, double* mean, double* std,
                 int64_t* n_pieces, int64_t* ppb_out) {
    if (n_rows <= 0 || n <= 0 || bin < 0) return -1;
    const int64_t len = bin == 0 ? n : (bin < n ? bin : n);
    if (len > kStatsMaxBin) return -1;
    StatsParams P{};
    P.rows = rows; P.is_int64 = is_int64; P.n_rows = n_rows; P.n = n; P.bin = len;
    P.nbins = (n + len - 1) / len;
    P.piece = piece > 0 ? piece : kStatsPieceBytes / (is_int64 ? 8 : 4);
    P.ppb = (len + P.piece - 1) / P.piece;
    std::vector<StatPart> part(P.ppb > 1 ? (size_t)(n_rows * P.nbins * P.ppb) : 0);
    P.part = part.data();
    P.offsets = offsets; P.gains = gains; P.status = status;
    P.count = count; P.mn = mn; P.mx = mx; P.mean = mean; P.std = std;
    const int64_t per_row = P.nbins * P.ppb;
    fasim::launch((int)(n_rows * per_row), 32, 0, [&](int b) {
        if (is_int64) stats_piece_warp<true>(P, b / per_row, b % per_row);
        else stats_piece_warp<false>(P, b / per_row, b % per_row);
    });
    if (P.ppb > 1)
        fasim::launch((int)(n_rows * P.nbins), 32, 0, [&](int b) { stats_merge_warp(P, b / P.nbins, b % P.nbins); });
    if (n_pieces) *n_pieces = per_row;
    if (ppb_out) *ppb_out = P.ppb;
    return 0;
}

// the finisher's correctly rounded conversion alone: v = w[0] + w[1] 2^64 + w[2] 2^128 + w[3] 2^192
double hs_dbl_u256(const unsigned long long* w) {
    U256 v;
    for (int i = 0; i < 4; ++i) v.w[i] = w[i];
    return dbl_u256(v);
}
}
