// hostsim_flags.cpp -- TEST HARNESS ONLY.  Compiles the kernel bodies of flacarray_b200/csrc/fa_flags.h for the host with
// the OS-thread SIMT emulator of fa_simt.h, driven as fab_flag_count and fab_flag_write drive them, so that the range
// search can be unit-tested without a GPU.  Built into its own library by hostsim_flags.py (the emulator of the other
// kernel bodies is hostsim.cpp); never linked into libflacarray_b200.so and never loaded by the Python package.
#include <vector>

#include "../../flacarray_b200/csrc/fa_flags.h"

namespace fasim {
thread_local ThreadCtx tls;
}

using namespace fa;

extern "C" {
// fab_flag_count followed by fab_flag_write, with the piece length as a parameter (piece <= 0: the library's
// kFlagPieceBytes; else a multiple of 32) so that small rows span many pieces.  The rows' output slots are the exclusive
// prefix of the counts, as the library's caller lays them out; *total receives their sum, and nothing is written when it
// exceeds cap.  Returns 0, the error bits fab_flag_count returns for its arguments, or -1 when cap is too small.
int hs_flag_ranges(const void* rows, int is_int64, int64_t n_rows, int64_t n, const void* lo, const void* hi,
                   const void* offsets, const void* gains, const int* status, int64_t pad, int64_t piece, int64_t sample0,
                   long long* nflag, long long* nrange, long long* first_out, long long* last_out, int64_t cap,
                   int64_t* total) {
    FlagParams P{};
    const int rc = flag_geometry(n_rows, n, is_int64, pad, &P, piece > 0 ? piece : 0);
    if (rc) return rc;
    if ((offsets == nullptr) != (gains == nullptr)) return kErrConvertType;
    std::vector<uint32_t> mask((size_t)(n_rows * P.wpr), 0xA5A5A5A5u);      // garbage: pass 1 writes every word it reads
    std::vector<FlagPiece> sum((size_t)(n_rows * P.ppr));
    std::vector<long long> base((size_t)n_rows, 0);
    P.rows = rows; P.lo = lo; P.hi = hi; P.offsets = offsets; P.gains = gains; P.status = status;
    P.mask = mask.data(); P.sum = sum.data(); P.nflag = nflag; P.nrange = nrange;
    const int64_t ppr = P.ppr;
    fasim::launch((int)(n_rows * ppr), 32, 0, [&](int b) {                 // k_flag_scan
        if (is_int64) flag_scan_warp<true>(P, b / ppr, b % ppr);
        else flag_scan_warp<false>(P, b / ppr, b % ppr);
    });
    fasim::launch((int)n_rows, 32, 0, [&](int b) { flag_offsets_warp(P, b); });    // k_flag_offsets
    int64_t t = 0;
    for (int64_t r = 0; r < n_rows; ++r) { base[(size_t)r] = t; t += nrange[r]; }
    *total = t;
    if (t > cap) return -1;
    P.base = base.data(); P.sample0 = sample0; P.first_out = first_out; P.last_out = last_out;
    fasim::launch((int)(n_rows * ppr), 32, 0, [&](int b) { flag_write_warp(P, b / ppr, b % ppr); });   // k_flag_write
    return 0;
}

// flag_bounds alone: the keep range [*L, *H] of a float row (is_int64: float64 restore, else float32 with off and coeff
// rounded to float)
void hs_flag_bounds(int is_int64, double off, double coeff, double lo, double hi, long long* L, long long* H) {
    if (is_int64) flag_bounds<true>(off, coeff, lo, hi, L, H);
    else flag_bounds<false>((double)(float)off, (double)(float)coeff, lo, hi, L, H);
}
}
