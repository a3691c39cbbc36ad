// hostsim_combine.cpp -- TEST HARNESS ONLY.  Host build of fab_combine_rows with the OS-thread SIMT emulator of fa_simt.h:
// the kernel body of flacarray_b200/csrc/fa_combine.h driven the way fab_combine_rows drives it (one block per (segment,
// column chunk)), with 32-thread blocks so that small arrays span several column chunks and long segments several row
// tiles.  Never linked into libflacarray_b200.so and never loaded by the Python package.
#include <cstdint>

#include "../../flacarray_b200/csrc/fa_combine.h"

namespace fasim {
thread_local ThreadCtx tls;
}

using namespace fa;

namespace {
constexpr int kThreads = 32;

template <bool I64, bool FLT>
void run(const CombineParams& P, int64_t gx) {
    fasim::launch((int)(gx * P.n_seg), kThreads, kThreads * sizeof(CombineRow), [&](int b) {
        combine_segment_cta<I64, FLT, kThreads>(P, b / gx, (int64_t)(b % gx) * (kThreads * kCombineCols),
                                                (CombineRow*)fasim::smem());
    });
}
}  // namespace

extern "C" {

// fab_combine_rows on host memory.  Returns 0, or -1 for arguments fab_combine_rows rejects before launching; *err
// receives the error bits the segment checks set.
int hs_combine_rows(const void* rows, int is_int64, int64_t n_rows, int64_t n, const void* offsets, const void* gains,
                    const int* status, const double* weights, const int64_t* seg, const int64_t* seg_out, int64_t n_seg,
                    double* out, int64_t n_out, int* err) {
    if (n_rows <= 0 || n <= 0 || n_seg <= 0 || n_out <= 0 || (offsets == nullptr) != (gains == nullptr)) return -1;
    *err = 0;
    CombineParams P{};
    P.rows = rows; P.n_rows = n_rows; P.n = n;
    P.offsets = offsets; P.gains = gains; P.status = status; P.weights = weights;
    P.seg = seg; P.seg_out = seg_out; P.n_seg = n_seg;
    P.out = out; P.n_out = n_out; P.err = err;
    const int64_t gx = (n + kThreads * kCombineCols - 1) / (kThreads * kCombineCols);
    if (is_int64) {
        if (offsets) run<true, true>(P, gx);
        else run<true, false>(P, gx);
    } else {
        if (offsets) run<false, true>(P, gx);
        else run<false, false>(P, gx);
    }
    return 0;
}
}
