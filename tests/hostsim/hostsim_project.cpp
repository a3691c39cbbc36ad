// hostsim_project.cpp -- TEST HARNESS ONLY.  Compiles the kernel bodies of flacarray_b200/csrc/fa_project.h for the host
// with the OS-thread SIMT emulator of fa_simt.h, driven as fab_project_rows drives them, so that the projections can be
// unit-tested without a GPU.  Built into its own library by hostsim_project.py (the emulator of the other kernel bodies
// is hostsim.cpp); never linked into libflacarray_b200.so and never loaded by the Python package.
#include <vector>

#include "../../flacarray_b200/csrc/fa_project.h"

namespace fasim {
thread_local ThreadCtx tls;
}

using namespace fa;

// 32-thread blocks (32 rows per block), so that small arrays span several row tiles; the pieces, chunks and passes are
// the library's.
namespace {
constexpr int kProjectSimThreads = 32;

template <bool I64, bool FLT, int CH>
void project_pieces(const ProjectParams& P) {
    typedef typename std::conditional<I64, long long, int32_t>::type T;
    const int64_t gx = (P.n_rows + kProjectSimThreads - 1) / kProjectSimThreads;
    const size_t rs_bytes = (size_t)kProjectSimThreads * (kProjectSub + 1) * sizeof(T);
    fasim::launch((int)(gx * P.npieces), kProjectSimThreads, rs_bytes + kProjectSub * CH * sizeof(double), [&](int b) {
        unsigned char* sm = fasim::smem();
        project_piece_cta<I64, FLT, kProjectSimThreads, CH>(P, (b % gx) * kProjectSimThreads, b / gx, (T*)sm,
                                                             (double*)(sm + ((rs_bytes + 15) & ~(size_t)15)));
    });
}

template <bool I64, bool FLT>
void project_rows(const ProjectParams& P, int ch) {
    switch (ch) {
        case 1: project_pieces<I64, FLT, 1>(P); break;
        case 2: project_pieces<I64, FLT, 2>(P); break;
        case 4: project_pieces<I64, FLT, 4>(P); break;
        case 8: project_pieces<I64, FLT, 8>(P); break;
        default: project_pieces<I64, FLT, kProjectMaxChunk>(P); break;
    }
}
}  // namespace

extern "C" {
// Returns 0 or the error bits fab_project_rows returns for its arguments (-1 for offsets without gains).
int hs_project_rows(const void* rows, int is_int64, int64_t n_rows, int64_t n, const void* offsets, const void* gains,
                    const int* status, const double* templates, int64_t n_tmpl, double* out) {
    ProjectParams P{};
    const int rc = project_geometry(n_rows, n, n_tmpl, &P);
    if (rc) return rc;
    if ((offsets == nullptr) != (gains == nullptr)) return -1;
    std::vector<double> part((size_t)project_partials(P));
    P.rows = rows; P.offsets = offsets; P.gains = gains; P.status = status;
    P.tmpl = templates; P.part = part.data(); P.out = out;
    const int ch = project_chunk(n_tmpl);
    if (is_int64) {
        if (offsets) project_rows<true, true>(P, ch);
        else project_rows<true, false>(P, ch);
    } else {
        if (offsets) project_rows<false, true>(P, ch);
        else project_rows<false, false>(P, ch);
    }
    fasim::launch((int)((n_rows * n_tmpl + kProjectSimThreads - 1) / kProjectSimThreads), kProjectSimThreads, 0, [&](int b) {
        const int64_t idx = (int64_t)b * kProjectSimThreads + tid();
        if (idx < n_rows * n_tmpl) project_fold(P, idx);
    });
    return 0;
}
}
