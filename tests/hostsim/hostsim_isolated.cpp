// hostsim_isolated.cpp -- TEST HARNESS ONLY.  Host build of the per-stream fault isolation (fab_decode_isolated) and
// of fab_verify with the OS-thread SIMT emulator of fa_simt.h, next to hostsim.cpp: the same kernel bodies of
// flacarray_b200/csrc driven the way the product drives them, so that per-stream status, the fill of failed rows and
// the no-store decoder can be unit-tested without a GPU.  Never linked into libflacarray_b200.so and never loaded by
// the Python package.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../flacarray_b200/csrc/fa_decode.h"
#include "../../flacarray_b200/csrc/fa_decode_tile.h"

namespace fasim {
thread_local ThreadCtx tls;
}

using namespace fa;

static CrcTables g_crc;
static bool g_crc_ready = false;
static const CrcTables* crc() {
    if (!g_crc_ready) { crc_tables_init(&g_crc); g_crc_ready = true; }
    return &g_crc;
}

extern "C" {

// fab_decode_isolated (data != NULL, store = 1) / fab_verify (data == NULL, store = 0, first = last = -1), driven like
// hs_decode mode 2: meta -> sync scan -> warp-tile kernel (storing / not storing) -> CRC pass -> general decoder on the
// flagged frames -> walker on the flagged streams -> fill of the rows of failed streams with 0.  status[n_sel] receives
// every stream's bits; the return value is the call-level error mask.  *info = streams walked + 1000 * frames left to
// the general decoder.
int hs_decode_isolated(const uint8_t* bytes, const long long* starts, const long long* nbytes, int64_t n_sel,
                       int64_t stream_size, int nch, int64_t first, int64_t last, int32_t* data, int store, int* status,
                       int* info) {
    int64_t n_decode = stream_size, first_decode = 0;
    if (first >= 0 && last >= 0) {
        if (last > stream_size || first > stream_size - 1 || first >= last) return kErrDecodeSampleRange;
        first_decode = first;
        n_decode = last - first;
    }
    // the blocksize hint of the library: the first stream's STREAMINFO min blocksize (4096 without one), >= 16
    int bsh = 4096;
    const uint8_t* s0 = n_sel > 0 ? bytes + starts[0] : nullptr;
    if (s0 && nbytes[0] >= 12 && memcmp(s0, "fLaC", 4) == 0 && ((s0[8] << 8) | s0[9]) > 0) bsh = (s0[8] << 8) | s0[9];
    if (bsh < 16) bsh = 16;
    const int nframes_cap = (int)((stream_size + bsh - 1) / bsh);
    std::vector<StreamMeta> meta((size_t)n_sel);
    std::vector<long long> fo((size_t)n_sel * (size_t)(nframes_cap + 1), -1);
    std::vector<int> flag((size_t)n_sel, 0);
    std::vector<unsigned char> fflag((size_t)n_sel * (size_t)nframes_cap, 0);
    int err = 0;
    DecParams P;
    P.bytes = bytes; P.starts = starts; P.nbytes = nbytes; P.n_sel = n_sel; P.stream_size = stream_size;
    P.nch = nch; P.first = first_decode; P.n_decode = n_decode; P.data = store ? data : nullptr; P.crc = crc();
    P.meta = meta.data(); P.frame_off = fo.data(); P.nframes_cap = nframes_cap; P.stream_flag = flag.data();
    P.err = &err; P.verify_crc16 = 1; P.frame_flag = nullptr; P.status = status;
    fasim::launch(1, 1, 0, [&](int) {
        for (int64_t k = 0; k < n_sel; ++k) meta_body(P, k);
    });
    fasim::launch((int)n_sel * 3, 32, 0, [&](int b) { sync_scan_warp(P, (int64_t)(b / 3), (int64_t)(b % 3), 3); });
    const int64_t nwin = (first_decode + n_decode - 1) / bsh - first_decode / bsh + 1;
    TileParams TP;
    TP.D = P; TP.j0 = first_decode / bsh; TP.nwin = nwin; TP.frame_flag = fflag.data();
    TP.restore = 0; TP.offsets = nullptr; TP.gains = nullptr; TP.W = WinParams{};
    const int64_t total = n_sel * nwin;
    fasim::launch((int)((total + 31) / 32), 32, sizeof(TileShared) + 64, [&](int b) {
        if (store) tile_warp_body<false, true>(TP, (int64_t)b * 32, (TileShared*)fasim::smem());
        else tile_warp_body<false, false>(TP, (int64_t)b * 32, (TileShared*)fasim::smem());
    });
    fasim::launch((int)total, 32, 0, [&](int b) { crc_frame_warp(TP, (int64_t)b); });
    int walked = 0, general = 0;
    fasim::launch(1, 1, 0, [&](int) {
        // k_dec_frames<false>: one thread per item
        DecParams Q = P;
        Q.frame_flag = fflag.data();
        for (int64_t idx = 0; idx < total; ++idx) {
            const WorkItem it = resolve_item<false>(Q, WinParams{}, nwin, idx);
            const int64_t k = it.k;
            if (k < 0 || flag[(size_t)k]) continue;
            const int bs = meta[(size_t)k].blocksize;
            const int64_t j0 = it.first / bs, j1 = (it.first + it.n - 1) / bs;
            if (j1 - j0 + 1 > it.nwin) { if (it.jrel == 0) flag[(size_t)k] |= 1; continue; }
            const int64_t j = j0 + it.jrel;
            if (j > j1) continue;
            if (fflag[(size_t)(k * nframes_cap + j)]) general++;
            frame_body(Q, k, j, it.first, it.n, it.out);
        }
        // k_dec_walker_iso
        for (int64_t k = 0; k < n_sel; ++k) { if (flag[(size_t)k] && flag[(size_t)k] != 4) walked++; walker_body<true>(P, k); }
    });
    // k_dec_fill_failed (integer output)
    if (store && data)
        for (int64_t k = 0; k < n_sel; ++k)
            if (status[k] != 0) memset(data + k * n_decode * nch, 0, (size_t)(n_decode * nch) * 4);
    if (info) *info = walked + 1000 * general;
    return err;
}
}
