// hostsim_windows.cpp -- TEST HARNESS ONLY.  Host build of the per-stream window decode (fab_decode_windows) with the
// OS-thread SIMT emulator of fa_simt.h, next to hostsim.cpp: the same kernel bodies of flacarray_b200/csrc driven the
// way the product drives them, so the window index space can be unit-tested without a GPU.  Never linked into
// libflacarray_b200.so and never loaded by the Python package.
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

// fab_decode_windows emulation, driven like hs_decode mode 2: item space (k_win_prep) -> meta -> sync scan -> warp-tile
// kernel -> general decoder on the flagged frames -> walker per window of a flagged stream.  Window w decodes samples
// [win_first[w], win_last[w]) of stream slot win_stream[w] to data[win_out[w] * nch ...].  bsh: hinted blocksize.
// *info = windows walked + 1000 * items left to the general decoder.
int hs_decode_windows(const uint8_t* bytes, const long long* starts, const long long* nbytes, int64_t n_sel,
                      int64_t stream_size, int nch, const long long* win_stream, const long long* win_first,
                      const long long* win_last, const long long* win_out, int64_t n_win, int bsh, int32_t* data,
                      int* info) {
    int nframes_cap = (int)((stream_size + 15) / 16) + 1;
    if (nframes_cap > (1 << 22)) nframes_cap = 1 << 22;
    std::vector<StreamMeta> meta((size_t)n_sel);
    std::vector<long long> fo((size_t)n_sel * (size_t)(nframes_cap + 1), -1);
    std::vector<int> flag((size_t)n_sel, 0);
    std::vector<unsigned char> fflag((size_t)n_sel * (size_t)nframes_cap, 0);
    std::vector<long long> item0((size_t)n_win + 1, 0);
    int err = 0;
    WinParams W;
    W.stream = win_stream; W.first = win_first; W.last = win_last; W.out = win_out; W.item0 = item0.data();
    W.n_win = n_win; W.bsh = bsh;
    for (int64_t w = 0; w < n_win; ++w) {
        int64_t cnt = 0;
        if (win_valid(W, w, n_sel, stream_size)) cnt = frames_in_window(win_first[w], win_last[w] - win_first[w], bsh);
        else err |= kErrDecodeSampleRange;
        item0[(size_t)w + 1] = item0[(size_t)w] + cnt;
    }
    const int64_t total = item0[(size_t)n_win];
    if (info) *info = 0;
    if (total == 0) return err;
    DecParams P;
    P.bytes = bytes; P.starts = starts; P.nbytes = nbytes; P.n_sel = n_sel; P.stream_size = stream_size;
    P.nch = nch; P.first = 0; P.n_decode = 0; P.data = data; P.crc = crc();
    P.meta = meta.data(); P.frame_off = fo.data(); P.nframes_cap = nframes_cap; P.stream_flag = flag.data();
    P.err = &err; P.verify_crc16 = 1; P.frame_flag = fflag.data();
    fasim::launch(1, 1, 0, [&](int) {
        for (int64_t k = 0; k < n_sel; ++k) meta_body(P, k);
    });
    fasim::launch((int)n_sel * 3, 32, 0, [&](int b) { sync_scan_warp(P, (int64_t)(b / 3), (int64_t)(b % 3), 3); });
    TileParams TP;
    TP.D = P; TP.j0 = 0; TP.nwin = 0; TP.frame_flag = fflag.data();
    TP.restore = 0; TP.offsets = nullptr; TP.gains = nullptr; TP.W = W;
    fasim::launch((int)((total + 31) / 32), 32, sizeof(TileShared) + 64, [&](int b) {
        tile_warp_body<true>(TP, (int64_t)b * 32, (TileShared*)fasim::smem());
    });
    fasim::launch((int)total, 32, 0, [&](int b) { crc_frame_warp<true>(TP, (int64_t)b); });
    int walked = 0, general = 0;
    fasim::launch(1, 1, 0, [&](int) {
        // k_dec_frames<true>: one thread per item
        for (int64_t idx = 0; idx < total; ++idx) {
            const WorkItem it = resolve_item<true>(P, W, 0, idx);
            const int64_t k = it.k;
            if (k < 0 || flag[(size_t)k]) continue;
            const int bs = meta[(size_t)k].blocksize;
            const int64_t j0 = it.first / bs, j1 = (it.first + it.n - 1) / bs;
            if (j1 - j0 + 1 > it.nwin) { if (it.jrel == 0) flag[(size_t)k] |= 1; continue; }
            const int64_t j = j0 + it.jrel;
            if (j > j1) continue;
            if (fflag[(size_t)(k * nframes_cap + j)]) general++;
            frame_body(P, k, j, it.first, it.n, it.out);
        }
        // k_dec_walker_win: one thread per window
        for (int64_t w = 0; w < n_win; ++w) {
            if (!win_valid(W, w, n_sel, stream_size) || win_last[w] == win_first[w]) continue;
            const int f = flag[(size_t)win_stream[w]];
            if (f && f != 4) walked++;
            walker_body(P, win_stream[w], win_first[w], win_last[w] - win_first[w], win_out[w]);
        }
    });
    if (info) *info = walked + 1000 * general;
    return err;
}
}
