// hostsim.cpp -- TEST HARNESS ONLY.  Compiles the kernel bodies of flacarray_b200/csrc for the host
// with the OS-thread SIMT emulator of fa_simt.h so their logic can be unit-tested in the GPU-less
// build container (bit packing, CRC, slot placement and scan, frame index, decode, statistics, weighted sums).  This file
// is never linked into libflacarray_b200.so and the Python package never loads it: the product has no CPU path.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../flacarray_b200/csrc/fa_combine.h"
#include "../../flacarray_b200/csrc/fa_decode.h"
#include "../../flacarray_b200/csrc/fa_decode_tile.h"
#include "../../flacarray_b200/csrc/fa_encode.h"
#include "../../flacarray_b200/csrc/fa_encode_fixed.h"
#include "../../flacarray_b200/csrc/fa_stats.h"

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

namespace {

// Stage 3 of the product's decode (dec_items) over `total` work items: warp-tile decoder, its CRC pass, then the general
// per-thread decoder on the frames the tile path flagged (k_dec_tile, k_dec_crc, k_dec_frames).
template <bool WIN, bool STORE>
void dec_items(const TileParams& TP, int64_t total) {
    fasim::launch((int)((total + 31) / 32), 32, sizeof(TileShared) + 64, [&](int b) {
        tile_warp_body<WIN, STORE>(TP, (int64_t)b * 32, (TileShared*)fasim::smem());
    });
    fasim::launch((int)total, 32, 0, [&](int b) { crc_frame_warp<WIN>(TP, (int64_t)b); });
    DecParams P = TP.D;
    P.frame_flag = TP.frame_flag;
    fasim::launch(1, 1, 0, [&](int) {
        for (int64_t idx = 0; idx < total; ++idx) frames_item<WIN>(P, TP.W, TP.nwin, idx);
    });
}

// frames [first, first + n) of stream k that the tile path left to the general decoder (a stream it did not hand on)
int64_t general_frames(const DecParams& P, const unsigned char* fflag, int64_t k, int64_t first, int64_t n) {
    const int bs = P.meta[k].blocksize;
    int64_t c = 0;
    for (int64_t j = first / bs; j <= (first + n - 1) / bs; ++j) c += fflag[k * (int64_t)P.nframes_cap + j];
    return c;
}

// The product's decode on the host: dec_uniform (fab_decode, fab_decode_isolated, fab_verify; win == nullptr) or
// fab_decode_windows (win set: its records, win->bsh = the blocksize hint), with the same sizing and the same stages in the
// same order, each through its kernel body.  status set: per-stream isolation, and data == nullptr is fab_verify.
// *info = streams (windows) walked + 1000 * frames (window items) left to the general decoder, counted from the flags the
// stages leave behind.
int run_decode(const uint8_t* bytes, const long long* starts, const long long* nbytes, int64_t n_sel, int64_t stream_size,
               int nch, int64_t first, int64_t last, int blocksize_hint, const WinParams* win, int32_t* data, int* status,
               int* info) {
    if (info) *info = 0;
    int64_t first_decode = 0, n_decode = stream_size;
    if (!win && first >= 0 && last >= 0) {
        if (last > stream_size || first > stream_size - 1 || first >= last) return kErrDecodeSampleRange;
        first_decode = first;
        n_decode = last - first;
    }
    if (win && win->n_win <= 0) return win->n_win < 0 ? kErrDecodeSampleRange : 0;
    int bsh = 0, cap = 0;
    if (dec_frames_cap(stream_size, win ? win->bsh : blocksize_hint, &bsh, &cap)) return kErrAlloc;
    int err = 0;
    WinParams W{};
    std::vector<long long> item0;
    int64_t total = 0, nwin = 0;
    if (win) {                                                // k_win_prep, with two-warp blocks
        W = *win;
        W.bsh = bsh;
        item0.assign((size_t)W.n_win + 1, 0);
        W.item0 = item0.data();
        constexpr int kNT = 64;
        fasim::launch(1, kNT, (kNT / 32 + 1) * 8, [&](int) {
            long long* wpre = (long long*)fasim::smem();
            win_prep_cta<kNT>(W, n_sel, stream_size, &err, wpre, wpre + kNT / 32);
        });
        total = item0[(size_t)W.n_win];
        if (total == 0) return err;
    } else {
        nwin = (first_decode + n_decode - 1) / bsh - first_decode / bsh + 1;
        total = n_sel * nwin;
    }
    std::vector<StreamMeta> meta((size_t)n_sel);
    std::vector<long long> fo((size_t)n_sel * (size_t)(cap + 1), -1);
    std::vector<int> flag((size_t)n_sel, 0);
    std::vector<unsigned char> fflag((size_t)n_sel * (size_t)cap, 0);
    DecParams P;
    P.bytes = bytes; P.starts = starts; P.nbytes = nbytes; P.n_sel = n_sel; P.stream_size = stream_size;
    P.nch = nch; P.first = first_decode; P.n_decode = win ? 0 : n_decode; P.data = data; P.crc = crc();
    P.meta = meta.data(); P.frame_off = fo.data(); P.nframes_cap = cap; P.stream_flag = flag.data();
    P.err = &err; P.verify_crc16 = 1; P.frame_flag = fflag.data(); P.status = status;
    // dec_index_streams: k_dec_meta, then k_dec_sync (three warps striding over each stream's rows)
    fasim::launch((int)n_sel, 32, 0, [&](int b) { meta_warp(P, b); });
    fasim::launch((int)n_sel * 3, 32, 0, [&](int b) { sync_scan_warp(P, (int64_t)(b / 3), (int64_t)(b % 3), 3); });
    TileParams TP;
    TP.D = P; TP.j0 = first_decode / bsh; TP.nwin = nwin; TP.frame_flag = fflag.data();
    TP.restore = 0; TP.offsets = nullptr; TP.gains = nullptr; TP.W = W;
    if (win) dec_items<true, true>(TP, total);
    else if (data) dec_items<false, true>(TP, total);
    else dec_items<false, false>(TP, total);
    fasim::launch(1, 1, 0, [&](int) {                         // k_dec_walker / _iso / _win, one thread per stream or window
        if (win) for (int64_t w = 0; w < W.n_win; ++w) walker_win(P, W, w);
        else if (status) for (int64_t k = 0; k < n_sel; ++k) walker_body<true>(P, k);
        else for (int64_t k = 0; k < n_sel; ++k) walker_body(P, k);
    });
    if (!win && status && data) {                             // k_dec_fill_failed (integer output)
        fasim::launch(1, 1, 0, [&](int) {
            for (int64_t s = 0; s < n_sel; ++s) {
                if (nch == 2) fill_failed<unsigned long long>(status, (unsigned long long*)data, n_decode, 0ull, s, 0, 1);
                else fill_failed<uint32_t>(status, (uint32_t*)data, n_decode, 0u, s, 0, 1);
            }
        });
    }
    if (info && err == 0) {
        int64_t walked = 0, general = 0;
        const int64_t n_unit = win ? W.n_win : n_sel;
        for (int64_t i = 0; i < n_unit; ++i) {
            const int64_t k = win ? W.stream[i] : i;
            const int64_t a = win ? W.first[i] : first_decode, n = win ? W.last[i] - a : n_decode;
            if (n <= 0) continue;
            if (flag[(size_t)k] != 0 && flag[(size_t)k] != 4) walked++;
            if (flag[(size_t)k] == 0) general += general_frames(P, fflag.data(), k, a, n);
        }
        *info = (int)(walked + 1000 * general);
    }
    return err;
}

}  // namespace

extern "C" {

int64_t hs_encode_bound(int64_t n_stream, int64_t stream_size, int nch, int level) {
    LevelPreset lp = level_preset(level);
    int64_t nf = (stream_size + lp.blocksize - 1) / lp.blocksize;
    return n_stream * (stream_header_bytes((int)nf) + nf * (16 + 2 + (int64_t)nch * (lp.blocksize * 4 + 8)));
}

}  // extern "C"

namespace {
// The product's encode on the host.  stats_out / plans_out [n_stream * nframes * nch] and fixed_out [n_stream * nframes],
// when not null, receive the records k_enc_analyze and k_enc_design left for every (frame, channel) and whether
// k_enc_fixed took the frame (its records are then left zero).
int run_encode(const void* data, int dtype, int64_t n_stream, int64_t stream_size, int level, const void* quanta,
               uint8_t* out, int64_t cap, long long* starts, long long* nbytes, void* offsets, void* gains,
               long long* total, FrameStats* stats_out, FramePlan* plans_out, uint8_t* fixed_out) {
    LevelPreset lp = level_preset(level);
    int nch = (dtype == kI64 || dtype == kF64) ? 2 : 1;
    int nf = (int)((stream_size + lp.blocksize - 1) / lp.blocksize);
    std::vector<float> window_v(4096 + 4, 0.f), window_qt_v(4096 + 4, 0.f);   // 16-byte aligned views below
    float* window = (float*)(((uintptr_t)window_v.data() + 15) & ~(uintptr_t)15);
    float* window_qt = (float*)(((uintptr_t)window_qt_v.data() + 15) & ~(uintptr_t)15);
    make_tukey_window(window, lp.blocksize);
    if (lp.blocksize == 4096) permute_window_qt(window, window_qt);
    if (dtype == kF32) {
        const float* d = (const float*)data;
        for (int64_t s = 0; s < n_stream; ++s) {
            float mn = d[s * stream_size], mx = mn;
            for (int64_t i = 1; i < stream_size; ++i) { float v = d[s * stream_size + i]; if (v < mn) mn = v; if (v > mx) mx = v; }
            quant_params_f32(mn, mx, quanta != nullptr, quanta ? ((const float*)quanta)[s] : 0.f, (float*)offsets + s, (float*)gains + s);
        }
    } else if (dtype == kF64) {
        const double* d = (const double*)data;
        for (int64_t s = 0; s < n_stream; ++s) {
            double mn = d[s * stream_size], mx = mn;
            for (int64_t i = 1; i < stream_size; ++i) { double v = d[s * stream_size + i]; if (v < mn) mn = v; if (v > mx) mx = v; }
            quant_params_f64(mn, mx, quanta != nullptr, quanta ? ((const double*)quanta)[s] : 0., (double*)offsets + s, (double*)gains + s);
        }
    }
    std::vector<long long> ends((size_t)n_stream, 0);
    std::vector<unsigned long long> desc((size_t)(n_stream * nf), 0ull);
    for (int64_t s = 0; s < n_stream; ++s) starts[s] = -1;
    uint32_t ticket = 0;
    int err = 0;
    static EncTables tab;
    static bool tab_ready = false;
    if (!tab_ready) { enc_tables_init(&tab); tab_ready = true; }
    EncParams P;
    P.data = data; P.dtype = dtype; P.offsets = offsets; P.gains = gains;
    P.n_stream = n_stream; P.stream_size = stream_size; P.nch = nch;
    P.blocksize = lp.blocksize; P.nframes = nf;
    P.max_lpc_order = lp.max_lpc_order; P.max_porder = lp.max_porder;
    P.qlp_precision = lp.blocksize <= 384 ? 13 : (lp.blocksize <= 1152 ? 14 : 15);
    P.window = window; P.window_qt = window_qt; P.crc = crc(); P.tab = &tab;
    P.out = out; P.out_capacity = cap; P.starts = starts; P.ends = ends.data(); P.desc = desc.data();
    P.ticket = &ticket; P.err = &err; P.hdr_bytes = stream_header_bytes(nf);
    // the three encoder kernels: analyze (one CTA per frame) -> design (one thread per record) -> encode
    const int64_t total_frames = n_stream * nf;
    std::vector<FrameStats> stats((size_t)(total_frames * nch));
    std::vector<FramePlan> plans((size_t)(total_frames * nch) + 1);
    // ldg128 needs 16-byte aligned plan records
    FramePlan* plan_base = (FramePlan*)(((uintptr_t)plans.data() + 15) & ~(uintptr_t)15);
    if ((uintptr_t)plan_base + (size_t)(total_frames * nch) * sizeof(FramePlan) > (uintptr_t)(plans.data() + plans.size()))
        return kErrAlloc;
    std::vector<PlanHeader> hdrs((size_t)(total_frames * nch));
    P.stats = stats.data(); P.plans = plan_base; P.hdrs = hdrs.data(); P.g_begin = 0; P.g_end = (uint32_t)total_frames;
    // slots for the frames of the (single) batch (analyze parks samples there, encode writes frames)
    const int64_t slot_bytes = (int64_t)((16 + 2 + (int64_t)nch * (lp.blocksize * 4 + 8) + 15) & ~15ll);
    std::vector<uint32_t> slots_w((size_t)(total_frames * slot_bytes / 4) + 8);
    std::vector<uint32_t> fsize((size_t)total_frames);
    unsigned long long base = 0;
    P.slots = (uint8_t*)(((uintptr_t)slots_w.data() + 15) & ~(uintptr_t)15); P.slot_bytes = slot_bytes;
    P.fsize = fsize.data(); P.base = &base;
    if (lp.blocksize == kFxBs && getenv("HS_NO_FIXED") == nullptr) {
        // levels 0..2: the warp-per-frame encoder first (the product's k_enc_fixed), the kernels below take the rest
        fasim::launch((int)total_frames, 32, sizeof(FxShared) + 16, [&](int b) {
            FxShared* ws = (FxShared*)(((uintptr_t)fasim::smem() + 15) & ~(uintptr_t)15);
            fixed_frame_warp(P, (uint32_t)b, ws);
        });
    }
    if (fixed_out)
        for (int64_t g = 0; g < total_frames; ++g) fixed_out[g] = fsize[(size_t)g] != 0u;
    fasim::launch(1, kEncThreads, sizeof(AnShared) + 16, [&](int) {
        AnShared* ash = (AnShared*)fasim::smem();
        if (lp.blocksize == kMaxBs) analyze_fill_window(P, ash);
        fa::sync();
        for (uint32_t g = 0; g < (uint32_t)total_frames; ++g) {
            if (lp.max_lpc_order > 8) { analyze_frame_cta<12, true>(P, g, ash); analyze_frame_cta<12, false>(P, g, ash); }
            else { analyze_frame_cta<8, true>(P, g, ash); analyze_frame_cta<8, false>(P, g, ash); }
        }
    });
    fasim::launch(1, 1, 0, [&](int) {
        for (int64_t i = 0; i < total_frames * nch; ++i) design_frame(P, i);
    });
    if (stats_out) memcpy(stats_out, stats.data(), (size_t)(total_frames * nch) * sizeof(FrameStats));
    if (plans_out) memcpy(plans_out, plan_base, (size_t)(total_frames * nch) * sizeof(FramePlan));
    // persistent CTAs: the emulator runs blocks one after the other, so one block drains every ticket
    fasim::launch(1, kEncThreads, enc_smem_bytes(nch), [&](int) {
        if (lp.max_lpc_order > 8) encode_frames_cta<12, true>(P, fasim::smem());
        else encode_frames_cta<8, true>(P, fasim::smem());
    });
    // the frames that are not full (one block striding over every frame, like the ticket kernel: it passes over the full ones)
    fasim::launch(1, kEncThreads, enc_smem_bytes(nch), [&](int) {
        if (lp.max_lpc_order > 8) encode_frames_cta<12, false>(P, fasim::smem(), 0, 1);
        else encode_frames_cta<8, false>(P, fasim::smem(), 0, 1);
    });
    fasim::launch(1, kScanThreads, (kScanThreads / 32 + 1) * 8, [&](int) { scan_batch_cta(P, (unsigned long long*)fasim::smem()); });
    fasim::launch((int)total_frames, 128, sizeof(CompactShared), [&](int b) {
        compact_frame_cta(P, (uint32_t)b, (CompactShared*)fasim::smem(), P.fsize[b], P.desc[P.g_begin + (uint32_t)b]);
    });
    fasim::launch(1, 1, 0, [&](int) {
        for (int64_t s = 0; s < n_stream; ++s)
            for (int f = 0; f < nf; ++f) finalize_entry(P, s, f, nbytes, total);
    });
    return err;
}
}  // namespace

extern "C" {

// dtype: 0 i32, 1 i64, 2 f32, 3 f64.  quanta may be NULL (auto) for float input.
int hs_encode(const void* data, int dtype, int64_t n_stream, int64_t stream_size, int level, const void* quanta,
              uint8_t* out, int64_t cap, long long* starts, long long* nbytes, void* offsets, void* gains,
              long long* total) {
    return run_encode(data, dtype, n_stream, stream_size, level, quanta, out, cap, starts, nbytes, offsets, gains, total,
                      nullptr, nullptr, nullptr);
}

// hs_encode that also returns the analysis and design records of every (frame, channel) (see run_encode)
int hs_encode_records(const void* data, int dtype, int64_t n_stream, int64_t stream_size, int level, const void* quanta,
                      uint8_t* out, int64_t cap, long long* starts, long long* nbytes, void* offsets, void* gains,
                      long long* total, FrameStats* stats_out, FramePlan* plans_out, uint8_t* fixed_out) {
    return run_encode(data, dtype, n_stream, stream_size, level, quanta, out, cap, starts, nbytes, offsets, gains, total,
                      stats_out, plans_out, fixed_out);
}

int hs_record_sizes(int* stats_bytes, int* plan_bytes) {
    *stats_bytes = (int)sizeof(FrameStats);
    *plan_bytes = (int)sizeof(FramePlan);
    return 0;
}

// mode 0: parallel-path emulation (meta -> sync scan -> per-frame decode -> walker for flagged streams)
// mode 1: walker only
// (modes 0 and 1: the serial reference the other paths are compared against)
// mode 2: the product's fab_decode (run_decode); *n_walked = streams walked + 1000 * frames left to the general decoder
int hs_decode(const uint8_t* bytes, const long long* starts, const long long* nbytes, int64_t n_sel,
              int64_t stream_size, int nch, int64_t first, int64_t last, int32_t* data, int mode, int* n_walked) {
    if (mode == 2)
        return run_decode(bytes, starts, nbytes, n_sel, stream_size, nch, first, last,
                          n_sel > 0 ? stream_blocksize_hint(bytes + starts[0], nbytes[0]) : 0, nullptr, data, nullptr,
                          n_walked);
    int64_t n_decode = stream_size;
    int64_t first_decode = 0;
    if (first >= 0 && last >= 0) {
        if (last > stream_size || first > stream_size - 1 || first >= last) return kErrDecodeSampleRange;
        first_decode = first;
        n_decode = last - first;
    }
    int nframes_cap = (int)((stream_size + 15) / 16) + 1;  // smallest legal blocksize is 16
    if (nframes_cap > (1 << 22)) nframes_cap = 1 << 22;
    std::vector<StreamMeta> meta((size_t)n_sel);
    std::vector<long long> fo((size_t)n_sel * (size_t)(nframes_cap + 1), -1);
    std::vector<int> flag((size_t)n_sel, 0);
    int err = 0;
    DecParams P;
    P.bytes = bytes; P.starts = starts; P.nbytes = nbytes; P.n_sel = n_sel; P.stream_size = stream_size;
    P.nch = nch; P.first = first_decode; P.n_decode = n_decode; P.data = data; P.crc = crc();
    P.meta = meta.data(); P.frame_off = fo.data(); P.nframes_cap = nframes_cap; P.stream_flag = flag.data();
    P.err = &err; P.verify_crc16 = 1; P.frame_flag = nullptr;
    fasim::launch(1, 1, 0, [&](int) {
        for (int64_t k = 0; k < n_sel; ++k) meta_body(P, k);
        if (mode == 1) for (int64_t k = 0; k < n_sel; ++k) if (flag[(size_t)k] == 0) flag[(size_t)k] = 1;
        if (mode == 0) {
            for (int64_t k = 0; k < n_sel; ++k)
                for (int64_t p = 0; p < nbytes[k]; ++p) sync_body(P, k, p);
            for (int64_t k = 0; k < n_sel; ++k) {
                if (flag[(size_t)k]) continue;
                int bs = meta[(size_t)k].blocksize;
                int64_t j0 = first_decode / bs, j1 = (first_decode + n_decode - 1) / bs;
                for (int64_t j = j0; j <= j1; ++j) frame_body(P, k, j);
            }
        }
        int walked = 0;
        for (int64_t k = 0; k < n_sel; ++k) { if (flag[(size_t)k] && flag[(size_t)k] != 4) walked++; walker_body(P, k); }
        if (n_walked) *n_walked = walked;
    });
    return err;
}

int hs_float_to_int(const void* data, int is64, int64_t n_stream, int64_t stream_size, const void* quanta, void* out,
                    void* offsets, void* gains) {
    for (int64_t s = 0; s < n_stream; ++s) {
        if (!is64) {
            const float* d = (const float*)data + s * stream_size;
            float mn = d[0], mx = d[0];
            for (int64_t i = 1; i < stream_size; ++i) { if (d[i] < mn) mn = d[i]; if (d[i] > mx) mx = d[i]; }
            float off, gain;
            quant_params_f32(mn, mx, quanta != nullptr, quanta ? ((const float*)quanta)[s] : 0.f, &off, &gain);
            ((float*)offsets)[s] = off; ((float*)gains)[s] = gain;
            for (int64_t i = 0; i < stream_size; ++i) ((int32_t*)out)[s * stream_size + i] = quant_f32(d[i], off, gain);
        } else {
            const double* d = (const double*)data + s * stream_size;
            double mn = d[0], mx = d[0];
            for (int64_t i = 1; i < stream_size; ++i) { if (d[i] < mn) mn = d[i]; if (d[i] > mx) mx = d[i]; }
            double off, gain;
            quant_params_f64(mn, mx, quanta != nullptr, quanta ? ((const double*)quanta)[s] : 0., &off, &gain);
            ((double*)offsets)[s] = off; ((double*)gains)[s] = gain;
            for (int64_t i = 0; i < stream_size; ++i) ((long long*)out)[s * stream_size + i] = quant_f64(d[i], off, gain);
        }
    }
    return 0;
}

void hs_int_to_float(const void* data, int is64, int64_t n_stream, int64_t stream_size, const void* offsets,
                     const void* gains, void* out) {
    for (int64_t s = 0; s < n_stream; ++s) {
        if (!is64) {
            float c = restore_coeff_f32(((const float*)gains)[s]);
            for (int64_t i = 0; i < stream_size; ++i)
                ((float*)out)[s * stream_size + i] = restore_f32(((const int32_t*)data)[s * stream_size + i], ((const float*)offsets)[s], c);
        } else {
            double c = restore_coeff_f64(((const double*)gains)[s]);
            for (int64_t i = 0; i < stream_size; ++i)
                ((double*)out)[s * stream_size + i] = restore_f64(((const long long*)data)[s * stream_size + i], ((const double*)offsets)[s], c);
        }
    }
}

uint32_t hs_crc16(const uint8_t* p, int64_t n) { return crc16_bytes(crc(), p, n); }

// the analysis pass's single-precision quantiser against the reference operation sequence (fa_quant.h)
int64_t hs_quant_fast_mismatches(const float* x, int64_t n, float off, float gain) {
    int64_t bad = 0;
    for (int64_t i = 0; i < n; ++i)
        if (quant_f32_fast(x[i], off, gain, gain > 0.0f) != quant_f32(x[i], off, gain)) bad++;
    return bad;
}

// fab_decode_isolated (data != NULL) / fab_verify (data == NULL, first = last = -1): status[n_sel] receives every
// stream's bits, the return value is the call-level error mask.
int hs_decode_isolated(const uint8_t* bytes, const long long* starts, const long long* nbytes, int64_t n_sel,
                       int64_t stream_size, int nch, int64_t first, int64_t last, int32_t* data, int* status, int* info) {
    return run_decode(bytes, starts, nbytes, n_sel, stream_size, nch, first, last,
                      n_sel > 0 ? stream_blocksize_hint(bytes + starts[0], nbytes[0]) : 0, nullptr, data, status, info);
}

// fab_decode_windows: window w decodes samples [win_first[w], win_last[w]) of stream slot win_stream[w] to
// data[win_out[w] * nch ...]; bsh: the blocksize hint.  *info = windows walked + 1000 * items left to the general decoder.
int hs_decode_windows(const uint8_t* bytes, const long long* starts, const long long* nbytes, int64_t n_sel,
                      int64_t stream_size, int nch, const long long* win_stream, const long long* win_first,
                      const long long* win_last, const long long* win_out, int64_t n_win, int bsh, int32_t* data,
                      int* info) {
    WinParams W{};
    W.stream = win_stream; W.first = win_first; W.last = win_last; W.out = win_out; W.n_win = n_win; W.bsh = bsh;
    return run_decode(bytes, starts, nbytes, n_sel, stream_size, nch, -1, -1, 0, &W, data, nullptr, info);
}

// Stage 1 alone, with the frame tables sized as the decode sizes them: the product's warp body (warp != 0) or the serial
// reference meta_body.  meta [n_sel] StreamMeta, frame_off [n_sel][cap + 1] (filled with -1 by the caller), flag and
// status [n_sel].  Returns cap, or -1 when the tables would be too large.
int hs_meta(const uint8_t* bytes, const long long* starts, const long long* nbytes, int64_t n_sel, int64_t stream_size,
            int nch, int warp, StreamMeta* meta, long long* frame_off, int64_t frame_off_len, int* flag, int* status) {
    int bsh = 0, cap = 0;
    if (dec_frames_cap(stream_size, stream_blocksize_hint(bytes + starts[0], nbytes[0]), &bsh, &cap)) return -1;
    if (frame_off_len < n_sel * (int64_t)(cap + 1)) return -1;
    int err = 0;
    DecParams P{};
    P.bytes = bytes; P.starts = starts; P.nbytes = nbytes; P.n_sel = n_sel; P.stream_size = stream_size; P.nch = nch;
    P.meta = meta; P.frame_off = frame_off; P.nframes_cap = cap; P.stream_flag = flag; P.err = &err; P.status = status;
    if (warp) fasim::launch((int)n_sel, 32, 0, [&](int b) { meta_warp(P, b); });
    else for (int64_t k = 0; k < n_sel; ++k) meta_body(P, k);
    return cap;
}

// fab_row_stats with the piece length as a parameter (piece <= 0: the library's kStatsPieceBytes), so that small rows
// exercise bins spanning many pieces.  bin == 0: one bin per row.  Returns 0 or the error bits fab_row_stats returns
// for its arguments.  *n_pieces receives nbins * ppb (the reducer's warps per row), *ppb_out the pieces per bin.
int hs_row_stats(const void* rows, int is_int64, int64_t n_rows, int64_t n, int64_t bin, int64_t piece, const void* offsets,
                 const void* gains, const int* status, long long* count, void* mn, void* mx, double* mean, double* std,
                 int64_t* n_pieces, int64_t* ppb_out) {
    StatsParams P{};
    const int rc = stats_geometry(n_rows, n, bin, is_int64, &P, piece);
    if (rc) return rc;
    std::vector<StatPart> part(P.ppb > 1 ? (size_t)(n_rows * P.nbins * P.ppb) : 0);
    P.part = part.data();
    P.rows = rows; P.offsets = offsets; P.gains = gains; P.status = status;
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

// fab_combine_rows on host memory, with 32-thread blocks (one block per (segment, column chunk)) so that small arrays span
// several column chunks and long segments several row tiles.
namespace {
constexpr int kCombineSimThreads = 32;

template <bool I64, bool FLT>
void combine(const CombineParams& P, int64_t gx) {
    fasim::launch((int)(gx * P.n_seg), kCombineSimThreads, kCombineSimThreads * sizeof(CombineRow), [&](int b) {
        combine_segment_cta<I64, FLT, kCombineSimThreads>(P, b / gx, (int64_t)(b % gx) * (kCombineSimThreads * kCombineCols),
                                                          (CombineRow*)fasim::smem());
    });
}
}  // namespace

extern "C" {
// Returns 0, or -1 for arguments fab_combine_rows rejects before launching; *err receives the error bits the segment
// checks set.
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
    const int64_t gx = (n + kCombineSimThreads * kCombineCols - 1) / (kCombineSimThreads * kCombineCols);
    if (is_int64) {
        if (offsets) combine<true, true>(P, gx);
        else combine<true, false>(P, gx);
    } else {
        if (offsets) combine<false, true>(P, gx);
        else combine<false, false>(P, gx);
    }
    return 0;
}
}
