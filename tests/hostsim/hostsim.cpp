// hostsim.cpp -- TEST HARNESS ONLY.  Compiles the kernel bodies of flacarray_b200/csrc for the host
// with the OS-thread SIMT emulator of fa_simt.h so their logic can be unit-tested in the GPU-less
// build container (bit packing, CRC, slot placement and scan, frame index, decode).  This file is never
// linked into libflacarray_b200.so and the Python package never loads it: the product has no CPU path.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../flacarray_b200/csrc/fa_decode.h"
#include "../../flacarray_b200/csrc/fa_decode_tile.h"
#include "../../flacarray_b200/csrc/fa_encode.h"
#include "../../flacarray_b200/csrc/fa_encode_fixed.h"

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

int64_t hs_encode_bound(int64_t n_stream, int64_t stream_size, int nch, int level) {
    LevelPreset lp = level_preset(level);
    int64_t nf = (stream_size + lp.blocksize - 1) / lp.blocksize;
    return n_stream * (stream_header_bytes((int)nf) + nf * (16 + 2 + (int64_t)nch * (lp.blocksize * 4 + 8)));
}

// dtype: 0 i32, 1 i64, 2 f32, 3 f64.  quanta may be NULL (auto) for float input.
int hs_encode(const void* data, int dtype, int64_t n_stream, int64_t stream_size, int level, const void* quanta,
              uint8_t* out, int64_t cap, long long* starts, long long* nbytes, void* offsets, void* gains,
              long long* total) {
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

// mode 0: parallel-path emulation (meta -> sync scan -> per-frame decode -> walker for flagged streams)
// mode 1: walker only
int hs_decode(const uint8_t* bytes, const long long* starts, const long long* nbytes, int64_t n_sel,
              int64_t stream_size, int nch, int64_t first, int64_t last, int32_t* data, int mode, int* n_walked) {
    int64_t n_decode = stream_size;
    int64_t first_decode = 0;
    if (first >= 0 && last >= 0) {
        if (last > stream_size || first > stream_size - 1 || first >= last) return kErrDecodeSampleRange;
        first_decode = first;
        n_decode = last - first;
    }
    int nframes_cap = (int)((stream_size + 15) / 16) + 1;  // smallest legal blocksize is 16
    if (nframes_cap > (1 << 22)) nframes_cap = 1 << 22;
    // mode 2 sizes the frame tables and the item space the way fab_decode does: from the blocksize hint the host
    // reads from the FIRST stream's STREAMINFO (min blocksize; 4096 without one), clamped to >= 16
    int bsh = 4096;
    if (mode == 2) {
        const uint8_t* s0 = n_sel > 0 ? bytes + starts[0] : nullptr;
        if (s0 && nbytes[0] >= 12 && memcmp(s0, "fLaC", 4) == 0 && ((s0[8] << 8) | s0[9]) > 0) bsh = (s0[8] << 8) | s0[9];
        if (bsh < 16) bsh = 16;
        nframes_cap = (int)((stream_size + bsh - 1) / bsh);
    }
    std::vector<StreamMeta> meta((size_t)n_sel);
    std::vector<long long> fo((size_t)n_sel * (size_t)(nframes_cap + 1), -1);
    std::vector<int> flag((size_t)n_sel, 0);
    int err = 0;
    DecParams P;
    P.bytes = bytes; P.starts = starts; P.nbytes = nbytes; P.n_sel = n_sel; P.stream_size = stream_size;
    P.nch = nch; P.first = first_decode; P.n_decode = n_decode; P.data = data; P.crc = crc();
    P.meta = meta.data(); P.frame_off = fo.data(); P.nframes_cap = nframes_cap; P.stream_flag = flag.data();
    P.err = &err; P.verify_crc16 = 1; P.frame_flag = nullptr;
    std::vector<unsigned char> fflag((size_t)n_sel * (size_t)nframes_cap, 0);
    if (mode == 2) {
        // throughput path emulation: meta -> sync scan -> warp-tile kernel -> general decoder on the
        // flagged frames -> walker on the flagged streams
        fasim::launch(1, 1, 0, [&](int) {
            for (int64_t k = 0; k < n_sel; ++k) meta_body(P, k);
        });
        // the product's warp-cooperative scan (three warps striding over each stream's rows)
        fasim::launch((int)n_sel * 3, 32, 0, [&](int b) { sync_scan_warp(P, (int64_t)(b / 3), (int64_t)(b % 3), 3); });
        int64_t nwin = (first_decode + n_decode - 1) / bsh - first_decode / bsh + 1;
        TileParams TP;
        TP.D = P; TP.j0 = first_decode / bsh; TP.nwin = nwin; TP.frame_flag = fflag.data();
        TP.restore = 0; TP.offsets = nullptr; TP.gains = nullptr;
        int64_t total = n_sel * nwin;
        // the product launches the tile decoder without the fused CRC and checks it in k_dec_crc
        fasim::launch((int)((total + 31) / 32), 32, sizeof(TileShared) + 64, [&](int b) {
            tile_warp_body(TP, (int64_t)b * 32, (TileShared*)fasim::smem());
        });
        fasim::launch((int)total, 32, 0, [&](int b) { crc_frame_warp(TP, (int64_t)b); });
        int walked = 0, general = 0;
        fasim::launch(1, 1, 0, [&](int) {
            DecParams Q = P;
            Q.frame_flag = fflag.data();
            for (int64_t k = 0; k < n_sel; ++k) {
                if (flag[(size_t)k]) continue;
                int bs = meta[(size_t)k].blocksize;
                int64_t j0 = first_decode / bs, j1 = (first_decode + n_decode - 1) / bs;
                for (int64_t j = j0; j <= j1; ++j) { if (fflag[(size_t)(k * nframes_cap + j)]) general++; frame_body(Q, k, j); }
            }
            for (int64_t k = 0; k < n_sel; ++k) { if (flag[(size_t)k] && flag[(size_t)k] != 4) walked++; walker_body(P, k); }
        });
        if (n_walked) *n_walked = walked + 1000 * general;
        return err;
    }
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
}
