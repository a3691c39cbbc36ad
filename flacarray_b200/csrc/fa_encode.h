// fa_encode.h -- FLAC encoder bodies.
//
// Replaces the libFLAC encoder the reference drives per stream in compress.c:184-237 (serial) and
// compress.c:337-390 (OpenMP), plus the byte bookkeeping of the write callbacks
// (compress.c:13-104) and the final prefix-sum/concatenation (compress.c:402-429).
//
// Five kernels per batch of <= 64 Ki (stream, frame) units (see "Fast path" below):
//   analyze_frame_cta  (k_enc_analyze)  statistics of every (frame, channel)            128-thread CTA per frame
//   design_frame       (k_enc_design)   predictor design                                one thread per (frame, channel)
//   encode_frames_cta  (k_encode)       residual, Rice, packing, CRC-16 -> frame slot   persistent 128-thread CTAs
//   scan_batch_cta     (k_enc_scan)     frame sizes -> byte offsets                     one CTA
//   compact_frame_cta  (k_enc_compact)  slot -> final place                             CTA per frame
//
// Code paths of k_encode per (frame, channel):
//   * full path   -- 4096-sample frames: rolled 8-sample sub-blocks, 32-bit integer work for narrow samples
//     (|x| < 2^22; the coefficient precision is lowered until sum|q|*max|x| provably fits, as libFLAC does
//     for <= 16-bit input), 64-bit work for wide samples (the low word of an int64), wasted bits;
//   * short path  -- 64 <= blocksize < 4096 (last frame of a stream, blocksize-1152 levels): the same stages
//     with the thread's 32 samples resident in registers and a warp-level Rice partition search;
//   * general path -- anything else (tiny frames, residuals that do not fit 32 bits, VERBATIM subframes):
//     64-bit arithmetic and per-sample bounds checks.  Slow, but only reached by frames the others reject.
#pragma once
#include "fa_bits.h"
#include "fa_quant.h"
#include <math.h>

namespace fa {

constexpr int kEncThreads = 128;
constexpr int kEncWarps = kEncThreads / 32;
constexpr int kSpt = 32;                     // samples per thread
constexpr int kMaxBs = kEncThreads * kSpt;   // 4096
constexpr int kMaxOrd = 12;                  // libFLAC presets never exceed order 12
constexpr int kMaxParts = 64;                // partition order <= 6
constexpr int kX32Len = 8704;                // >= words of the largest (2-channel VERBATIM) frame + 1
constexpr int kNarrowBits = 22;              // fast path: -2^22 <= x < 2^22

enum { kI32 = 0, kI64 = 1, kF32 = 2, kF64 = 3 };

// libFLAC compression_levels_[] (SURVEY App. B): blocksize for set_blocksize(0), max LPC order, max
// residual partition order.  Stereo decorrelation is not searched: on (low word, high word) pairs it
// buys < 0.01 % (SURVEY 8a-E), so 2-channel frames are always "independent".
struct LevelPreset { int blocksize, max_lpc_order, max_porder; };
inline LevelPreset level_preset(int level) {
    const LevelPreset t[9] = {{1152, 0, 3}, {1152, 0, 3}, {1152, 0, 3}, {4096, 6, 4}, {4096, 8, 4},
                              {4096, 8, 5}, {4096, 8, 6}, {4096, 12, 6}, {4096, 12, 6}};
    return t[level];
}

// tukey(0.5) window of the nominal blocksize (libFLAC window.c FLAC__window_tukey); short last frames
// use its prefix.  Host side, computed once per (context, blocksize).
inline void make_tukey_window(float* w, int L) {
    for (int n = 0; n < L; ++n) w[n] = 1.0f;
    int Np = (int)(0.5f / 2.0f * (float)L) - 1;
    if (Np > 0) {
        for (int n = 0; n <= Np; ++n) {
            w[n] = (float)(0.5 - 0.5 * cos(3.14159265358979323846 * n / Np));
            w[L - Np - 1 + n] = (float)(0.5 - 0.5 * cos(3.14159265358979323846 * (n + Np) / Np));
        }
    }
}

// the window in the order the full-frame analysis reads it: element (quad q, thread t, e) = w[32 t + 4 q + e]
inline void permute_window_qt(const float* w, float* out) {
    for (int i = 0; i < kMaxBs; ++i) out[((((i >> 2) & 7) * kEncThreads + (i >> 5)) << 2) + (i & 3)] = w[i];
}

// CRC-16 position tables (host-initialised): x32[m] = x^(32 m) mod P, inv8[k] = x^(-8 k) mod P.
struct EncTables {
    uint16_t x32[kX32Len];
    uint16_t inv8[4];
};
inline uint32_t gf16_mul_host(uint32_t a, uint32_t b) {
    uint32_t r = 0;
    for (int i = 15; i >= 0; --i) {
        r <<= 1;
        if (r & 0x10000u) r ^= 0x18005u;
        if ((b >> i) & 1u) r ^= a;
    }
    return r & 0xFFFFu;
}
inline void enc_tables_init(EncTables* t) {
    uint32_t x8 = 1;
    for (int i = 0; i < 8; ++i) { x8 <<= 1; if (x8 & 0x10000u) x8 ^= 0x18005u; }
    uint32_t x32 = gf16_mul_host(gf16_mul_host(x8, x8), gf16_mul_host(x8, x8));
    uint32_t v = 1;
    for (int m = 0; m < kX32Len; ++m) { t->x32[m] = (uint16_t)v; v = gf16_mul_host(v, x32); }
    // P = (x + 1)(x^15 + x + 1): x has multiplicative order 32767 mod P, so x^-8 = x^(32767 - 8)
    uint32_t inv = 1, base = 2;
    for (int e = 32767 - 8; e; e >>= 1) { if (e & 1) inv = gf16_mul_host(inv, base); base = gf16_mul_host(base, base); }
    t->inv8[0] = 1;
    for (int k = 1; k < 4; ++k) t->inv8[k] = (uint16_t)gf16_mul_host(t->inv8[k - 1], inv);
}

// Bytes before the first frame of every stream: "fLaC" + STREAMINFO + APPLICATION(faB2 table, last).
inline int stream_header_bytes(int nframes) { return 4 + 4 + 34 + 4 + 8 + 3 * nframes; }

struct FrameStats;
struct FramePlan;
struct PlanHeader;

struct EncParams {
    const void* data;
    int dtype;                 // kI32 / kI64 / kF32 / kF64
    const void* offsets;       // per-stream float/double (kF32/kF64), written by the quantise pre-pass
    const void* gains;
    int64_t n_stream, stream_size;
    int nch;
    int blocksize, nframes;    // per stream
    int max_lpc_order, max_porder, qlp_precision;
    const float* window;       // tukey(0.5) of length blocksize, zero-padded to kMaxBs floats
    const float* window_qt;    // the same window for blocksize kMaxBs in the parked [quad][thread][4] order
    const CrcTables* crc;
    const EncTables* tab;
    uint8_t* out;
    int64_t out_capacity;
    long long* starts;         // [n_stream] byte offset of every stream; must be preset to -1
    long long* ends;           // [n_stream]
    unsigned long long* desc;  // [n_stream * nframes] inclusive byte prefix of every frame (written by k_enc_scan)
    uint32_t* ticket;          // zeroed work counter of this batch (frames are taken in any order)
    int* err;
    int hdr_bytes;
    uint8_t* slots;            // batch scratch: frame (g - g_begin) is written at slots + (g - g_begin) * slot_bytes
    int64_t slot_bytes;        // worst-case frame size rounded up to 16
    uint32_t* fsize;           // [g - g_begin] bytes of the frame (body + CRC-16)
    unsigned long long* base;  // running total of bytes before this batch (device scalar)
    FrameStats* stats;         // [(g - g_begin) * nch + c]
    FramePlan* plans;
    PlanHeader* hdrs;          // [(g - g_begin) * nch + c] subframe preambles built by k_enc_design
    uint32_t g_begin, g_end;   // (stream, frame) units covered by this batch of launches
};

// Levels 0..2 (blocksize 1152): fa_encode_fixed.h encodes full frames one warp each and publishes their size in fsize
// (zeroed before); the kernels of this file skip those frames and take what that path declined.
constexpr int kFxBs = 1152;
FA_D bool fixed_done(const EncParams& P, uint32_t g) { return P.blocksize == kFxBs && P.fsize[g - P.g_begin] != 0u; }

// Records exchanged between the three encoder kernels, one per (frame, channel):
//   k_enc_analyze -> FrameStats -> k_enc_design -> FramePlan -> k_encode
struct FrameStats {
    int32_t mode;              // 0 general path, 1 CONSTANT, 2 predictive (narrow samples), 3 predictive (wide samples)
    int32_t wasted;
    int32_t mn, mx;            // of the samples >> wasted
    uint32_t bad, pad;         // wide: fixed-predictor orders whose residual leaves the int32 range
    unsigned long long fe[5];  // fixed-predictor error sums of the samples >> wasted
    double ac[kMaxOrd + 1];    // windowed autocorrelation of the samples >> wasted
};
struct FramePlan {             // 48 bytes, read with three 16-byte broadcast loads
    uint8_t mode, wasted, ok0, ok1, ord0, ord1, shift1, prec1, wide1, maxp0, maxp1, pad[5];
    int16_t qlp[kMaxOrd];
    uint32_t fixed_bits;       // estimated size of the FIXED subframe with one Rice partition (full frames: see enc_channel_full)
    uint32_t pad2;
};

// Everything of a full frame's subframe that is known before its residual is computed, as a ready-made MSB-first bit
// string per candidate: [frame header (channel 0 only)] subframe header byte, warm-up samples, and for LPC the
// precision, shift and coefficients.  Built by the design thread (which runs serial code anyway), so that no
// thread of k_encode has to emit ~50 fields one after the other while its 127 neighbours wait.  nbits == 0:
// not built (wasted bits, no such candidate): k_encode's thread 0 then emits the header itself.
struct PlanHeader {            // 128 bytes
    uint32_t nbits_lpc, nbits_fix;
    uint32_t lpc[22];          // <= 88 + 8 + 12 * 32 + 9 + 12 * 15 = 669 bits
    uint32_t fix[8];           // <= 88 + 8 + 4 * 32 = 224 bits
};

struct Plan {
    int type;      // 0 constant, 1 verbatim, 2 fixed, 3 lpc
    int order, wasted, shift, prec, porder, rice2;
    int wide;      // lpc: residual needs 64-bit accumulation
    uint32_t res_bits;  // estimated bits of the residual section
    int32_t qlp[kMaxOrd];
};

constexpr int kStagePitch = kEncThreads + 1;
struct AnShared {              // k_enc_analyze: per-warp partials of the block reductions
    uint32_t w_or[kEncWarps];
    int32_t w_mn[kEncWarps], w_mx[kEncWarps];
    uint32_t w_bad[kEncWarps];
    unsigned long long w_fe[kEncWarps][5];
    double w_ac[kEncWarps][kMaxOrd + 1];
    int32_t stage[8 * kStagePitch * 4];  // full frames: the channel's int32 samples, [quad][thread][4], quad rows kStagePitch
                                         // 16-byte units apart (odd: a warp may store eight quads of one thread at once); afterwards every
                                         // warp's own quads hold its per-lane autocorrelation partials
    float wqt[kEncThreads * kSpt];       // the window in the same [quad][thread][4] order (filled once per CTA)
};

struct DesignIO {              // k_enc_design: thread-private working set of design_fixed / design_lpc
    unsigned long long t_fe[5];
    double t_ac[kMaxOrd + 1];
    Plan cand[2];
    int cand_ok[2];
    int maxp[2];
    double lpc_hist[kMaxOrd][kMaxOrd];
};

// Working set of the short-frame and general paths.  It lives in the 16 KB sample buffer of the full-frame
// path (`EncCtx::res`), which those paths never use: the hot path's shared memory stays small enough for six
// resident CTAs per SM.
struct EncShared {
    // per-warp partials of the block reductions
    uint32_t w_or[kEncWarps];
    int32_t w_mn[kEncWarps], w_mx[kEncWarps];
    uint32_t w_bad[kEncWarps];
    unsigned long long w_fe[kEncWarps][5];
    double w_ac[kEncWarps][kMaxOrd + 1];
    // totals
    uint32_t t_or;
    int32_t t_mn, t_mx;
    unsigned long long t_fe[5];
    double t_ac[kMaxOrd + 1];
    // design
    Plan cand[2];  // [0] fixed, [1] lpc
    int cand_ok[2];
    int maxp[2];
    int mode;      // fast path: 0 = rejected, 1 = constant, 2 = predictive
    int wasted;
    double lpc_hist[kMaxOrd][kMaxOrd];
    unsigned long long csum[2][kEncThreads];   // per-thread-chunk sum |residual|
    unsigned long long psum[2][kMaxParts];
    uint8_t kpar[2][2 * kMaxParts];            // params for porder p at offset (1 << p) - 1
    uint32_t scan[kEncWarps];
};

// State that lives across frames and paths (never aliased).
struct EncHot {
    unsigned long long mbar;                   // completion barrier of the TMA copy into the sample buffer
    uint32_t scan[kEncWarps];
    uint8_t crc8[256];                         // CRC-8 table (frame headers)
    uint32_t hdr_tmp[40];                      // full-frame path: header words built by thread 0 ahead of the packing (ow-indexed)
    alignas(16) int32_t warm[kMaxOrd];         // full-frame path: the channel's first samples (>> wasted), saved before the in-place pass
    // full-frame path: per-warp partials of (estimated bits at the finest partition order, sum |residual|, flags)
    // (two sets: the second residual pass of a channel must not overwrite what slower warps still read)
    uint32_t x_bits[2][kEncWarps];
    unsigned long long x_sum[2][kEncWarps];
    uint32_t x_flag[2][kEncWarps];             // bit 0: a residual does not fit, bit 1: some parameter >= 15
    // deferred tail words of the packing sessions (OR-ed in when the frame is retired)
    uint32_t tail_val[2][kEncThreads];
    uint16_t tail_word[2][kEncThreads];
    // the frame that is packed in `out` and waits to be retired (copy to its slot)
    int prev_nbytes;
    uint32_t prev_g;
    uint32_t gq[2];     // tickets, fetched one frame ahead (the atomic's latency is off the critical path)
    int gq_f[2], gq_bs[2];   // ... with their frame number and blocksize (thread 0 does the divisions, also ahead)
    // ... and with the frame's plans and the first 16 bytes of its prebuilt headers (both channels), copied in by
    // thread 0 with cp.async one frame ahead: the ticket -> plan -> header chain of dependent global loads (three L2
    // round trips in a row at the start of every frame) is off the critical path
    alignas(16) U4 pf_plan[2][2][3];
    alignas(16) U4 pf_hdr[2][2];
    int prev_valid2[2];  // (frame pending in `out`, by iteration parity)
};

FA_HD size_t enc_out_words(int nch) { return ((size_t)nch * (kMaxBs * 4 + 64) + 64) / 4; }
FA_D int ow(int w) { return w + (w >> 4); }   // padded word index: per-thread strides of ~16 words stay off one bank
constexpr size_t kEncHotBytes = (sizeof(EncHot) + 127) & ~(size_t)127;
static_assert(sizeof(EncShared) <= (size_t)kMaxBs * 4, "the cold working set must fit the sample buffer");
inline size_t enc_smem_bytes(int nch) {
    size_t words = enc_out_words(nch);
    // EncHot | sample / residual buffer of one full frame-channel (128-byte aligned: TMA destination) | staged frame (padded)
    return kEncHotBytes + (size_t)kMaxBs * 4 + (words + (words >> 4) + 8) * 4 + 16;
}

// ---- small helpers -----------------------------------------------------------------------------------
FA_D double shfl_xor_d(double v, int m) {
    unsigned long long u;
    memcpy(&u, &v, 8);
    uint32_t lo = shfl_xor((uint32_t)u, m), hi = shfl_xor((uint32_t)(u >> 32), m);
    u = ((unsigned long long)hi << 32) | lo;
    memcpy(&v, &u, 8);
    return v;
}
FA_D double shfl_down_d(double v, int d) {
    unsigned long long u;
    memcpy(&u, &v, 8);
    uint32_t lo = shfl_down((uint32_t)u, d), hi = shfl_down((uint32_t)(u >> 32), d);
    u = ((unsigned long long)hi << 32) | lo;
    memcpy(&v, &u, 8);
    return v;
}
FA_D unsigned long long warp_sum_u64(unsigned long long v) {
    for (int m = 16; m >= 1; m >>= 1) v += shfl_xor64(v, m);
    return v;
}
// exact warp sum of 32-bit partials as a 64-bit value: two REDUX over the 16-bit halves
FA_D unsigned long long warp_sum_u32_wide(uint32_t v) {
    uint32_t lo = redux_add(v & 0xFFFFu), hi = redux_add(v >> 16);
    return ((unsigned long long)hi << 16) + lo;
}
FA_D double warp_sum_d(double v) {
    for (int m = 16; m >= 1; m >>= 1) v = dadd(v, shfl_xor_d(v, m));
    return v;
}
// Sum 8 doubles across the warp with 18 shuffles: every step halves the values a lane carries.
// Afterwards lane l holds the total of value index ((l >> 4) & 1) * 4 + ((l >> 3) & 1) * 2 + ((l >> 2) & 1).
FA_D double warp_sum8_d(const double* v) {
    const int ln = lane();
    double a[4], b[2], c;
    const bool u16 = (ln & 16) != 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        double keep = u16 ? v[4 + i] : v[i], send = u16 ? v[i] : v[4 + i];
        a[i] = dadd(keep, shfl_xor_d(send, 16));
    }
    const bool u8 = (ln & 8) != 0;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        double keep = u8 ? a[2 + i] : a[i], send = u8 ? a[i] : a[2 + i];
        b[i] = dadd(keep, shfl_xor_d(send, 8));
    }
    const bool u4 = (ln & 4) != 0;
    {
        double keep = u4 ? b[1] : b[0], send = u4 ? b[0] : b[1];
        c = dadd(keep, shfl_xor_d(send, 4));
    }
    c = dadd(c, shfl_xor_d(c, 2));
    c = dadd(c, shfl_xor_d(c, 1));
    return c;
}

FA_D uint32_t gf16_mul(uint32_t a, uint32_t b) {  // a * b mod x^16 + x^15 + x^2 + 1
    uint32_t r = 0;
#pragma unroll
    for (int i = 15; i >= 0; --i) {
        r <<= 1;
        r ^= (r & 0x10000u) ? 0x18005u : 0u;
        r ^= ((b >> i) & 1u) ? a : 0u;
    }
    return r & 0xFFFFu;
}

// Word index of in-frame sample i inside the parked [8][128][4] block of a full frame-channel.
FA_HD int park_word(int i) { return ((((i >> 2) & 7) * kEncThreads + (i >> 5)) << 2) + (i & 3); }

FA_D bool fits_res(int64_t v) { return v >= -2147483647LL && v <= 2147483647LL; }

FA_D int max_porder_for(int bs, int order, int level_max) {
    int p = 0;
    while (p < level_max && !((bs >> p) & 1)) p++;   // largest p with 2^p | bs, capped
    while (p > 0 && (bs >> p) <= order) p--;
    return p;
}

// Rice parameter and estimated bits of one partition (libFLAC set_partitioned_rice_, estimate mode)
FA_D uint32_t rice_estimate(unsigned long long sum, uint32_t n, int& k_out) {
    int k = 0;
    if (sum > n) {
        k = (64 - clz64(sum - 1)) - (32 - clz32(n));
        if (k < 0) k = 0;
        if (k < 30 && ((unsigned long long)n << k) < sum) k++;
        if (k < 30 && ((unsigned long long)n << k) < sum) k++;
        if (k > 30) k = 30;
    }
    k_out = k;
    unsigned long long pb = 4ull + (unsigned long long)(1 + k) * n + (k ? (sum >> (k - 1)) : (sum << 1));
    pb -= (n >> 1);
    return pb > (1ull << 25) ? (1u << 25) : (uint32_t)pb;
}

FA_D int utf8_put(uint8_t* p, uint64_t v) {
    if (v < 0x80) { p[0] = (uint8_t)v; return 1; }
    int n = v < 0x800 ? 2 : v < 0x10000 ? 3 : v < 0x200000 ? 4 : v < 0x4000000 ? 5 : v < 0x80000000ull ? 6 : 7;
    const uint8_t lead[8] = {0, 0, 0xC0, 0xE0, 0xF0, 0xF8, 0xFC, 0xFE};
    for (int i = n - 1; i > 0; --i) { p[i] = (uint8_t)(0x80 | (v & 0x3F)); v >>= 6; }
    p[0] = (uint8_t)(lead[n] | v);
    return n;
}
FA_D int utf8_len(uint64_t v) {
    return v < 0x80 ? 1 : v < 0x800 ? 2 : v < 0x10000 ? 3 : v < 0x200000 ? 4 : v < 0x4000000 ? 5 : v < 0x80000000ull ? 6 : 7;
}

FA_D int blocksize_code(int bs) {
    if (bs == 192) return 1;
    if (bs == 576) return 2;
    if (bs == 1152) return 3;
    if (bs == 2304) return 4;
    if (bs == 4608) return 5;
    for (int c = 8; c <= 15; ++c) if (bs == (256 << (c - 8))) return c;
    return bs <= 256 ? 6 : 7;
}
FA_D int frame_header_bytes(int bs, int f) {
    int bc = blocksize_code(bs);
    return 4 + utf8_len((uint64_t)f) + (bc == 6 ? 1 : bc == 7 ? 2 : 0) + 1;
}

// ---- bit packer: 64-bit accumulator -> staged frame words ----------------------------------------------
// Write protocol of the staged frame: while packing, a thread plain-stores every word it completes --
// including its first one, whose leading bits may belong to the previous thread and are stored as
// zeros.  The trailing partial word of a session is NOT stored: it is recorded and OR-ed in after a
// barrier, when the frame is retired.  The sessions tile the frame, so every word except the frame's
// final partial word has exactly one plain-storing thread (the one whose session contains its last
// bit), and all ORs come after all plain stores: no atomics, no "first word" test and no pre-zeroed
// buffer are needed.  The final partial word is cleared by thread 0 once the frame size is known.
struct Pk {
    uint32_t* out;
    uint64_t acc;
    int fill;            // bits pending in acc (MSB side), < 32 between calls
    int word;            // next word to write
};
FA_D void pk_begin(Pk& pk, uint32_t* out, int bitpos) {
    pk.out = out; pk.acc = 0; pk.fill = bitpos & 31; pk.word = bitpos >> 5;
}
FA_D void pk_flush(Pk& pk) {
    pk.out[ow(pk.word)] = (uint32_t)(pk.acc >> 32);
    pk.word++;
    pk.acc <<= 32;
    pk.fill -= 32;
}
// nb in [1, 32], v < 2^nb
FA_D void pk_emit(Pk& pk, uint32_t v, int nb) {
    pk.acc |= (uint64_t)v << (64 - pk.fill - nb);
    pk.fill += nb;
    if (pk.fill >= 32) pk_flush(pk);
}
FA_D void pk_zeros(Pk& pk, uint32_t q) {
    while (q >= 32) { pk_emit(pk, 0u, 32); q -= 32; }
    if (q) pk_emit(pk, 0u, (int)q);
}
FA_D void pk_rice(Pk& pk, uint32_t u, int k) {
    uint32_t q = u >> k;
    uint32_t low = (u & ((1u << k) - 1u)) | (1u << k);
    uint32_t len = q + (uint32_t)k + 1u;
    if (len <= 32u) {
        pk_emit(pk, low, (int)len);
    } else {
        pk_zeros(pk, q);
        pk_emit(pk, low, k + 1);
    }
}
// record the trailing partial word (value 0 when the session ended on a word boundary)
FA_D void pk_end(const Pk& pk, uint32_t& tail_val, uint16_t& tail_word) {
    tail_val = (uint32_t)(pk.acc >> 32);
    tail_word = (uint16_t)pk.word;
}

// ---- byte-prefix words: [61:0] bytes (the two top bits were the status of the first version's look-back)
constexpr unsigned long long kDescAgg = 1ull << 62, kDescPre = 2ull << 62, kDescMask = (1ull << 62) - 1;

// Frame placement.  Every frame of a batch is first written to its own 16-byte aligned worst-case slot, so
// the encoder CTAs are completely independent (no ticket order, no look-back, no waiting for stragglers:
// with the decoupled look-back of the first version a single late CTA stalled the retire of every
// successor, and the stall grew with the number of resident CTAs).  k_enc_scan then turns the frame
// sizes into byte offsets and k_enc_compact moves the frames to their final place: the compressed
// bytes cross HBM three times instead of once, which costs ~1 ms at cfg2 and is far cheaper than the
// serialisation it removes.

// ---- sample source ------------------------------------------------------------------------------------
struct FrameSrc {
    const void* base;   // element (stream s, frame sample 0)
    int dtype, bs;
    bool vec;           // 16-byte vector loads are aligned
    float off32, gain32;
    double off64, gain64;
};

// channel c of in-frame sample i (general path; 0 <= i < bs)
FA_D int32_t src_sample(const FrameSrc& S, int c, int i) {
    if (S.dtype == kI32) return ((const int32_t*)S.base)[i];
    if (S.dtype == kF32) return quant_f32(((const float*)S.base)[i], S.off32, S.gain32);
    long long v;
    if (S.dtype == kI64) v = ((const long long*)S.base)[i];
    else v = quant_f64(((const double*)S.base)[i], S.off64, S.gain64);
    return c == 0 ? (int32_t)(uint32_t)((unsigned long long)v & 0xFFFFFFFFull) : (int32_t)(v >> 32);
}

// Fast path: xw[H + j] = sample (32 t + j), xw[0..H) = the H samples before them (zeros for thread 0).
// FULL: the frame has 4096 samples; otherwise samples at or beyond S.bs read as zero.
template <int H, bool FULL>
FA_D void load_chunk(const FrameSrc& S, int c, int t, int32_t* xw) {
    const int i0 = t * kSpt - H;
    const int bs = S.bs;
    if (S.dtype == kI32 || S.dtype == kF32) {
        const uint32_t* p = (const uint32_t*)S.base + i0;
#pragma unroll
        for (int q = 0; q < (H + kSpt) / 4; ++q) {
            U4 v;
            v.x = v.y = v.z = v.w = 0;
            const bool hist = q * 4 < H;
            const int i = i0 + 4 * q;
            if (!(hist && t == 0) && (FULL || i < bs)) {
                if (S.vec && (FULL || i + 4 <= bs)) v = ldg128(p + 4 * q);
                else {
                    v.x = ldg32(p + 4 * q);
                    if (FULL || i + 1 < bs) v.y = ldg32(p + 4 * q + 1);
                    if (FULL || i + 2 < bs) v.z = ldg32(p + 4 * q + 2);
                    if (FULL || i + 3 < bs) v.w = ldg32(p + 4 * q + 3);
                }
                if (S.dtype == kF32) {
                    float f0, f1, f2, f3;
                    memcpy(&f0, &v.x, 4); memcpy(&f1, &v.y, 4); memcpy(&f2, &v.z, 4); memcpy(&f3, &v.w, 4);
                    v.x = (uint32_t)quant_f32(f0, S.off32, S.gain32);
                    v.y = (FULL || i + 1 < bs) ? (uint32_t)quant_f32(f1, S.off32, S.gain32) : 0u;
                    v.z = (FULL || i + 2 < bs) ? (uint32_t)quant_f32(f2, S.off32, S.gain32) : 0u;
                    v.w = (FULL || i + 3 < bs) ? (uint32_t)quant_f32(f3, S.off32, S.gain32) : 0u;
                }
            }
            xw[4 * q] = (int32_t)v.x; xw[4 * q + 1] = (int32_t)v.y; xw[4 * q + 2] = (int32_t)v.z; xw[4 * q + 3] = (int32_t)v.w;
        }
    } else {
        const unsigned long long* p = (const unsigned long long*)S.base + i0;
#pragma unroll
        for (int q = 0; q < (H + kSpt) / 2; ++q) {
            unsigned long long e0 = 0, e1 = 0;
            const bool hist = q * 2 < H;
            const int i = i0 + 2 * q;
            const bool v1 = FULL || i + 1 < bs;
            if (!(hist && t == 0) && (FULL || i < bs)) {
                if (S.vec && v1) {
                    U4 v = ldg128(p + 2 * q);
                    e0 = ((unsigned long long)v.y << 32) | v.x;
                    e1 = ((unsigned long long)v.w << 32) | v.z;
                } else {
                    e0 = p[2 * q];
                    if (v1) e1 = p[2 * q + 1];
                }
                if (S.dtype == kF64) {
                    double d0, d1;
                    memcpy(&d0, &e0, 8); memcpy(&d1, &e1, 8);
                    e0 = (unsigned long long)quant_f64(d0, S.off64, S.gain64);
                    e1 = v1 ? (unsigned long long)quant_f64(d1, S.off64, S.gain64) : 0ull;
                }
            }
            xw[2 * q] = c == 0 ? (int32_t)(uint32_t)e0 : (int32_t)(uint32_t)(e0 >> 32);
            xw[2 * q + 1] = c == 0 ? (int32_t)(uint32_t)e1 : (int32_t)(uint32_t)(e1 >> 32);
        }
    }
}

// ---- frame / subframe headers (thread 0, through its packing session) ----------------------------------
FA_D int build_frame_header(uint8_t* h, const uint8_t* crc8, int bs, int f, int nch) {   // h[16]; returns the byte count
    int n = 0;
    int bc = blocksize_code(bs);
    h[n++] = 0xFF; h[n++] = 0xF8;
    h[n++] = (uint8_t)((bc << 4) | 9);                       // 44.1 kHz like the reference's default
    h[n++] = (uint8_t)(((nch == 2 ? 1 : 0) << 4) | (7 << 1));  // independent channels, 32 bps
    n += utf8_put(h + n, (uint64_t)f);
    if (bc == 6) h[n++] = (uint8_t)(bs - 1);
    else if (bc == 7) { h[n++] = (uint8_t)((bs - 1) >> 8); h[n++] = (uint8_t)(bs - 1); }
    uint32_t c = 0;
    for (int i = 0; i < n; ++i) c = crc8[c ^ h[i]];
    h[n++] = (uint8_t)c;
    return n;
}
FA_D void emit_frame_header(Pk& pk, const uint8_t* crc8, int bs, int f, int nch) {
    uint8_t h[16];
    const int n = build_frame_header(h, crc8, bs, f, nch);
    for (int i = 0; i < n; ++i) pk_emit(pk, h[i], 8);
}
// append nb (1..32) bits of v (< 2^nb) to a zero-initialised MSB-first bit string of *n bits
FA_D void hdr_put(uint32_t* w, uint32_t& n, uint32_t v, int nb) {
    const int word = (int)(n >> 5), off = (int)(n & 31);
    const uint64_t x = (uint64_t)v << (64 - off - nb);
    w[word] |= (uint32_t)(x >> 32);
    if (off + nb > 32) w[word + 1] |= (uint32_t)x;
    n += (uint32_t)nb;
}

// subframe header byte (+ wasted-bits unary), warm-up samples are emitted by the caller
FA_D void emit_subframe_header(Pk& pk, int ptype, int order, int wasted) {
    int typebits = ptype == 0 ? 0 : ptype == 1 ? 1 : ptype == 2 ? (8 + order) : (32 + order - 1);
    pk_emit(pk, ((uint32_t)typebits << 1) | (wasted ? 1u : 0u), 8);
    if (wasted) { pk_zeros(pk, (uint32_t)(wasted - 1)); pk_emit(pk, 1u, 1); }
}
FA_D void emit_sample(Pk& pk, int32_t v, int bps) {  // bps in [1, 32]
    pk_emit(pk, bps == 32 ? (uint32_t)v : ((uint32_t)v & ((1u << bps) - 1u)), bps);
}
FA_D void emit_lpc_params(Pk& pk, const Plan& pl) {
    pk_emit(pk, (uint32_t)(pl.prec - 1), 4);
    pk_emit(pk, (uint32_t)pl.shift & 31u, 5);
    for (int j = 0; j < pl.order; ++j) pk_emit(pk, (uint32_t)pl.qlp[j] & ((1u << pl.prec) - 1u), pl.prec);
}
FA_D int subframe_header_bits(int ptype, int order, int wasted, int bps, int prec) {
    int b = 8 + wasted;
    if (ptype == 0) return b + bps;
    if (ptype == 1) return b;
    return b + order * bps + 6 + (ptype == 3 ? 9 + order * prec : 0);
}

// ---- Rice partition search: one warp per candidate ------------------------------------------------------
// libFLAC's estimate-based partition-order / Rice-parameter search (find_best_partition_order_ /
// set_partitioned_rice_ without escape codes) over the finest-level sums in sh->psum[cand].
FA_D void rice_search_warp(EncShared* sh, int cand, int bs, int order, int maxp) {
    unsigned long long* ps = sh->psum[cand];
    uint32_t best_bits = 0xFFFFFFFFu;
    int best_p = maxp, best_r2 = 0;
    for (int p = maxp; p >= 0; --p) {
        int nparts = 1 << p;
        uint32_t bits = 0;
        bool big = false;
        for (int part = lane(); part < nparts; part += 32) {
            unsigned long long sum = ps[part];
            uint32_t n = (uint32_t)(bs >> p) - (part == 0 ? (uint32_t)order : 0u);
            int k = 0;
            if (sum > n) {
                k = (64 - clz64(sum - 1)) - (32 - clz32(n));
                if (k < 0) k = 0;
                while (k < 30 && ((unsigned long long)n << k) < sum) k++;
                if (k > 30) k = 30;
            }
            sh->kpar[cand][(1 << p) - 1 + part] = (uint8_t)k;
            big = big || k >= 15;
            unsigned long long pb = 4ull + (unsigned long long)(1 + k) * n + (k ? (sum >> (k - 1)) : (sum << 1));
            pb -= (n >> 1);
            bits += pb > (1ull << 25) ? (1u << 25) : (uint32_t)pb;
        }
        bits = redux_add(bits) + 6;
        int r2 = ballot(big) != 0 ? 1 : 0;
        if (r2) bits += (uint32_t)nparts;   // 5-bit parameters
        if (bits < best_bits) { best_bits = bits; best_p = p; best_r2 = r2; }
        // merge to the next coarser level
        if (p > 0) {
            unsigned long long a[2] = {0, 0};
            int half = nparts >> 1;
            int cnt = 0;
            for (int j = lane(); j < half; j += 32) a[cnt++] = ps[2 * j] + ps[2 * j + 1];
            syncwarp();
            cnt = 0;
            for (int j = lane(); j < half; j += 32) ps[j] = a[cnt++];
            syncwarp();
        }
    }
    if (lane() == 0) {
        sh->cand[cand].porder = best_p;
        sh->cand[cand].res_bits = best_bits;
        sh->cand[cand].rice2 = best_r2;
    }
    syncwarp();
}

// ---- design (one thread): fixed order choice, Levinson-Durbin, order choice, coefficient quantisation --
// libFLAC fixed.c / lpc.c procedure.  `narrow_maxabs` > 0 selects the fast path's rule for the
// coefficient precision: the largest precision <= `precision` for which every prediction sum and
// residual provably fits 32-bit arithmetic; if that would cost more than 3 bits the plan is marked
// `wide` (64-bit residual) at full precision instead.
template <class D>
FA_D void design_fixed(D* sh, int bs, int bps, uint32_t bad, int level_maxp) {
    unsigned long long te[5];
    for (int k = 0; k < 5; ++k) te[k] = ((bad >> k) & 1) ? ~0ull : sh->t_fe[k];
    unsigned long long m34 = te[3] < te[4] ? te[3] : te[4];
    unsigned long long m234 = te[2] < m34 ? te[2] : m34;
    unsigned long long m1234 = te[1] < m234 ? te[1] : m234;
    int order;
    if (te[0] < m1234) order = 0;
    else if (te[1] < m234) order = 1;
    else if (te[2] < m34) order = 2;
    else if (te[3] < te[4]) order = 3;
    else order = 4;
    Plan& pl = sh->cand[0];
    pl.type = 2; pl.order = order; pl.shift = 0; pl.prec = 0; pl.wide = 0;
    bool ok = te[order] != ~0ull;
    if (ok && te[order] > 0) {
        float rb = flog2(0.6931472f * (float)te[order] / (float)(bs - 4));
        ok = rb < (float)bps;
    }
    sh->cand_ok[0] = ok ? 1 : 0;
    sh->maxp[0] = max_porder_for(bs, order, level_maxp);
}

FA_D bool quantize_coefs(const double* coefs, int order, int precision, int32_t* q, int& shift_out) {
    int prec = precision - 1;
    int32_t qmax = (1 << prec) - 1, qmin = -(1 << prec);
    double cmax = 0.0;
    for (int i = 0; i < order; ++i) { double d = fabs(coefs[i]); if (d > cmax) cmax = d; }
    if (!(cmax > 0.0)) return false;
    int log2cmax;
    (void)frexp(cmax, &log2cmax);
    log2cmax--;
    int shift = prec - log2cmax - 1;
    if (shift > 15) shift = 15;
    if (shift < 0) return false;
    double e = 0.0;
    for (int i = 0; i < order; ++i) {
        e += coefs[i] * (double)(1 << shift);
        double rq = e < 0.0 ? -floor(-e + 0.5) : floor(e + 0.5);  // lround: half away from zero
        long long v = (long long)rq;
        if (v > qmax) v = qmax; else if (v < qmin) v = qmin;
        e -= (double)v;
        q[i] = (int32_t)v;
    }
    shift_out = shift;
    return true;
}

template <class D>
FA_D void design_lpc(D* sh, int bs, int bps, int max_order, int precision, int level_maxp, uint32_t narrow_maxabs) {
    Plan& pl = sh->cand[1];
    sh->cand_ok[1] = 0;
    const double* autoc = sh->t_ac;
    if (max_order <= 0 || !(autoc[0] != 0.0)) return;
    double lpc[kMaxOrd], error[kMaxOrd];
    double err = autoc[0];
    int mo = max_order;
    for (int i = 0; i < mo; ++i) {
        double r = -autoc[i + 1];
        for (int j = 0; j < i; ++j) r -= lpc[j] * autoc[i - j];
        r /= err;
        lpc[i] = r;
        int j;
        for (j = 0; j < (i >> 1); ++j) {
            double tmp = lpc[j];
            lpc[j] += r * lpc[i - 1 - j];
            lpc[i - 1 - j] += r * tmp;
        }
        if (i & 1) lpc[j] += lpc[j] * r;
        err *= (1.0 - r * r);
        for (j = 0; j <= i; ++j) sh->lpc_hist[i][j] = (double)(float)(-lpc[j]);
        error[i] = err;
        if (err == 0.0) { mo = i + 1; break; }
    }
    // FLAC__lpc_compute_best_order (log2 in single precision: only the order choice depends on it)
    float escale = 0.5f / (float)bs;
    float best_bits = 3.0e38f;
    int order = 1;
    for (int idx = 0; idx < mo; ++idx) {
        double e = error[idx];
        float b;
        if (e > 0.0) { b = 0.5f * flog2(escale * (float)e); if (b < 0.0f) b = 0.0f; }
        else if (e < 0.0) b = 1e32f;
        else b = 0.0f;
        float bits = b * (float)(bs - (idx + 1)) + (float)((idx + 1) * (bps + precision));
        if (bits < best_bits) { best_bits = bits; order = idx + 1; }
    }
    {
        double e = error[order - 1];
        float b;
        float es = 0.5f / (float)(bs - order);
        if (e > 0.0) { b = 0.5f * flog2(es * (float)e); if (b < 0.0f) b = 0.0f; }
        else if (e < 0.0) b = 1e32f;
        else b = 0.0f;
        if (!(b < (float)bps)) return;
    }
    const double* coefs = sh->lpc_hist[order - 1];
    int shift = 0;
    int prec = precision;
    bool have = false;
    pl.wide = 1;
    if (narrow_maxabs) {
        // 32-bit datapath conditions: |sum q x| <= sumq * maxabs < 2^30 and |x - pred| < 2^26.
        // sumq ~ sumc * 2^shift with shift = p - 2 - floor(log2 cmax): solve for the largest p, verify.
        double sumc = 0.0, cmax = 0.0;
        for (int i = 0; i < order; ++i) { double d = fabs(coefs[i]); sumc += d; if (d > cmax) cmax = d; }
        if (cmax > 0.0) {
            int e, lc;
            (void)frexp(sumc * (double)narrow_maxabs, &e);   // sumc * maxabs < 2^e
            (void)frexp(cmax, &lc);                          // floor(log2 cmax) = lc - 1
            int p = 32 - e + (lc - 1);
            if (p > precision) p = precision;
            for (int tries = 0; tries < 2 && p >= 5 && p >= precision - 6; ++tries, --p) {
                int32_t q[kMaxOrd];
                int sft;
                if (!quantize_coefs(coefs, order, p, q, sft)) break;
                unsigned long long sumq = 0;
                for (int i = 0; i < order; ++i) sumq += (unsigned long long)(q[i] < 0 ? -q[i] : q[i]);
                unsigned long long mac = sumq * narrow_maxabs;
                // lowering the precision must stay invisible next to the residual itself: coefficient
                // rounding error ~ 2^-(shift+1) per tap against the predicted residual RMS
                double qerr = (double)narrow_maxabs * sqrt((double)order) / (double)(2u << sft);
                double sigma = sqrt(error[order - 1] / (double)bs);
                bool harmless = p == precision || qerr < 0.25 * sigma;
                if (harmless && mac < (1ull << 30) && (unsigned long long)narrow_maxabs + (mac >> sft) < (1ull << 26)) {
                    for (int i = 0; i < order; ++i) pl.qlp[i] = q[i];
                    shift = sft;
                    prec = p;
                    pl.wide = 0;
                    have = true;
                    break;
                }
            }
        }
    }
    if (!have && !quantize_coefs(coefs, order, prec, pl.qlp, shift)) return;
    for (int i = order; i < kMaxOrd; ++i) pl.qlp[i] = 0;
    pl.type = 3;
    pl.order = order;
    pl.shift = shift;
    pl.prec = prec;
    sh->cand_ok[1] = 1;
    sh->maxp[1] = max_porder_for(bs, order, level_maxp);
}

// ---- residuals of the thread's 32 samples for a compile-time predictor order ---------------------------
// xw[H + j] = sample j of the chunk.  r[j] = x[j] - ((sum_m coef[m] * x[j - 1 - m]) >> shift).
template <int H, int ORD>
FA_D void residual32(const int32_t* xw, const int32_t* coef, int shift, int32_t* r) {
#pragma unroll
    for (int j = 0; j < kSpt; ++j) {
        int32_t sum = 0;
#pragma unroll
        for (int m = 0; m < ORD; ++m) sum += coef[m] * xw[H + j - 1 - m];
        r[j] = xw[H + j] - (sum >> shift);
    }
}
template <int H>
FA_D void residual32_dispatch(int order, const int32_t* xw, const int32_t* coef, int shift, int32_t* r) {
    switch (order) {
    case 0: residual32<H, 0>(xw, coef, shift, r); break;
    case 1: residual32<H, 1>(xw, coef, shift, r); break;
    case 2: residual32<H, 2>(xw, coef, shift, r); break;
    case 3: residual32<H, 3>(xw, coef, shift, r); break;
    case 4: residual32<H, 4>(xw, coef, shift, r); break;
    case 5: residual32<H, 5>(xw, coef, shift, r); break;
    case 6: residual32<H, 6>(xw, coef, shift, r); break;
    case 7: residual32<H, 7>(xw, coef, shift, r); break;
    case 8: residual32<H, 8>(xw, coef, shift, r); break;
    default:
        if constexpr (H > 8) {
            switch (order) {
            case 9: residual32<H, 9>(xw, coef, shift, r); break;
            case 10: residual32<H, 10>(xw, coef, shift, r); break;
            case 11: residual32<H, 11>(xw, coef, shift, r); break;
            default: residual32<H, 12>(xw, coef, shift, r); break;
            }
        }
        break;
    }
}
// 64-bit accumulation (narrow samples, full-precision coefficients); bit j of the result is set when
// residual j fits the Rice coder
template <int H>
FA_D uint32_t residual64(int order, const int32_t* xw, const int32_t* coef, int shift, int32_t* r) {
    uint32_t ok = 0;
#pragma unroll
    for (int j = 0; j < kSpt; ++j) {
        int64_t sum = 0;
#pragma unroll
        for (int m = 0; m < H; ++m) sum += (int64_t)coef[m] * (int64_t)xw[H + j - 1 - m];   // coef[m] = 0 beyond `order`
        int64_t v = (int64_t)xw[H + j] - (sum >> shift);
        if (fits_res(v)) ok |= 1u << j;
        r[j] = (int32_t)v;
    }
    (void)order;
    return ok;
}

FA_D void fixed_coefs(int order, int32_t* c, int n) {
    // (1), (2, -1), (3, -3, 1), (4, -6, 4, -1): selected arithmetically, no table in local memory
    const int32_t c0 = order;
    const int32_t c1 = order == 2 ? -1 : order == 3 ? -3 : order == 4 ? -6 : 0;
    const int32_t c2 = order == 3 ? 1 : order == 4 ? 4 : 0;
    const int32_t c3 = order == 4 ? -1 : 0;
#pragma unroll
    for (int q = 0; q < n; ++q) c[q] = q == 0 ? c0 : q == 1 ? c1 : q == 2 ? c2 : q == 3 ? c3 : 0;
}


// ------------------------------------------------------------------------------------------------------
// Retiring a packed frame: copy to its slot in HBM.  The frame packed during iteration n of the CTA
// loop is retired during iteration n + 1 (before the staged buffer is needed again).  The frame's
// CRC-16 is computed and appended by k_enc_compact, which reads every byte of the frame anyway.
// ------------------------------------------------------------------------------------------------------
struct EncCtx {
    EncHot* hot;
    EncShared* sh;       // short-frame / general paths only: aliases `res`
    uint32_t* out;
    int32_t* res;        // full-frame path: [8][128][4] samples of the channel (TMA destination), zigzag residuals in place
    int out_words_padded;
    uint32_t tma_phase;  // parity of the next TMA completion (block-uniform)
#if defined(FAB_PHASE_TIMING) && defined(__CUDACC__)
    long long ph[12];
    long long last;
#endif
    bool retired;   // block-uniform: the previous frame has left `out`
};

// All threads, after the barrier at the top of the CTA loop (+ one more barrier behind the tail ORs): the
// coalesced copy of the staged frame to its slot.
// skip0: thread 0 takes no share of the work (it builds the next frame's header meanwhile)
FA_D void retire_copyout(const EncParams& P, const EncCtx& X, bool skip0 = false) {
    const EncHot* hot = X.hot;
    const int nthr = skip0 ? kEncThreads - 1 : kEncThreads;
    const int t = skip0 ? tid() - 1 : tid();
    const uint32_t* out = X.out;
    const int nbytes_body = hot->prev_nbytes;
    const uint32_t i = hot->prev_g - P.g_begin;
    if (t == 0) P.fsize[i] = (uint32_t)(nbytes_body + 2);
    // the slot is 16-byte aligned: four staged (big-endian) words per 16-byte store; the bytes past the
    // frame end inside the last store are don't-care (the slot is a worst-case frame rounded up to 16)
    uint8_t* dst = P.slots + (long long)i * P.slot_bytes;
    const int nvec = (nbytes_body + 15) >> 4;
    for (int v = t < 0 ? nvec : t; v < nvec; v += nthr) {
        const int w = 4 * v;          // four consecutive words never straddle a pad word (ow pads every 16)
        const int o = ow(w);
        U4 q;
        q.x = bswap32(out[o]); q.y = bswap32(out[o + 1]); q.z = bswap32(out[o + 2]); q.w = bswap32(out[o + 3]);
        sts128(dst + 16 * (size_t)v, q);
    }
}

// Generic (non-overlapped) retire sequence with its own barriers.
FA_D void retire_full(const EncParams& P, EncCtx& X) {
    if (X.retired) return;
    sync();
    retire_copyout(P, X);
    sync();
    X.retired = true;
}

// Inclusive byte prefix of every frame of the batch (one CTA of kScanThreads threads): desc[g] = bytes of
// everything up to and including frame g (stream headers included, at the first frame of each stream).
// Every warp scans one contiguous segment with coalesced 32-wide steps, the 32 segment totals are
// scanned by one thread, and a second coalesced pass adds the segment bases.
constexpr int kScanThreads = 1024;
FA_D void scan_batch_cta(const EncParams& P, unsigned long long* sh_part /*[kScanThreads / 32 + 1]*/) {
    const int t = tid(), ln = lane(), wp = warp();
    const uint32_t n = P.g_end - P.g_begin;
    constexpr uint32_t kW = kScanThreads / 32;
    const uint32_t seg = (((n + kW - 1) / kW) + 31u) & ~31u;      // elements per warp, a multiple of 32
    const uint32_t lo = (uint32_t)wp * seg;
    unsigned long long run = 0;
    constexpr int kRows = 8;      // rows of 32 sizes loaded together: the scan itself is short, the trips to HBM are not
    for (uint32_t i0 = lo; i0 < lo + seg && i0 < n; i0 += 32 * kRows) {
        uint32_t v[kRows];
#pragma unroll
        for (int r = 0; r < kRows; ++r) {
            const uint32_t j = i0 + 32u * r + (uint32_t)ln;
            v[r] = 0;
            if (i0 + 32u * r < lo + seg && j < n)
                v[r] = P.fsize[j] + (((P.g_begin + j) % (uint32_t)P.nframes) == 0 ? (uint32_t)P.hdr_bytes : 0u);
        }
#pragma unroll
        for (int r = 0; r < kRows; ++r) {
            const uint32_t j = i0 + 32u * r + (uint32_t)ln;
            uint32_t inc = v[r];
            for (int d = 1; d < 32; d <<= 1) {
                uint32_t o = shfl_up(inc, d);
                if (ln >= d) inc += o;
            }
            if (i0 + 32u * r < lo + seg && j < n) P.desc[P.g_begin + j] = run + inc;
            run += shfl(inc, 31);
        }
    }
    if (ln == 0) sh_part[wp] = run;
    sync();
    if (t == 0) {
        unsigned long long acc = *P.base;
        for (uint32_t w = 0; w < kW; ++w) { unsigned long long v = sh_part[w]; sh_part[w] = acc; acc += v; }
        sh_part[kW] = acc;
    }
    sync();
    const unsigned long long base = sh_part[wp];
    for (uint32_t i0 = lo; i0 < lo + seg && i0 < n; i0 += 32 * kRows) {
        unsigned long long d[kRows];
#pragma unroll
        for (int r = 0; r < kRows; ++r) {
            const uint32_t j = i0 + 32u * r + (uint32_t)ln;
            d[r] = (i0 + 32u * r < lo + seg && j < n) ? P.desc[P.g_begin + j] : 0ull;
        }
#pragma unroll
        for (int r = 0; r < kRows; ++r) {
            const uint32_t j = i0 + 32u * r + (uint32_t)ln;
            if (i0 + 32u * r < lo + seg && j < n) P.desc[P.g_begin + j] = d[r] + base;
        }
    }
    if (t == 0) *P.base = sh_part[kW];
}

// One CTA (128 threads): frame i of the batch from its slot to its final place (any byte alignment), plus
// the frame's CRC-16, which is appended here: the compaction reads every byte of the frame anyway and is
// memory-bound, so the ~15 instructions per word ride along instead of sitting on k_encode's chain.
// The CRC is linear (zero initial state, no final XOR): the body is cut into 16-byte chunks, rows of 128
// chunks are loaded with one coalesced access each and RIGHT-aligned so that the last row is full; every
// thread keeps a Horner accumulator over its column in the trinomial domain of fa_bits.h (rows are 2048 bytes
// apart: * t^16384 = two shifts; no tables), the 128 columns are combined by a butterfly of power-of-two shifts and the
// (< 16) trailing bytes are appended.  The same registers feed the copy: the destination is cut into ALIGNED
// 16-byte blocks, block k = the last `a` bytes of chunk k - 1 (from the left neighbour lane) and the first 16 - a
// bytes of chunk k, a = destination address mod 16, assembled with funnel shifts (AW = a / 4 selects the words at
// compile time) and written with one 16-byte store; the (< 16) bytes before the first and the (< 32) bytes
// behind the last aligned block are stored bytewise.
struct CompactShared { uint32_t wcrc[4], wpx[4]; };
FA_D U4 u4_zero_enc() { U4 z; z.x = z.y = z.z = z.w = 0; return z; }

template <int AW>
FA_D uint32_t compact_rows(const uint32_t* src, uint8_t* dst_al, uint32_t a, uint32_t n16, uint32_t& px_out) {
    const int t = tid(), ln = lane();
    const uint32_t rows = (n16 + 127u) >> 7;
    const uint32_t first = (rows << 7) - n16;     // threads below this have no chunk in row 0
    const uint32_t sh = (a & 3u) ? 8u * (4u - (a & 3u)) : 32u;
    const int64_t kb0 = a ? 1 : 0;                // first destination block that lies inside the frame
    uint32_t c = 0, px = 0;
    int64_t ci = (int64_t)t - (int64_t)first;
    U4 q = u4_zero_enc(), pq = u4_zero_enc();
    if (ci >= 0) q = ldg128(src + (ci << 2));
    if (ln == 0 && ci >= 1) pq = ldg128(src + ((ci - 1) << 2));     // lane 0's left neighbour sits in another warp
#pragma unroll 2
    for (uint32_t r = 0; r < rows; ++r) {
        const int64_t cn = ci + 128;
        U4 qn = u4_zero_enc(), pn = u4_zero_enc();
        if (r + 1 < rows) {
            qn = ldg128(src + (cn << 2));
            if (ln == 0) pn = ldg128(src + ((cn - 1) << 2));
        }
        // words 3 - AW .. 3 of the chunk on the left
        U4 p;
        p.w = shfl_up(q.w, 1);
        p.z = AW >= 1 ? shfl_up(q.z, 1) : 0u;
        p.y = AW >= 2 ? shfl_up(q.y, 1) : 0u;
        p.x = AW >= 3 ? shfl_up(q.x, 1) : 0u;
        if (ln == 0) p = pq;
        if (ci >= 0) {
            // rows are 2048 bytes apart: * t^16384 = * (t^8 + t) in the trinomial domain (c < 2^18 -> < 2^26)
            c = crct_fold(crct_mulc<0x102u>(c) ^ crct_chunk(q));
            px ^= q.x ^ q.y ^ q.z ^ q.w;
            if (ci >= kb0) {
                const uint32_t W[8] = {p.x, p.y, p.z, p.w, q.x, q.y, q.z, q.w};
                U4 o;
                o.x = funnel_rc(W[3 - AW], W[4 - AW], sh);
                o.y = funnel_rc(W[4 - AW], W[5 - AW], sh);
                o.z = funnel_rc(W[5 - AW], W[6 - AW], sh);
                o.w = funnel_rc(W[6 - AW], W[7 - AW], sh);
                sts128(dst_al + 16 * ci, o);
            }
        }
        q = qn; pq = pn; ci = cn;
    }
    px_out = px;
    return crct_fold(crct_fold(c));
}

// len = P.fsize[i] (body + the two CRC bytes), end = P.desc[P.g_begin + i] (inclusive byte prefix), loaded by the caller
FA_D void compact_frame_cta(const EncParams& P, uint32_t i, CompactShared* cs, uint32_t len, unsigned long long end) {
    if ((long long)end > P.out_capacity) {
        if (tid() == 0) atom_or_global(P.err, kErrEncodeCollect);
        return;
    }
    const uint32_t body = len - 2u;
    uint8_t* dst = P.out + (end - len);
    const uint8_t* sb = P.slots + (long long)i * P.slot_bytes;      // 16-byte aligned
    const uint32_t* src = (const uint32_t*)sb;
    const int t = tid(), ln = lane(), wp = warp();
    const uint32_t a = (uint32_t)((uintptr_t)dst & 15u);
    uint8_t* dst_al = dst - a;
    const uint32_t n16 = body >> 4;
    uint32_t c, px;
    switch (a >> 2) {
        case 0: c = compact_rows<0>(src, dst_al, a, n16, px); break;
        case 1: c = compact_rows<1>(src, dst_al, a, n16, px); break;
        case 2: c = compact_rows<2>(src, dst_al, a, n16, px); break;
        default: c = compact_rows<3>(src, dst_al, a, n16, px); break;
    }
    // thread t's column value still has to move 16 * (127 - t) bytes: lanes first (groups of 1 .. 16), then warps
    {
        uint32_t u;
        u = shfl_xor(c, 1);  if (ln & 1) c = crct_fold(crct_mulc<0x106u>(u)) ^ c;      // * t^128
        u = shfl_xor(c, 2);  if (ln & 2) c = crct_fold(crct_mulc<0x012u>(u)) ^ c;      // * t^256
        u = shfl_xor(c, 4);  if (ln & 4) c = crct_fold(crct_mulc<0x104u>(u)) ^ c;      // * t^512
        u = shfl_xor(c, 8);  if (ln & 8) c = crct_fold(crct_mulc<0x016u>(u)) ^ c;      // * t^1024
        u = shfl_xor(c, 16); if (ln & 16) c = crct_fold(crct_mulc<0x114u>(u)) ^ c;     // * t^2048
    }
    px = redux_xor(px);
    if (ln == 31) { cs->wcrc[wp] = c; cs->wpx[wp] = px; }
    // the bytes outside the aligned blocks: src [0, hb) in front, src [done, body) behind
    const uint32_t h = a ? 16u - a : 0u;
    const uint32_t hb = h < body ? h : body;
    const uint32_t done = n16 > (a ? 1u : 0u) ? 16u * n16 - a : hb;
    if ((uint32_t)t < hb) dst[t] = sb[t];
    if (t >= 32 && t < 96) {
        const uint32_t k = done + (uint32_t)(t - 32);
        if (k < body) dst[k] = sb[k];
    }
    sync();
    if (t == 0) {
        uint32_t v = 0, x = 0;
        for (int w = 0; w < 4; ++w) {                                  // warps are 512 bytes apart: * t^4096
            v = crct_fold(crct_mulc<0x116u>(v)) ^ cs->wcrc[w];
            x ^= cs->wpx[w];
        }
        for (uint32_t k = n16 << 4; k < body; ++k) { v = crct_byte(v, sb[k]); x ^= sb[k]; }
        v = crct_finish(v, x);
        dst[body] = (uint8_t)(v >> 8);
        dst[body + 1] = (uint8_t)v;
    }
}

// Stream header and frame-size table, from the finished byte prefixes (one thread per stream
// header, one per table entry).  desc[g] holds the inclusive byte prefix of frame g.
FA_D void finalize_entry(const EncParams& P, int64_t s, int f, long long* nbytes_out, long long* total_out) {
    const uint32_t g = (uint32_t)(s * P.nframes + f);
    const unsigned long long pre_prev = g == 0 ? 0ull : (P.desc[g - 1] & kDescMask);
    const unsigned long long pre = P.desc[g] & kDescMask;
    const uint32_t g0 = (uint32_t)(s * P.nframes);
    const unsigned long long sstart = g0 == 0 ? 0ull : (P.desc[g0 - 1] & kDescMask);
    uint8_t* sp = P.out + sstart;
    if ((long long)pre > P.out_capacity) return;   // error already flagged by the encoder
    const uint32_t frame_bytes = (uint32_t)(pre - pre_prev) - (f == 0 ? (uint32_t)P.hdr_bytes : 0u);
    uint8_t* e = sp + 54 + 3 * f;
    e[0] = (uint8_t)(frame_bytes >> 16); e[1] = (uint8_t)(frame_bytes >> 8); e[2] = (uint8_t)frame_bytes;
    if (f == 0) {
        sp[0] = 'f'; sp[1] = 'L'; sp[2] = 'a'; sp[3] = 'C';
        sp[4] = 0x00; sp[5] = 0; sp[6] = 0; sp[7] = 34;
        uint8_t* si = sp + 8;
        for (int i = 0; i < 34; ++i) si[i] = 0;
        si[0] = si[2] = (uint8_t)(P.blocksize >> 8);
        si[1] = si[3] = (uint8_t)P.blocksize;
        const uint32_t sr = 44100;
        si[10] = (uint8_t)(sr >> 12); si[11] = (uint8_t)(sr >> 4);
        si[12] = (uint8_t)(((sr & 0xF) << 4) | ((P.nch - 1) << 1) | 1);
        unsigned long long ts = (unsigned long long)P.stream_size;
        if (ts >> 36) ts = 0;  // does not fit the 36-bit field: "unknown"
        si[13] = (uint8_t)(0xF0 | ((ts >> 32) & 0xF));
        si[14] = (uint8_t)(ts >> 24); si[15] = (uint8_t)(ts >> 16); si[16] = (uint8_t)(ts >> 8); si[17] = (uint8_t)ts;
        uint8_t* ap = sp + 42;
        uint32_t alen = 8 + 3 * (uint32_t)P.nframes;
        ap[0] = 0x82; ap[1] = (uint8_t)(alen >> 16); ap[2] = (uint8_t)(alen >> 8); ap[3] = (uint8_t)alen;
        ap[4] = 'f'; ap[5] = 'a'; ap[6] = 'B'; ap[7] = '2';
        uint32_t nf = (uint32_t)P.nframes;
        ap[8] = (uint8_t)(nf >> 24); ap[9] = (uint8_t)(nf >> 16); ap[10] = (uint8_t)(nf >> 8); ap[11] = (uint8_t)nf;
        // bookkeeping: compress.c:402-411 (starts = exclusive prefix), pyx:331-332 (nbytes = diff)
        const unsigned long long send = P.desc[g0 + (uint32_t)P.nframes - 1] & kDescMask;
        P.starts[s] = (long long)sstart;
        nbytes_out[s] = (long long)(send - sstart);
        if (s == P.n_stream - 1 && total_out) *total_out = (long long)send;
    }
}

// ------------------------------------------------------------------------------------------------------
// Fast path, split over three kernels so that no thread ever waits for the serial predictor design:
//   analyze_channel (k_enc_analyze, one CTA per frame): sample statistics, fixed-predictor error sums,
//       windowed autocorrelation -> FrameStats;
//   design_frame (k_enc_design, one THREAD per (frame, channel)): fixed order choice, Levinson-Durbin,
//       order choice, coefficient quantisation -> FramePlan;
//   enc_channel_full / enc_channel_fast (k_encode, persistent CTAs): residuals, Rice parameters, bit
//       packing, CRC-16, copy to the frame's slot.
// The samples are read (and float input quantised) twice; the path is instruction-bound, not
// HBM-bound, and the second read buys a design stage that runs at full machine width.
// Eligible frames: 64 <= blocksize <= 4096 samples; anything else (and any frame whose predictive
// subframe would not beat VERBATIM) takes the general path below.
// ------------------------------------------------------------------------------------------------------
FA_D int fast_level_maxp(int bs, int level_max) {
    if (bs == kMaxBs) return level_max;
    // partitions must be whole thread chunks: partition size a multiple of 32 (or a single partition)
    int z = ctz32((uint32_t)bs);
    int lim = z > 5 ? z - 5 : 0;
    return level_max < lim ? level_max : lim;
}

template <int H, bool FULL>
FA_D void analyze_channel(const EncParams& P, AnShared* sh, const FrameSrc& S, int c, FrameStats* st,
                          int32_t* park) {
    const int t = tid();
    const int ln = lane(), wp = warp();
    const int bs = FULL ? kMaxBs : S.bs;
    const int i0 = t * kSpt;
    const int nvalid = FULL ? kSpt : (bs - i0 >= kSpt ? kSpt : (bs > i0 ? bs - i0 : 0));
    int32_t xw[H + kSpt];
    load_chunk<H, FULL>(S, c, t, xw);
    if (FULL && park != nullptr) {
        // park the channel's int32 samples (quantised / split once, here) for k_encode in the order its threads
        // consume them: [quad q][thread t][4] -- every store and every later load is one coalesced 512-byte
        // access per warp, and the whole 16 KB block is what k_encode's TMA copy brings into shared memory
#pragma unroll
        for (int q = 0; q < kSpt / 4; ++q) {
            U4 v;
            v.x = (uint32_t)xw[H + 4 * q]; v.y = (uint32_t)xw[H + 4 * q + 1];
            v.z = (uint32_t)xw[H + 4 * q + 2]; v.w = (uint32_t)xw[H + 4 * q + 3];
            sts128(park + ((q * kEncThreads + t) << 2), v);
        }
    }

    // ---- pass 1: statistics, fixed-predictor error sums (libFLAC fixed.c: sum |e_k| over i >= 4),
    //      windowed autocorrelation (lpc.c: float data * float window, double accumulation)
    uint32_t orv = 0;
    int32_t mn = 0x7fffffff, mx = (int32_t)0x80000000u;
    uint32_t fe0 = 0, fe1 = 0, fe2 = 0, fe3 = 0, fe4 = 0;
    {
        uint32_t p1 = (uint32_t)xw[H - 1] - (uint32_t)xw[H - 2];
        uint32_t p1b = (uint32_t)xw[H - 2] - (uint32_t)xw[H - 3];
        uint32_t p1c = (uint32_t)xw[H - 3] - (uint32_t)xw[H - 4];
        uint32_t p2 = p1 - p1b, p2b = p1b - p1c;
        uint32_t p3 = p2 - p2b;
#pragma unroll
        for (int j = 0; j < kSpt; ++j) {
            int32_t a0 = xw[H + j];
            if (FULL || j < nvalid) {
                orv |= (uint32_t)a0;
                mn = a0 < mn ? a0 : mn;
                mx = a0 > mx ? a0 : mx;
            }
            uint32_t d1 = (uint32_t)a0 - (uint32_t)xw[H + j - 1];
            uint32_t d2 = d1 - p1, d3 = d2 - p2, d4 = d3 - p3;
            p1 = d1; p2 = d2; p3 = d3;
            if ((j >= 4 || t != 0) && (FULL || j < nvalid)) {
                fe0 = sad_acc(a0, 0, fe0);
                fe1 = sad_acc((int32_t)d1, 0, fe1);
                fe2 = sad_acc((int32_t)d2, 0, fe2);
                fe3 = sad_acc((int32_t)d3, 0, fe3);
                fe4 = sad_acc((int32_t)d4, 0, fe4);
            }
        }
    }
    const bool do_lpc = P.max_lpc_order > 0;
    double ac[H + 1];
#pragma unroll
    for (int l = 0; l <= H; ++l) ac[l] = 0.0;
    if (do_lpc) {
        double wv[H + 1];
#pragma unroll
        for (int l = 0; l <= H; ++l) wv[l] = 0.0;
        // the thread's window values sit in shared memory, [q][t] x 4 floats (filled once per CTA)
        // history: wv[l] = windowed sample (i0 - l)
#pragma unroll
        for (int q = 0; q < H / 4; ++q) {
            if (t != 0) {
                U4 w4 = ldg128(P.window + t * kSpt - H + 4 * q);
                float w0, w1, w2, w3;
                memcpy(&w0, &w4.x, 4); memcpy(&w1, &w4.y, 4); memcpy(&w2, &w4.z, 4); memcpy(&w3, &w4.w, 4);
                wv[H - 4 * q] = (double)fmul((float)xw[4 * q], w0);
                wv[H - 4 * q - 1] = (double)fmul((float)xw[4 * q + 1], w1);
                wv[H - 4 * q - 2] = (double)fmul((float)xw[4 * q + 2], w2);
                wv[H - 4 * q - 3] = (double)fmul((float)xw[4 * q + 3], w3);
            }
        }
        float wq[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int j = 0; j < kSpt; ++j) {
            if ((j & 3) == 0) {
                U4 w4 = ldg128(P.window + t * kSpt + j);
                memcpy(&wq[0], &w4.x, 4); memcpy(&wq[1], &w4.y, 4); memcpy(&wq[2], &w4.z, 4); memcpy(&wq[3], &w4.w, 4);
            }
            wv[0] = (double)fmul((float)xw[H + j], wq[j & 3]);
#pragma unroll
            for (int l = 0; l <= H; ++l) ac[l] = dfma(wv[0], wv[l], ac[l]);
#pragma unroll
            for (int l = H; l >= 1; --l) wv[l] = wv[l - 1];
        }
    }

    // ---- block reduction: REDUX for the integers, transposing butterfly for the doubles
    {
        uint32_t wor = redux_or(orv);
        int32_t wmn = redux_min(mn), wmx = redux_max(mx);
        unsigned long long s0 = warp_sum_u32_wide(fe0), s1 = warp_sum_u32_wide(fe1), s2 = warp_sum_u32_wide(fe2),
                           s3 = warp_sum_u32_wide(fe3), s4 = warp_sum_u32_wide(fe4);
        if (ln == 0) {
            sh->w_or[wp] = wor; sh->w_mn[wp] = wmn; sh->w_mx[wp] = wmx;
            sh->w_fe[wp][0] = s0; sh->w_fe[wp][1] = s1; sh->w_fe[wp][2] = s2; sh->w_fe[wp][3] = s3; sh->w_fe[wp][4] = s4;
        }
        if (do_lpc) {
            double v8 = warp_sum8_d(ac);
            if ((ln & 3) == 0) sh->w_ac[wp][((ln >> 4) & 1) * 4 + ((ln >> 3) & 1) * 2 + ((ln >> 2) & 1)] = v8;
#pragma unroll
            for (int l = 8; l <= H; ++l) {
                double v = warp_sum_d(ac[l]);
                if (ln == 0) sh->w_ac[wp][l] = v;
            }
        } else if (ln <= H) {
            sh->w_ac[wp][ln] = 0.0;
        }
    }
    sync();
    // ---- every thread: frame totals of the sample statistics -> mode (block-uniform)
    uint32_t t_or = 0;
    int32_t a = 0x7fffffff, b = (int32_t)0x80000000u;
#pragma unroll
    for (int w = 0; w < kEncWarps; ++w) {
        t_or |= sh->w_or[w];
        a = sh->w_mn[w] < a ? sh->w_mn[w] : a;
        b = sh->w_mx[w] > b ? sh->w_mx[w] : b;
    }
    int mode = 2, wasted = 0;
    if (a == b) mode = 1;                                           // CONSTANT
    else {
        wasted = ctz32(t_or);                                       // t_or != 0: the samples differ
        // the 32-bit sums of pass 1 are only valid for narrow (unshifted) samples
        if (a < -(1 << kNarrowBits) || b >= (1 << kNarrowBits)) mode = 3;
    }
    if (mode == 3) {
        // wide samples (up to the full int32 range, e.g. the low word of an int64): the fixed-predictor
        // statistics are redone with 64-bit differences (libFLAC: FLAC__fixed_compute_best_predictor_wide);
        // orders whose residual leaves the int32 range are excluded.  The autocorrelation stays valid.
        if (wasted) {
#pragma unroll
            for (int i = 0; i < H + kSpt; ++i) xw[i] >>= wasted;
        }
        unsigned long long we[5] = {0, 0, 0, 0, 0};
        uint32_t bad = 0;
        int64_t q1 = (int64_t)xw[H - 1] - (int64_t)xw[H - 2];
        int64_t q1b = (int64_t)xw[H - 2] - (int64_t)xw[H - 3];
        int64_t q1c = (int64_t)xw[H - 3] - (int64_t)xw[H - 4];
        int64_t q2 = q1 - q1b, q2b = q1b - q1c;
        int64_t q3 = q2 - q2b;
#pragma unroll
        for (int j = 0; j < kSpt; ++j) {
            int64_t e[5];
            e[0] = (int64_t)xw[H + j];
            e[1] = e[0] - (int64_t)xw[H + j - 1];
            e[2] = e[1] - q1; e[3] = e[2] - q2; e[4] = e[3] - q3;
            q1 = e[1]; q2 = e[2]; q3 = e[3];
            if ((j >= 4 || t != 0) && (FULL || j < nvalid)) {
#pragma unroll
                for (int k = 0; k < 5; ++k) {
                    if (!fits_res(e[k])) bad |= 1u << k;
                    we[k] += (unsigned long long)(e[k] < 0 ? -e[k] : e[k]);
                }
            }
        }
        uint32_t wbad = redux_or(bad);
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            unsigned long long v = warp_sum_u64(we[k]);
            if (ln == 0) sh->w_fe[wp][k] = v;
        }
        if (ln == 0) sh->w_bad[wp] = wbad;
        sync();
    }
    // ---- writers: statistics of the samples >> wasted.  Every difference is a multiple of 2^wasted and
    //      float(x) * w scales exactly, so shifting / scaling the narrow sums is exact.
    if (t < 5) {
        unsigned long long v = 0;
        for (int w = 0; w < kEncWarps; ++w) v += sh->w_fe[w][t];
        if (mode == 2) v >>= wasted;
        st->fe[t] = v;
    } else if (t >= 8 && t < 8 + H + 1) {
        int l = t - 8;
        double v = dadd(dadd(sh->w_ac[0][l], sh->w_ac[1][l]), dadd(sh->w_ac[2][l], sh->w_ac[3][l]));
        if (wasted) v *= 1.0 / (double)(1ull << (2 * wasted));
        st->ac[l] = v;
    } else if (t == 31) {
        uint32_t tb = 0;
        if (mode == 3) for (int w = 0; w < kEncWarps; ++w) tb |= sh->w_bad[w];
        st->mode = mode; st->wasted = wasted; st->mn = a >> wasted; st->mx = b >> wasted; st->bad = tb; st->pad = 0;
    }
    sync();   // the partials are reused by the next channel
}


// ------------------------------------------------------------------------------------------------------
// Full frames (4096 samples), two phases per (frame, channel):
//   stage   convert the thread's 32 input samples to int32 exactly once (float -> quantise, int64 -> low /
//           high word), PARK them for k_encode ([quad][thread][4] in the frame's slot, both channels of an
//           8-byte type in one go) and stage the channel in shared memory in the same layout;
//   stats   from shared memory (conflict-free LDS.128, rolled trips of B samples): OR / min / max, the five
//           fixed-predictor error sums, the windowed autocorrelation -> block reduction -> FrameStats.
// The predictor history of a chunk is the end of its left neighbour's chunk, read from the staged channel:
// nothing is converted twice.
// ------------------------------------------------------------------------------------------------------
FA_D uint32_t f2u(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
FA_D float u2f(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
FA_D float fabs32(float f) { return u2f(f2u(f) & 0x7FFFFFFFu); }

// utils.c:232-240 for one sample without the double-precision detour.  For gain > 0 the reference's
// (int)((double)y +- 0.5), y = gain * (x - off), is trunc(y +- 0.5) of the EXACT sum (the double add is exact for
// 1 <= |y| < 2^22, and below 1 it is exact or nowhere near an integer).  A single-precision add that rounds towards
// zero never crosses an integer on the way (an integer between the rounded and the exact sum would itself be a
// float closer to the exact sum), so its truncation is the same integer (checked over all 2.5e9 floats |y| < 2^22);
// the sign of y is the sign of x - off, and y = +-0 gives 0 either way.  Wide values, NaN and non-positive gains
// take the reference's sequence.
FA_D int32_t quant_f32_fast(float x, float off, float gain, bool gain_pos) {
    const float st = fsub(x, off);
    const float y = fmul(gain, st);
    if (gain_pos && fabs32(y) < 4194304.0f) return trunc_fadd(y, u2f((f2u(y) & 0x80000000u) | 0x3F000000u));
    return quant_f32(x, off, gain);
}

// Four samples at once: ONE test (and one branch) for the rare sequence instead of one per sample -- the per-sample
// version spent four of its ten instructions on BSSY / BRA / BSYNC.
FA_D U4 quant_quad_f32(const U4& w, float off, float gain, bool gain_pos) {
    const float y0 = fmul(gain, fsub(u2f(w.x), off)), y1 = fmul(gain, fsub(u2f(w.y), off));
    const float y2 = fmul(gain, fsub(u2f(w.z), off)), y3 = fmul(gain, fsub(u2f(w.w), off));
    const bool fast = gain_pos & (fabs32(y0) < 4194304.0f) & (fabs32(y1) < 4194304.0f) & (fabs32(y2) < 4194304.0f) &
                      (fabs32(y3) < 4194304.0f);       // (false for NaN)
    U4 r;
    if (fast) {
        r.x = (uint32_t)trunc_fadd(y0, u2f((f2u(y0) & 0x80000000u) | 0x3F000000u));
        r.y = (uint32_t)trunc_fadd(y1, u2f((f2u(y1) & 0x80000000u) | 0x3F000000u));
        r.z = (uint32_t)trunc_fadd(y2, u2f((f2u(y2) & 0x80000000u) | 0x3F000000u));
        r.w = (uint32_t)trunc_fadd(y3, u2f((f2u(y3) & 0x80000000u) | 0x3F000000u));
    } else {
        r.x = (uint32_t)quant_f32_fast(u2f(w.x), off, gain, gain_pos);
        r.y = (uint32_t)quant_f32_fast(u2f(w.y), off, gain, gain_pos);
        r.z = (uint32_t)quant_f32_fast(u2f(w.z), off, gain, gain_pos);
        r.w = (uint32_t)quant_f32_fast(u2f(w.w), off, gain, gain_pos);
    }
    return r;
}

FA_D U4 ld128(const void* p) { return lds128(p); }    // plain (coherent) 16-byte load, any address space

// Stage channel c of the frame; c == 0 converts the input (and parks every channel), c == 1 re-reads the high
// words this thread parked a moment ago.
FA_D void analyze_stage(const FrameSrc& S, int c, int t, int32_t* park_frame, int32_t* stage) {
    if (c > 0) {
#pragma unroll
        for (int q = 0; q < kSpt / 4; ++q) {
            const int o = (q * kEncThreads + t) << 2;
            sts128(stage + ((q * kStagePitch + t) << 2), ld128(park_frame + c * kMaxBs + o));
        }
        return;
    }
    if (S.dtype == kI32 || S.dtype == kF32) {
        const bool gain_pos = S.gain32 > 0.0f;
        if (S.vec) {
            // coalesced: the warp reads its 32 threads' 4 KB of input as eight rows of 512 contiguous bytes; lane L of warp
            // w holds, in row k, quad L & 7 of thread 32 w + 4 k + (L >> 3).  Quantising is elementwise, so every lane
            // converts what it loaded and stores it where its owner expects it (8 lanes = the 8 quads of one thread:
            // 64-byte runs in the parked copy, distinct banks in the staged one thanks to the odd row pitch).
            const int wq = t >> 5, L = t & 31;
            const uint32_t* p = (const uint32_t*)S.base + wq * (32 * kSpt);
            U4 v[kSpt / 4];
#pragma unroll
            for (int k = 0; k < kSpt / 4; ++k) v[k] = ldg128(p + ((k * 32 + L) << 2));
#pragma unroll
            for (int k = 0; k < kSpt / 4; ++k) {
                U4 w = v[k];
                if (S.dtype == kF32) w = quant_quad_f32(w, S.off32, S.gain32, gain_pos);
                const int T = wq * 32 + 4 * k + (L >> 3), q = L & 7;
                sts128(park_frame + ((q * kEncThreads + T) << 2), w);
                sts128(stage + ((q * kStagePitch + T) << 2), w);
            }
        } else {
            const uint32_t* p = (const uint32_t*)S.base + t * kSpt;
#pragma unroll 1
            for (int q = 0; q < kSpt / 4; ++q) {      // (unaligned input: scalar loads, rolled)
                U4 w;
                w.x = ldg32(p + 4 * q); w.y = ldg32(p + 4 * q + 1); w.z = ldg32(p + 4 * q + 2); w.w = ldg32(p + 4 * q + 3);
                if (S.dtype == kF32) {
                    w.x = (uint32_t)quant_f32_fast(u2f(w.x), S.off32, S.gain32, gain_pos);
                    w.y = (uint32_t)quant_f32_fast(u2f(w.y), S.off32, S.gain32, gain_pos);
                    w.z = (uint32_t)quant_f32_fast(u2f(w.z), S.off32, S.gain32, gain_pos);
                    w.w = (uint32_t)quant_f32_fast(u2f(w.w), S.off32, S.gain32, gain_pos);
                }
                sts128(park_frame + ((q * kEncThreads + t) << 2), w);
                sts128(stage + ((q * kStagePitch + t) << 2), w);
            }
        }
    } else {
        const unsigned long long* p = (const unsigned long long*)S.base + t * kSpt;
#pragma unroll 2
        for (int q = 0; q < kSpt / 4; ++q) {
            unsigned long long e[4];
            if (S.vec) {
                const U4 a = ldg128(p + 4 * q), b = ldg128(p + 4 * q + 2);
                e[0] = ((unsigned long long)a.y << 32) | a.x; e[1] = ((unsigned long long)a.w << 32) | a.z;
                e[2] = ((unsigned long long)b.y << 32) | b.x; e[3] = ((unsigned long long)b.w << 32) | b.z;
            } else {
#pragma unroll
                for (int i = 0; i < 4; ++i) e[i] = p[4 * q + i];
            }
            if (S.dtype == kF64) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    double d;
                    memcpy(&d, &e[i], 8);
                    e[i] = (unsigned long long)quant_f64(d, S.off64, S.gain64);
                }
            }
            U4 lo, hi;
            lo.x = (uint32_t)e[0]; lo.y = (uint32_t)e[1]; lo.z = (uint32_t)e[2]; lo.w = (uint32_t)e[3];
            hi.x = (uint32_t)(e[0] >> 32); hi.y = (uint32_t)(e[1] >> 32); hi.z = (uint32_t)(e[2] >> 32); hi.w = (uint32_t)(e[3] >> 32);
            const int o = (q * kEncThreads + t) << 2;
            sts128(park_frame + o, lo);
            sts128(park_frame + kMaxBs + o, hi);
            sts128(stage + ((q * kStagePitch + t) << 2), lo);
        }
    }
}

FA_D void analyze_fill_window(const EncParams& P, AnShared* sh) {      // once per CTA (blocksize-4096 levels)
    for (int i = tid(); i < kEncThreads * kSpt / 4; i += kEncThreads) sts128(sh->wqt + 4 * i, ldg128(P.window_qt + 4 * i));
}

// One trip of the autocorrelation pass: B2 staged samples of thread t -> windowed doubles `cur`, every product with the
// lags 0..H (history beyond the trip start comes from `prev`, the previous trip in natural order) -> ac.
template <int H, int B2>
FA_D void analyze_ac_trip(const int32_t* stage, const float* wqt, int it, int t, bool flat, double* cur, const double* prev,
                          double* ac) {
    int32_t x[B2];
#pragma unroll
    for (int qq = 0; qq < B2 / 4; ++qq) {
        const U4 v = lds128(stage + (((it * (B2 / 4) + qq) * kStagePitch + t) << 2));
        x[4 * qq] = (int32_t)v.x; x[4 * qq + 1] = (int32_t)v.y; x[4 * qq + 2] = (int32_t)v.z; x[4 * qq + 3] = (int32_t)v.w;
    }
    if (flat) {
#pragma unroll
        for (int j = 0; j < B2; ++j) cur[j] = (double)(float)x[j];
    } else {
#pragma unroll
        for (int qq = 0; qq < B2 / 4; ++qq) {
            const U4 w4 = lds128(wqt + (((it * (B2 / 4) + qq) * kEncThreads + t) << 2));
            cur[4 * qq] = (double)fmul((float)x[4 * qq], u2f(w4.x));
            cur[4 * qq + 1] = (double)fmul((float)x[4 * qq + 1], u2f(w4.y));
            cur[4 * qq + 2] = (double)fmul((float)x[4 * qq + 2], u2f(w4.z));
            cur[4 * qq + 3] = (double)fmul((float)x[4 * qq + 3], u2f(w4.w));
        }
    }
#pragma unroll
    for (int j = 0; j < B2; ++j) {
#pragma unroll
        for (int l = 0; l <= H; ++l) {
            const double other = l <= j ? cur[j - l] : prev[B2 + j - l];
            ac[l] = dfma(cur[j], other, ac[l]);
        }
    }
}

template <int H>
FA_D void analyze_channel_full(const EncParams& P, AnShared* sh, const FrameSrc& S, int c, FrameStats* st,
                               int32_t* park_frame) {
    constexpr int B = H <= 8 ? 8 : 16;          // samples per rolled trip (>= H: the history of a trip is the trip before)
    const int t = tid();
    const int ln = lane(), wp = warp();
    int32_t* stage = sh->stage;
    analyze_stage(S, c, t, park_frame, stage);
    sync();
    const bool do_lpc = P.max_lpc_order > 0;
    // ---- history: the H samples before the chunk (zeros before the frame)
    int32_t hx[H];
    double hw[H];         // hw[l - 1] = windowed sample (32 t - l)
#pragma unroll
    for (int i = 0; i < H; ++i) { hx[i] = 0; hw[i] = 0.0; }
    if (t != 0) {
#pragma unroll
        for (int qq = 0; qq < H / 4; ++qq) {
            const U4 v = lds128(stage + (((8 - H / 4 + qq) * kStagePitch + (t - 1)) << 2));
            hx[4 * qq] = (int32_t)v.x; hx[4 * qq + 1] = (int32_t)v.y; hx[4 * qq + 2] = (int32_t)v.z; hx[4 * qq + 3] = (int32_t)v.w;
        }
        if (do_lpc) {
#pragma unroll
            for (int qq = 0; qq < H / 4; ++qq) {
                const U4 w4 = lds128(sh->wqt + (((8 - H / 4 + qq) * kEncThreads + (t - 1)) << 2));
                hw[H - 1 - 4 * qq] = (double)fmul((float)hx[4 * qq], u2f(w4.x));
                hw[H - 2 - 4 * qq] = (double)fmul((float)hx[4 * qq + 1], u2f(w4.y));
                hw[H - 3 - 4 * qq] = (double)fmul((float)hx[4 * qq + 2], u2f(w4.z));
                hw[H - 4 - 4 * qq] = (double)fmul((float)hx[4 * qq + 3], u2f(w4.w));
            }
        }
    }
    sync();    // every history read is done: from here on a warp only touches its own quads of the staged channel
    // ---- statistics, fixed-predictor error sums (libFLAC fixed.c: sum |e_k| over i >= 4), windowed
    //      autocorrelation (lpc.c: float data * float window, double accumulation)
    uint32_t orv = 0;
    int32_t mn = 0x7fffffff, mx = (int32_t)0x80000000u;
    uint32_t fe0 = 0, fe1 = 0, fe2 = 0, fe3 = 0, fe4 = 0;
    uint32_t p1 = (uint32_t)hx[H - 1] - (uint32_t)hx[H - 2];
    uint32_t p2, p3;
    int32_t xprev = hx[H - 1];
    {
        const uint32_t p1b = (uint32_t)hx[H - 2] - (uint32_t)hx[H - 3];
        const uint32_t p1c = (uint32_t)hx[H - 3] - (uint32_t)hx[H - 4];
        const uint32_t p2b = p1b - p1c;
        p2 = p1 - p1b;
        p3 = p2 - p2b;
    }
    double ac[H + 1];
#pragma unroll
    for (int l = 0; l <= H; ++l) ac[l] = 0.0;
#pragma unroll 1
    for (int it = 0; it < kSpt / B; ++it) {     // (rolled: unrolling the trips makes ptxas hoist every load and spill)
        int32_t x[B];
#pragma unroll
        for (int qq = 0; qq < B / 4; ++qq) {
            const U4 v = lds128(stage + (((it * (B / 4) + qq) * kStagePitch + t) << 2));
            x[4 * qq] = (int32_t)v.x; x[4 * qq + 1] = (int32_t)v.y; x[4 * qq + 2] = (int32_t)v.z; x[4 * qq + 3] = (int32_t)v.w;
        }
        const bool head = it == 0 && t == 0;     // the frame's first four samples stay out of the fixed-predictor sums
#pragma unroll
        for (int j = 0; j < B; ++j) {
            const int32_t a0 = x[j];
            orv |= (uint32_t)a0;
            mn = a0 < mn ? a0 : mn;
            mx = a0 > mx ? a0 : mx;
            const uint32_t d1 = (uint32_t)a0 - (uint32_t)xprev;
            const uint32_t d2 = d1 - p1, d3 = d2 - p2, d4 = d3 - p3;
            p1 = d1; p2 = d2; p3 = d3;
            xprev = a0;
            if (j >= 4 || !head) {
                fe0 = sad_acc(a0, 0, fe0);
                fe1 = sad_acc((int32_t)d1, 0, fe1);
                fe2 = sad_acc((int32_t)d2, 0, fe2);
                fe3 = sad_acc((int32_t)d3, 0, fe3);
                fe4 = sad_acc((int32_t)d4, 0, fe4);
            }
        }
    }
    // ---- the integer statistics go to the per-warp partials now (REDUX): their registers are free for the second pass
    {
        uint32_t wor = redux_or(orv);
        int32_t wmn = redux_min(mn), wmx = redux_max(mx);
        unsigned long long s0 = warp_sum_u32_wide(fe0), s1 = warp_sum_u32_wide(fe1), s2 = warp_sum_u32_wide(fe2),
                           s3 = warp_sum_u32_wide(fe3), s4 = warp_sum_u32_wide(fe4);
        if (ln == 0) {
            sh->w_or[wp] = wor; sh->w_mn[wp] = wmn; sh->w_mx[wp] = wmx;
            sh->w_fe[wp][0] = s0; sh->w_fe[wp][1] = s1; sh->w_fe[wp][2] = s2; sh->w_fe[wp][3] = s3; sh->w_fe[wp][4] = s4;
        }
        // (reconverge HERE: without it ptxas lets lane 0 run the whole loop below on its own, apart from lanes 1..31 --
        // every instruction of the second pass was issued twice per warp)
        syncwarp();
    }
    // (a second pass over the staged samples: one loop with both the integer statistics and the double-precision
    // products needs more than the 80 registers six resident CTAs leave per thread, and ptxas spills in the loop)
    if (do_lpc) {
        // tukey(0.5) over 4096 samples is exactly 1.0f on samples 1023 .. 3072: warps 1 and 2 skip the table
        const bool flat = wp == 1 || wp == 2;
        // (nine accumulators, eight history values and the trip's eight samples as doubles need ~96 registers: at 80
        // ptxas kept three accumulators in local memory, one spill access per sample.  Measured per 10^9 samples:
        // 6 CTAs/SM with spills 7.98 ms, 6 CTAs with 4-sample trips 7.75, 5 CTAs with 8-sample trips 7.40)
#ifndef FAB_AN_B2
#define FAB_AN_B2 8
#endif
        constexpr int B2 = FAB_AN_B2;
#ifndef FAB_AN_NO_PINGPONG
        if constexpr (H == B2) {
            // the history of a trip is exactly the trip before it: two trips per turn, each writing the array the other
            // one reads as its history -- no register moves between trips (they were 2 of ~54 instructions per sample)
            double pa[B2], pb[B2];
#pragma unroll
            for (int j = 0; j < B2; ++j) pa[j] = hw[B2 - 1 - j];
#pragma unroll 1
            for (int it = 0; it < kSpt / B2; it += 2) {
                analyze_ac_trip<H, B2>(stage, sh->wqt, it, t, flat, pb, pa, ac);
                analyze_ac_trip<H, B2>(stage, sh->wqt, it + 1, t, flat, pa, pb, ac);
            }
        } else
#endif
#pragma unroll 1
        for (int it = 0; it < kSpt / B2; ++it) {
            int32_t x[B2];
#pragma unroll
            for (int qq = 0; qq < B2 / 4; ++qq) {
                const U4 v = lds128(stage + (((it * (B2 / 4) + qq) * kStagePitch + t) << 2));
                x[4 * qq] = (int32_t)v.x; x[4 * qq + 1] = (int32_t)v.y; x[4 * qq + 2] = (int32_t)v.z; x[4 * qq + 3] = (int32_t)v.w;
            }
            double cw[B2];      // windowed samples of this trip
            if (flat) {
#pragma unroll
                for (int j = 0; j < B2; ++j) cw[j] = (double)(float)x[j];
            } else {
#pragma unroll
                for (int qq = 0; qq < B2 / 4; ++qq) {
                    const U4 w4 = lds128(sh->wqt + (((it * (B2 / 4) + qq) * kEncThreads + t) << 2));
                    cw[4 * qq] = (double)fmul((float)x[4 * qq], u2f(w4.x));
                    cw[4 * qq + 1] = (double)fmul((float)x[4 * qq + 1], u2f(w4.y));
                    cw[4 * qq + 2] = (double)fmul((float)x[4 * qq + 2], u2f(w4.z));
                    cw[4 * qq + 3] = (double)fmul((float)x[4 * qq + 3], u2f(w4.w));
                }
            }
#pragma unroll
            for (int j = 0; j < B2; ++j) {
#pragma unroll
                for (int l = 0; l <= H; ++l) {
                    const double other = l <= j ? cw[j - l] : hw[l - j - 1];
                    ac[l] = dfma(cw[j], other, ac[l]);
                }
            }
            // history of the next trip: the trip's samples, then what remains of the old history
#pragma unroll
            for (int l = H; l >= 1; --l) hw[l - 1] = l <= B2 ? cw[B2 - l] : hw[l - 1 - B2];
        }
    }

    // ---- the autocorrelation partials: through the warp's own, consumed quads of the staged channel
    {
        if (do_lpc) {
            // every lane parks its partials, then a few lanes per lag sum them in lane order: a fixed
            // order (deterministic bytes) at a fraction of the instructions of a register butterfly over doubles
            // (the partials overwrite the warp's own, consumed quads of the staged channel: lag l goes to half (l & 1) of
            // quad (l >> 1), rotated by l columns so that the column reads below are conflict-free)
            syncwarp();
#pragma unroll
            for (int l = 0; l <= H; ++l)
                ((double*)(stage + (((l >> 1) * kStagePitch + 32 * wp) << 2) + (l & 1) * 64))[(ln + l) & 31] = ac[l];
            syncwarp();
            // NP lanes per lag, each sums a contiguous third (half) of the 32 columns; the parts meet in the first one
            constexpr int NP = (H + 1) * 3 <= 32 ? 3 : 2;
            const int l = ln / NP, part = ln - l * NP;
            double acc = 0.0;
            if (l <= H) {
                const double* r = (const double*)(stage + (((l >> 1) * kStagePitch + 32 * wp) << 2) + (l & 1) * 64);
                const int c0 = (part * 32) / NP, c1 = ((part + 1) * 32) / NP;
                constexpr int kMin = 32 / NP;        // every part has kMin or kMin + 1 columns
#pragma unroll
                for (int k = 0; k < kMin; ++k) acc = dadd(acc, r[(c0 + k + l) & 31]);
                if (c1 - c0 > kMin) acc = dadd(acc, r[(c0 + kMin + l) & 31]);
            }
            const double a1 = shfl_down_d(acc, 1), a2 = shfl_down_d(acc, 2);
            if (part == 0 && l <= H) sh->w_ac[wp][l] = NP == 3 ? dadd(dadd(acc, a1), a2) : dadd(acc, a1);
        } else if (ln <= H) {
            sh->w_ac[wp][ln] = 0.0;
        }
    }
    sync();
    // ---- every thread: frame totals of the sample statistics -> mode (block-uniform)
    uint32_t t_or = 0;
    int32_t a = 0x7fffffff, b = (int32_t)0x80000000u;
#pragma unroll
    for (int w = 0; w < kEncWarps; ++w) {
        t_or |= sh->w_or[w];
        a = sh->w_mn[w] < a ? sh->w_mn[w] : a;
        b = sh->w_mx[w] > b ? sh->w_mx[w] : b;
    }
    int mode = 2, wasted = 0;
    if (a == b) mode = 1;                                           // CONSTANT
    else {
        wasted = ctz32(t_or);                                       // t_or != 0: the samples differ
        // the 32-bit sums above are only valid for narrow (unshifted) samples
        if (a < -(1 << kNarrowBits) || b >= (1 << kNarrowBits)) mode = 3;
    }
    if (mode == 3) {
        // wide samples (up to the full int32 range, e.g. the low word of an int64): the fixed-predictor
        // statistics are redone with 64-bit differences on the samples >> wasted (libFLAC:
        // FLAC__fixed_compute_best_predictor_wide); orders whose residual leaves the int32 range are excluded.
        // The autocorrelation stays valid.
        unsigned long long we[5] = {0, 0, 0, 0, 0};
        uint32_t bad = 0;
        // (the four samples before the chunk are fetched again -- the last quad thread t - 1 parked -- rather than kept
        // in registers across the loops above, which are short of registers as it is)
        U4 hq = u4_zero_enc();
        if (t != 0) hq = ld128(park_frame + c * kMaxBs + ((7 * kEncThreads + (t - 1)) << 2));
        const int32_t h4[4] = {(int32_t)hq.x >> wasted, (int32_t)hq.y >> wasted, (int32_t)hq.z >> wasted, (int32_t)hq.w >> wasted};
        int64_t q1 = (int64_t)h4[3] - (int64_t)h4[2];
        int64_t q1b = (int64_t)h4[2] - (int64_t)h4[1];
        int64_t q1c = (int64_t)h4[1] - (int64_t)h4[0];
        int64_t q2 = q1 - q1b, q2b = q1b - q1c;
        int64_t q3 = q2 - q2b;
        int64_t prev = (int64_t)h4[3];
#pragma unroll 1
        for (int q = 0; q < kSpt / 4; ++q) {
            const U4 v = ld128(park_frame + c * kMaxBs + ((q * kEncThreads + t) << 2));   // (this thread parked them itself)
            const int32_t xs[4] = {(int32_t)v.x >> wasted, (int32_t)v.y >> wasted, (int32_t)v.z >> wasted, (int32_t)v.w >> wasted};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                int64_t e[5];
                e[0] = (int64_t)xs[j];
                e[1] = e[0] - prev;
                e[2] = e[1] - q1; e[3] = e[2] - q2; e[4] = e[3] - q3;
                q1 = e[1]; q2 = e[2]; q3 = e[3];
                prev = e[0];
                if (q > 0 || t != 0) {
#pragma unroll
                    for (int k = 0; k < 5; ++k) {
                        if (!fits_res(e[k])) bad |= 1u << k;
                        we[k] += (unsigned long long)(e[k] < 0 ? -e[k] : e[k]);
                    }
                }
            }
        }
        uint32_t wbad = redux_or(bad);
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            unsigned long long v = warp_sum_u64(we[k]);
            if (ln == 0) sh->w_fe[wp][k] = v;
        }
        if (ln == 0) sh->w_bad[wp] = wbad;
        sync();
    }
    // ---- writers: statistics of the samples >> wasted.  Every difference is a multiple of 2^wasted and
    //      float(x) * w scales exactly, so shifting / scaling the narrow sums is exact.
    if (t < 5) {
        unsigned long long v = 0;
        for (int w = 0; w < kEncWarps; ++w) v += sh->w_fe[w][t];
        if (mode == 2) v >>= wasted;
        st->fe[t] = v;
    } else if (t >= 8 && t < 8 + H + 1) {
        int l = t - 8;
        double v = dadd(dadd(sh->w_ac[0][l], sh->w_ac[1][l]), dadd(sh->w_ac[2][l], sh->w_ac[3][l]));
        if (wasted) v *= 1.0 / (double)(1ull << (2 * wasted));
        st->ac[l] = v;
    } else if (t == 31) {
        uint32_t tb = 0;
        if (mode == 3) for (int w = 0; w < kEncWarps; ++w) tb |= sh->w_bad[w];
        st->mode = mode; st->wasted = wasted; st->mn = a >> wasted; st->mx = b >> wasted; st->bad = tb; st->pad = 0;
    }
    sync();   // the partials and the staged channel are reused by the next channel / frame
}

// One thread: pull full frame g of the input towards the L2 (the CTA that will analyse it is busy with another frame).
FA_D void analyze_prefetch(const EncParams& P, uint32_t g) {
    const int64_t s = (int64_t)(g / (uint32_t)P.nframes);
    const int f = (int)(g % (uint32_t)P.nframes);
    const int64_t samp0 = (int64_t)f * P.blocksize;
    if (P.stream_size - samp0 < P.blocksize) return;
    const int esize = (P.dtype == kI32 || P.dtype == kF32) ? 4 : 8;
    const unsigned char* base = (const unsigned char*)P.data + (s * P.stream_size + samp0) * esize;
    if (((uintptr_t)base & 15) == 0) prefetch_l2_bulk(base, (uint32_t)(P.blocksize * esize));
}

// FULL: the caller is the kernel for full (4096-sample) frames and skips every other frame; !FULL: the kernel for the
// rest (last frame of a stream, blocksize-1152 levels).  Two kernels because inlining both bodies into one makes
// ptxas spill inside the full-frame loops (3.8 KB of spill stores against 84 bytes).
template <int H, bool FULL>
FA_D void analyze_frame_cta(const EncParams& P, uint32_t g, AnShared* sh) {
    const int64_t s = (int64_t)(g / (uint32_t)P.nframes);
    const int f = (int)(g % (uint32_t)P.nframes);
    const int64_t samp0 = (int64_t)f * P.blocksize;
    const int bs = (int)((P.stream_size - samp0) < P.blocksize ? (P.stream_size - samp0) : P.blocksize);
    FrameStats* st = P.stats + (size_t)(g - P.g_begin) * P.nch;
    if ((bs == kMaxBs) != FULL) return;
    if (!FULL && fixed_done(P, g)) return;
    if (bs < 64) {
        if (tid() < P.nch) st[tid()].mode = 0;
        return;
    }
    FrameSrc S;
    S.dtype = P.dtype; S.bs = bs;
    S.off32 = 0.f; S.gain32 = 0.f; S.off64 = 0.; S.gain64 = 0.;
    if (P.dtype == kF32) { S.off32 = ((const float*)P.offsets)[s]; S.gain32 = ((const float*)P.gains)[s]; }
    if (P.dtype == kF64) { S.off64 = ((const double*)P.offsets)[s]; S.gain64 = ((const double*)P.gains)[s]; }
    const int esize = (P.dtype == kI32 || P.dtype == kF32) ? 4 : 8;
    S.base = (const unsigned char*)P.data + (s * P.stream_size + samp0) * esize;
    S.vec = (((uintptr_t)S.base) & 15) == 0;
    // full frames are parked as planar int32 in the frame's (still unused) output slot: k_encode then reads
    // plain integers (quantised / split exactly once) through one TMA copy per channel
    int32_t* slot = (int32_t*)(P.slots + (int64_t)(g - P.g_begin) * P.slot_bytes);
    for (int c = 0; c < P.nch; ++c) {
        if constexpr (FULL) analyze_channel_full<H>(P, sh, S, c, st + c, slot);
        else analyze_channel<H, false>(P, sh, S, c, st + c, nullptr);
    }
}

// One thread: the plan of (frame, channel) record i of the batch.
FA_D void design_frame(const EncParams& P, int64_t i) {
    const uint32_t g = P.g_begin + (uint32_t)(i / P.nch);
    const int f = (int)(g % (uint32_t)P.nframes);
    const int64_t samp0 = (int64_t)f * P.blocksize;
    const int bs = (int)((P.stream_size - samp0) < P.blocksize ? (P.stream_size - samp0) : P.blocksize);
    if (fixed_done(P, g)) return;
    const FrameStats& st = P.stats[i];
    FramePlan pl;
    memset(&pl, 0, sizeof(pl));
    pl.mode = (uint8_t)st.mode;
    if (bs == kMaxBs && st.mode >= 2 && (P.max_porder < 2 || P.max_porder > 7)) pl.mode = 0;   // (no preset does this)
    if (pl.mode >= 2) {
        DesignIO d;
        for (int k = 0; k < 5; ++k) d.t_fe[k] = st.fe[k];
        for (int l = 0; l <= kMaxOrd; ++l) d.t_ac[l] = l <= P.max_lpc_order ? st.ac[l] : 0.0;
        const int bps = 32 - st.wasted;
        const int level_maxp = fast_level_maxp(bs, P.max_porder);
        uint32_t maxabs = 0;
        if (st.mode == 2) maxabs = (uint32_t)(-(int64_t)st.mn > (int64_t)st.mx ? -(int64_t)st.mn : (int64_t)st.mx);
        design_fixed(&d, bs, bps, st.bad, level_maxp);
        design_lpc(&d, bs, bps, P.max_lpc_order, P.qlp_precision, level_maxp, maxabs);
        pl.wasted = (uint8_t)st.wasted;
        if (d.cand_ok[0]) {
            // size of the FIXED subframe with a single Rice partition, from the analysis pass's sum |e| (the first four
            // samples are not in that sum; at most `order` of them are warm-up): what k_encode compares the LPC
            // candidate's like-for-like estimate with before it spends a second residual pass on the fixed predictor
            int k0 = 0;
            const uint32_t o = (uint32_t)d.cand[0].order;
            uint32_t rb = rice_estimate(d.t_fe[o], (uint32_t)bs - o, k0);
            pl.fixed_bits = o * (uint32_t)bps + rb + 6u + (k0 >= 15 ? 1u : 0u);
        }
        pl.ok0 = (uint8_t)d.cand_ok[0];
        pl.ok1 = (uint8_t)d.cand_ok[1];
        pl.ord0 = (uint8_t)d.cand[0].order;
        pl.maxp0 = (uint8_t)d.maxp[0];
        if (d.cand_ok[1]) {
            pl.ord1 = (uint8_t)d.cand[1].order;
            pl.shift1 = (uint8_t)d.cand[1].shift;
            pl.prec1 = (uint8_t)d.cand[1].prec;
            pl.wide1 = (uint8_t)d.cand[1].wide;
            pl.maxp1 = (uint8_t)d.maxp[1];
            for (int j = 0; j < kMaxOrd; ++j) pl.qlp[j] = (int16_t)d.cand[1].qlp[j];
        }
    }
    P.plans[i] = pl;
    if (P.hdrs != nullptr) {
        PlanHeader ph;
        memset(&ph, 0, sizeof(ph));
        if (bs == kMaxBs && pl.mode >= 2 && pl.wasted == 0) {
            const int c = (int)(i % P.nch);
            const int32_t* park = (const int32_t*)(P.slots + (int64_t)(g - P.g_begin) * P.slot_bytes) + (int64_t)c * kMaxBs;
            uint8_t fh[16];
            const int nfh = c == 0 ? build_frame_header(fh, P.crc->crc8, bs, f, P.nch) : 0;
            if (pl.ok1) {
                uint32_t n = 0;
                for (int b = 0; b < nfh; ++b) hdr_put(ph.lpc, n, fh[b], 8);
                hdr_put(ph.lpc, n, (uint32_t)(32 + pl.ord1 - 1) << 1, 8);
                for (int j = 0; j < pl.ord1; ++j) hdr_put(ph.lpc, n, (uint32_t)park[park_word(j)], 32);
                hdr_put(ph.lpc, n, (uint32_t)(pl.prec1 - 1), 4);
                hdr_put(ph.lpc, n, (uint32_t)pl.shift1 & 31u, 5);
                for (int j = 0; j < pl.ord1; ++j) hdr_put(ph.lpc, n, (uint32_t)(int32_t)pl.qlp[j] & ((1u << pl.prec1) - 1u), pl.prec1);
                ph.nbits_lpc = n;
            }
            if (pl.ok0) {
                uint32_t n = 0;
                for (int b = 0; b < nfh; ++b) hdr_put(ph.fix, n, fh[b], 8);
                hdr_put(ph.fix, n, (uint32_t)(8 + pl.ord0) << 1, 8);
                for (int j = 0; j < pl.ord0; ++j) hdr_put(ph.fix, n, (uint32_t)park[park_word(j)], 32);
                ph.nbits_fix = n;
            }
        }
        P.hdrs[i] = ph;
    }
}

// residuals of a fixed predictor by repeated differences (order <= 4 subtractions per sample)
template <int H>
FA_D void fixed_residual32(int order, const int32_t* xw, int32_t* r) {
    uint32_t p1 = (uint32_t)xw[H - 1] - (uint32_t)xw[H - 2];
    uint32_t p1b = (uint32_t)xw[H - 2] - (uint32_t)xw[H - 3];
    uint32_t p1c = (uint32_t)xw[H - 3] - (uint32_t)xw[H - 4];
    uint32_t p2 = p1 - p1b, p2b = p1b - p1c;
    uint32_t p3 = p2 - p2b;
#pragma unroll
    for (int j = 0; j < kSpt; ++j) {
        uint32_t d0 = (uint32_t)xw[H + j];
        uint32_t d1 = d0 - (uint32_t)xw[H + j - 1];
        uint32_t d2 = d1 - p1, d3 = d2 - p2, d4 = d3 - p3;
        p1 = d1; p2 = d2; p3 = d3;
        r[j] = (int32_t)(order == 0 ? d0 : order == 1 ? d1 : order == 2 ? d2 : order == 3 ? d3 : d4);
    }
}

template <int H, bool FULL>
FA_D bool enc_channel_fast(const EncParams& P, EncCtx& X, const FrameSrc& S, int c, int f, uint32_t g, int bitpos0,
                           int& bitpos_end) {
    EncShared* sh = X.sh;
    EncHot* hot = X.hot;
    uint32_t* out = X.out;
    const int t = tid();
    const int ln = lane(), wp = warp();
    const int bs = FULL ? kMaxBs : S.bs;
    const int i0 = t * kSpt;
    const int nvalid = FULL ? kSpt : (bs - i0 >= kSpt ? kSpt : (bs > i0 ? bs - i0 : 0));
    // ---- the plan of this (frame, channel): three broadcast loads, decoded in registers
    const unsigned char* pp = (const unsigned char*)(P.plans + ((size_t)(g - P.g_begin) * P.nch + c));
    const U4 pa = ldg128(pp), pb = ldg128(pp + 16), pc = ldg128(pp + 32);
    const int mode = (int)(pa.x & 0xFFu);
    if (mode == 0) return false;
    const int wasted = (int)((pa.x >> 8) & 0xFFu);
    const int bps = 32 - wasted;
    const int ok0 = (int)((pa.x >> 16) & 0xFFu), ok1 = (int)(pa.x >> 24);
    const int ord0 = (int)(pa.y & 0xFFu), ord1 = (int)((pa.y >> 8) & 0xFFu);
    const int shift1 = (int)((pa.y >> 16) & 0xFFu), prec1 = (int)(pa.y >> 24);
    const int wide1 = (int)(pa.z & 0xFFu), maxp0 = (int)((pa.z >> 8) & 0xFFu), maxp1 = (int)((pa.z >> 16) & 0xFFu);
    const bool wide = mode == 3;
    int32_t xw[H + kSpt];
    load_chunk<H, FULL>(S, c, t, xw);
    const bool retiring = !X.retired;

    if (mode == 1) {
        if (retiring) {
            sync();
            retire_copyout(P, X);
            X.retired = true;
        }
        // (as in enc_channel_full: every thread is done with the copy-out of the previous frame before thread 0 packs
        // this one into `out` and overwrites prev_g / prev_nbytes)
        sync();
        bitpos_end = bitpos0 + (c == 0 ? 8 * frame_header_bytes(bs, f) : 0) + subframe_header_bits(0, 0, 0, 32, 0);
        if (t == 0) {
            Pk pk;
            pk_begin(pk, out, bitpos0);
            if (c == 0) emit_frame_header(pk, hot->crc8, bs, f, P.nch);
            emit_subframe_header(pk, 0, 0, 0);
            emit_sample(pk, xw[H], 32);
            pk_end(pk, hot->tail_val[c][0], hot->tail_word[c][0]);
        }
        return true;
    }
    if (wasted) {
#pragma unroll
        for (int i = 0; i < H + kSpt; ++i) xw[i] >>= wasted;
    }

    // ---- pass 2: per-chunk sums of |residual| for both candidates
    const int js = (t == 0) ? 0 : -1;   // thread 0 skips its first `order` samples (warm-up)
    int32_t r[kSpt];
    if (t < 2) sh->cand_ok[t] = t == 0 ? ok0 : ok1;
    if (ok0) {
        unsigned long long asum;
        if (!wide) {
            fixed_residual32<H>(ord0, xw, r);
            uint32_t a32 = 0;
#pragma unroll
            for (int j = 0; j < kSpt; ++j)
                if ((j >= H || js < 0 || j >= ord0) && (FULL || j < nvalid)) a32 = sad_acc(r[j], 0, a32);
            asum = a32;
        } else {
            int32_t cf[H];
            fixed_coefs(ord0, cf, H);
            uint32_t fitmask = residual64<H>(ord0, xw, cf, 0, r);
            asum = 0;
#pragma unroll
            for (int j = 0; j < kSpt; ++j)
                if ((j >= H || js < 0 || j >= ord0) && (FULL || j < nvalid))
                    asum += (unsigned long long)(r[j] < 0 ? -(int64_t)r[j] : (int64_t)r[j]);
            uint32_t vmask = nvalid >= 32 ? 0xFFFFFFFFu : ((1u << nvalid) - 1u);
            if (t == 0) vmask &= ~((1u << ord0) - 1u);
            if ((fitmask & vmask) != vmask) asum = ~0ull;
        }
        sh->csum[0][t] = asum;
    }
    int32_t coef[H];
    {
        const uint32_t qw[8] = {pb.x, pb.y, pb.z, pb.w, pc.x, pc.y, pc.z, pc.w};
#pragma unroll
        for (int m = 0; m < H; ++m) coef[m] = (int32_t)(int16_t)(uint16_t)(qw[m >> 1] >> (16 * (m & 1)));
    }
    if (ok1) {
        unsigned long long asum = 0;
        if (!wide1) {
            residual32_dispatch<H>(ord1, xw, coef, shift1, r);
            uint32_t a32 = 0;
#pragma unroll
            for (int j = 0; j < kSpt; ++j)
                if ((j >= H || js < 0 || j >= ord1) && (FULL || j < nvalid)) a32 = sad_acc(r[j], 0, a32);
            asum = a32;
        } else {
            uint32_t fitmask = residual64<H>(ord1, xw, coef, shift1, r);
#pragma unroll
            for (int j = 0; j < kSpt; ++j)
                if ((j >= H || js < 0 || j >= ord1) && (FULL || j < nvalid))
                    asum += (unsigned long long)(r[j] < 0 ? -(int64_t)r[j] : (int64_t)r[j]);
            uint32_t vmask = nvalid >= 32 ? 0xFFFFFFFFu : ((1u << nvalid) - 1u);
            if (t == 0) vmask &= ~((1u << ord1) - 1u);
            if ((fitmask & vmask) != vmask) asum = ~0ull;   // a residual does not fit: poisons the candidate
        }
        sh->csum[1][t] = asum;
    }
    sync();   // B3: chunk sums, cand_ok and (retiring) the byte offset of the previous frame are visible
    if (retiring) retire_copyout(P, X);   // previous frame: CRC partials + copy to HBM
    if (wp < 2 && sh->cand_ok[wp]) {
        const int cd = wp;
        const int maxp = cd == 0 ? maxp0 : maxp1;
        const int cpp = FULL ? (kEncThreads >> maxp) : (maxp > 0 ? ((bs >> maxp) >> 5) : kEncThreads);   // chunks per finest partition
        bool poisoned = false;
        for (int part = ln; part < (1 << maxp); part += 32) {
            unsigned long long v = 0;
            for (int q = 0; q < cpp; ++q) {
                unsigned long long cs = sh->csum[cd][part * cpp + q];
                poisoned = poisoned || cs == ~0ull;
                v += cs;
            }
            sh->psum[cd][part] = v;
        }
        if (ballot(poisoned) != 0) {
            if (ln == 0) sh->cand_ok[cd] = 0;
            syncwarp();
        } else {
            syncwarp();
            rice_search_warp(sh, cd, bs, cd == 0 ? ord0 : ord1, maxp);
        }
    }
    sync();   // B4
    if (retiring) X.retired = true;    // the copy-out (before B4) is ordered before the packing below by B5
    // ---- every thread: pick the winner (stream_encoder.c process_subframe_: smallest estimate wins)
    const uint32_t verbatim_bits = (uint32_t)bps * (uint32_t)bs;
    int win = -1;
    {
        uint32_t best = verbatim_bits;
        for (int cd = 0; cd < 2; ++cd) {
            if (!sh->cand_ok[cd]) continue;
            const uint32_t ord = (uint32_t)(cd == 0 ? ord0 : ord1);
            uint32_t bits = ord * (uint32_t)bps + sh->cand[cd].res_bits + (cd == 1 ? 9u + ord * (uint32_t)prec1 : 0u);
            if (bits < best) { best = bits; win = cd; }
        }
    }
    // (block-uniform; the barrier keeps the general path's writes to sh->cand behind the reads above)
    if (win < 0) { sync(); return false; }
    const int order = win == 0 ? ord0 : ord1;
    const int porder = sh->cand[win].porder, rice2 = sh->cand[win].rice2, plen = rice2 ? 5 : 4;
    if (win == 0) {
        if (wide) {
            int32_t cf[H];
            fixed_coefs(order, cf, H);
            (void)residual64<H>(order, xw, cf, 0, r);
        } else {
            fixed_residual32<H>(order, xw, r);
        }
    }
    // ---- exact code lengths of the chunk, block scan
    int part;
    bool part_start;
    if (FULL) {
        const int psh = 12 - porder;             // log2(partition size)
        part = i0 >> psh;
        part_start = (i0 & ((1 << psh) - 1)) == 0;
    } else {
        const int psize = bs >> porder;          // a multiple of 32 when porder > 0
        part = porder > 0 ? i0 / psize : 0;
        part_start = nvalid > 0 && i0 == part * psize;
        if (nvalid == 0) part = 0;
    }
    const int k = sh->kpar[win][(1 << porder) - 1 + part];
    uint32_t lens = part_start ? (uint32_t)plen : 0u;
    uint32_t qmax = 0;
    int nres = 0;
#pragma unroll
    for (int j = 0; j < kSpt; ++j) {
        if ((j >= H || js < 0 || j >= order) && (FULL || j < nvalid)) {
            uint32_t u = ((uint32_t)r[j] << 1) ^ (uint32_t)(r[j] >> 31);
            uint32_t q = u >> k;
            lens += q;
            qmax = q > qmax ? q : qmax;
            nres++;
        }
    }
    lens += (uint32_t)nres * (uint32_t)(k + 1);
    uint32_t inc = lens;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t n = shfl_up(inc, d);
        if (ln >= d) inc += n;
    }
    if (ln == 31) sh->scan[wp] = inc;
    sync();   // B5
    uint32_t wbase = 0, total = 0;
#pragma unroll
    for (int w = 0; w < kEncWarps; ++w) {
        uint32_t x = sh->scan[w];
        if (w < wp) wbase += x;
        total += x;
    }
    const uint32_t excl = wbase + inc - lens;
    const int ptype = win == 0 ? 2 : 3;
    const int prec = win == 0 ? 0 : prec1;
    const int hdr_bits = subframe_header_bits(ptype, order, wasted, bps, prec);
    if ((uint32_t)hdr_bits + total >= verbatim_bits + 8u) return false;   // VERBATIM is smaller: general path
    const int sub0 = bitpos0 + (c == 0 ? 8 * frame_header_bytes(bs, f) : 0);
    const int body0 = sub0 + hdr_bits;

    // ---- pack
    bitpos_end = body0 + (int)total;
    Pk pk;
    if (t == 0) {
        pk_begin(pk, out, bitpos0);
        if (c == 0) emit_frame_header(pk, hot->crc8, bs, f, P.nch);
        emit_subframe_header(pk, ptype, order, wasted);
        for (int j = 0; j < order; ++j) emit_sample(pk, xw[H + j], bps);
        if (ptype == 3) {
            pk_emit(pk, (uint32_t)(prec1 - 1), 4);
            pk_emit(pk, (uint32_t)shift1 & 31u, 5);
            for (int j = 0; j < order; ++j) pk_emit(pk, (uint32_t)coef[j] & ((1u << prec1) - 1u), prec1);
        }
        pk_emit(pk, (uint32_t)rice2, 2);
        pk_emit(pk, (uint32_t)porder, 4);
    } else {
        pk_begin(pk, out, body0 + (int)excl);
    }
    if (FULL || nvalid > 0) {
        if (part_start) pk_emit(pk, (uint32_t)k, plen);
        if (qmax + (uint32_t)k + 1u <= 32u) {
            // every code of the chunk fits one emit: branch-free loop on a (hi, lo) register pair
            uint32_t hi = (uint32_t)(pk.acc >> 32), lo = 0;
            int fill = pk.fill, word = pk.word;
            const uint32_t kbit = 1u << k, kmask = kbit - 1u;
            const int k1 = k + 1;
#pragma unroll
            for (int j = 0; j < kSpt; ++j) {
                if ((j >= H || js < 0 || j >= order) && (FULL || j < nvalid)) {
                    uint32_t u = ((uint32_t)r[j] << 1) ^ (uint32_t)(r[j] >> 31);
                    uint32_t low = (u & kmask) | kbit;
                    int len = (int)(u >> k) + k1;
                    uint64_t v = (uint64_t)low << (64 - fill - len);
                    hi |= (uint32_t)(v >> 32);
                    lo |= (uint32_t)v;
                    fill += len;
                    if (fill >= 32) {
                        out[ow(word)] = hi;
                        word++;
                        hi = lo;
                        lo = 0;
                        fill -= 32;
                    }
                }
            }
            pk.acc = (uint64_t)hi << 32;
            pk.fill = fill;
            pk.word = word;
        } else {
#pragma unroll 1
            for (int j = 0; j < kSpt; ++j) {
                if ((j >= H || js < 0 || j >= order) && (FULL || j < nvalid)) {
                    int32_t rv = r[0];
#pragma unroll
                    for (int q = 1; q < kSpt; ++q) rv = (q == j) ? r[q] : rv;   // keeps r[] in registers
                    uint32_t u = ((uint32_t)rv << 1) ^ (uint32_t)(rv >> 31);
                    pk_rice(pk, u, k);
                }
            }
        }
        pk_end(pk, hot->tail_val[c][t], hot->tail_word[c][t]);
    }
    return true;
}

// short frames (the last frame of a stream, blocksize-1152 levels): the generic variant, out of line
// (by value: a by-reference context would force the hot path's copy of it into local memory)
template <int H>
FA_DNOINL int enc_channel_short(const EncParams P, EncCtx X, const FrameSrc S, int c, int f, uint32_t g, int bitpos0) {
    int bitpos_end = -1;
    bool done = enc_channel_fast<H, false>(P, X, S, c, f, g, bitpos0, bitpos_end);
    if (!done) {
        // the short path has retired the previous frame before giving up
        X.retired = true;
        return -1;
    }
    return bitpos_end;
}

// ------------------------------------------------------------------------------------------------------
// Full 4096-sample frames: the hot path.
//
// Input: the channel's int32 samples as k_enc_analyze parked them ([quad][thread][4], 16 KB).  One TMA bulk
// copy (cp.async.bulk -> UBLKCP, completion on an mbarrier) brings the block into shared memory while the
// threads fetch the plan and their predictor history; every later access is a conflict-free LDS.128 / STS.128
// of the thread's own quads.  Per (frame, channel):
//   residual pass   ONE candidate (the LPC plan if there is one, else the fixed predictor): residuals of the
//                   thread's 32 samples in two rolled trips of 16, zigzag-coded IN PLACE over the samples,
//                   sum |r|.  The fixed predictor is only evaluated (second pass, samples re-fetched by TMA)
//                   when the LPC residual does not fit or when the analysis pass's exact sum |e| says the fixed
//                   subframe is smaller, both compared as single-partition estimates.
//   estimate        Rice parameter and estimated bits of the finest partitions by shuffles inside the
//                   2^(7 - max_porder) threads that share one; partition order = the level's maximum or 0.
//   lengths + scan  exact code lengths of the chunk -> warp / block exclusive scan (barrier B5)
//   pack            right-aligned 64-bit accumulator in two registers, one predicated store per completed
//                   word; the trailing partial word is OR-ed in when the frame is retired.
// Three barriers per (frame, channel): top of the CTA loop, partials (B3), scan (B5).  The previous frame is
// copied to its slot between B3 and B5 while thread 0 builds this channel's header.
// ------------------------------------------------------------------------------------------------------
FA_D uint32_t zigzag32(int32_t r) { return ((uint32_t)r << 1) ^ (uint32_t)(r >> 31); }

// Residuals of the thread's 32 samples for a predictor of at most NC coefficients (coef[m] = 0 beyond the
// order; a fixed predictor is passed as its literal coefficients with shift 0).  buf: the channel's samples,
// replaced by the zigzag-coded residuals.  WIDE: 64-bit accumulation, and residuals that do not fit the Rice
// coder clear `fit_out`.  Thread 0's first `order` samples are warm-up: left out of the sum and of the check.
template <int NC, bool WIDE>
FA_D void residual_pass(int32_t* buf, EncHot* hot, const int32_t* park, int t, int wasted, const int32_t* coef, int shift,
                        int order, unsigned long long& sum_out, bool& fit_out) {
    int32_t w[NC + 16];
    if (t == 0) {
#pragma unroll
        for (int i = 0; i < NC; ++i) w[i] = 0;
    } else {
        // the NC samples before the chunk = the last quads of thread t - 1 (L2 hits: the TMA copy has just read them)
#pragma unroll
        for (int qq = 0; qq < NC / 4; ++qq) {
            const U4 v = ldg128(park + (((8 - NC / 4 + qq) * kEncThreads + (t - 1)) << 2));
            w[4 * qq] = (int32_t)v.x; w[4 * qq + 1] = (int32_t)v.y; w[4 * qq + 2] = (int32_t)v.z; w[4 * qq + 3] = (int32_t)v.w;
        }
        if (wasted) {
#pragma unroll
            for (int i = 0; i < NC; ++i) w[i] >>= wasted;
        }
    }
    uint32_t a = 0;
    unsigned long long b = 0;
    uint32_t bad = 0;
#pragma unroll 1
    for (int h = 0; h < 2; ++h) {
        int32_t* p = buf + ((h * 4 * kEncThreads + t) << 2);
#pragma unroll
        for (int qq = 0; qq < 4; ++qq) {
            const U4 v = lds128(p + qq * (kEncThreads * 4));
            w[NC + 4 * qq] = (int32_t)v.x; w[NC + 4 * qq + 1] = (int32_t)v.y;
            w[NC + 4 * qq + 2] = (int32_t)v.z; w[NC + 4 * qq + 3] = (int32_t)v.w;
        }
        if (wasted) {
#pragma unroll
            for (int i = 0; i < 16; ++i) w[NC + i] >>= wasted;
        }
        if (h == 0 && t == 0) {
#pragma unroll
            for (int qq = 0; qq < kMaxOrd / 4; ++qq) {
                U4 v;
                v.x = (uint32_t)w[NC + 4 * qq]; v.y = (uint32_t)w[NC + 4 * qq + 1];
                v.z = (uint32_t)w[NC + 4 * qq + 2]; v.w = (uint32_t)w[NC + 4 * qq + 3];
                sts128(&hot->warm[4 * qq], v);
            }
        }
        uint32_t u[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            if (!WIDE) {
                int32_t sum = 0;
#pragma unroll
                for (int m = 0; m < NC; ++m) sum += coef[m] * w[NC + i - 1 - m];
                const int32_t r = w[NC + i] - (sum >> shift);
                a = sad_acc(r, 0, a);
                u[i] = zigzag32(r);
            } else {
                int64_t sum = 0;
#pragma unroll
                for (int m = 0; m < NC; ++m) sum += (int64_t)coef[m] * (int64_t)w[NC + i - 1 - m];
                const int64_t v = (int64_t)w[NC + i] - (sum >> shift);
                if (!fits_res(v)) bad |= 1u << i;
                const int32_t r = (int32_t)v;
                u[i] = zigzag32(r);
                b += ((unsigned long long)u[i] + 1ull) >> 1;     // |r|
            }
        }
        if (h == 0 && t == 0) {
#pragma unroll
            for (int i = 0; i < NC; ++i) {
                if (i < order) {
                    const unsigned long long ar = ((unsigned long long)u[i] + 1ull) >> 1;
                    if (WIDE) b -= ar; else a -= (uint32_t)ar;
                    bad &= ~(1u << i);
                }
            }
        }
#pragma unroll
        for (int qq = 0; qq < 4; ++qq) {
            U4 v;
            v.x = u[4 * qq]; v.y = u[4 * qq + 1]; v.z = u[4 * qq + 2]; v.w = u[4 * qq + 3];
            sts128(p + qq * (kEncThreads * 4), v);
        }
#pragma unroll
        for (int i = 0; i < NC; ++i) w[i] = w[16 + i];
    }
    sum_out = WIDE ? b : (unsigned long long)a;
    fit_out = bad == 0;
}

template <int H, bool WIDE>
FA_D void residual_dispatch(int32_t* buf, EncHot* hot, const int32_t* park, int t, int wasted, const int32_t* coef, int shift,
                            int order, unsigned long long& sum_out, bool& fit_out) {
    if (order <= 4) residual_pass<4, WIDE>(buf, hot, park, t, wasted, coef, shift, order, sum_out, fit_out);
    else if (H <= 8 || order <= 8) residual_pass<8, WIDE>(buf, hot, park, t, wasted, coef, shift, order, sum_out, fit_out);
    else residual_pass<H, WIDE>(buf, hot, park, t, wasted, coef, shift, order, sum_out, fit_out);
}

#if defined(FAB_PHASE_TIMING) && defined(__CUDACC__)
#define FAB_TICK(k) do { long long now_ = clock64(); X.ph[k] += now_ - X.last; X.last = now_; } while (0)
#else
#define FAB_TICK(k) do { } while (0)
#endif

// park: the channel's parked samples in HBM (16-byte aligned)
template <int H>
FA_D bool enc_channel_full(const EncParams& P, EncCtx& X, const int32_t* park, int c, int f, uint32_t g, int bitpos0,
                           int& bitpos_end, int slot) {
    EncHot* hot = X.hot;
    uint32_t* out = X.out;
    int32_t* res = X.res;
    const int t = tid();
    const int ln = lane(), wp = warp();
    constexpr int bs = kMaxBs;
    // ---- the channel's samples: one TMA copy into the sample buffer.  Every thread is done with the buffer's
    //      previous contents: channel 0 starts behind the barrier at the top of the CTA loop
    //      (channel 0's copy was started by the caller, ahead of the copy-out of the previous frame)
    if (c > 0) {
        sync();
        if (t == 0) {
            fence_proxy_async();
            bulk_load(res, park, (uint32_t)(kMaxBs * 4), &hot->mbar);
        }
    }
    // ---- the plan of this (frame, channel): prefetched into shared memory one frame ahead, decoded in registers
    const U4 pa = lds128(&hot->pf_plan[slot][c][0]), pb = lds128(&hot->pf_plan[slot][c][1]), pc = lds128(&hot->pf_plan[slot][c][2]);
    const int mode = (int)(pa.x & 0xFFu);
    const int wasted = (int)((pa.x >> 8) & 0xFFu);
    const int bps = 32 - wasted;
    const int ok0 = (int)((pa.x >> 16) & 0xFFu), ok1 = (int)(pa.x >> 24);
    const int ord0 = (int)(pa.y & 0xFFu), ord1 = (int)((pa.y >> 8) & 0xFFu);
    const int shift1 = (int)((pa.y >> 16) & 0xFFu), prec1 = (int)(pa.y >> 24);
    const bool wide = mode == 3;
    const bool wide1 = wide || (pa.z & 0xFFu) != 0;
    const uint32_t fixed_bits = pc.z;
    FAB_TICK(1);
    mbar_wait(&hot->mbar, X.tma_phase);
    X.tma_phase ^= 1u;
    FAB_TICK(2);
    if (mode == 0) return false;     // (the copy has landed: the general path may reuse the buffer)

    if (mode == 1) {
        // the other paths pass a barrier before they write `out`; this one must too: the previous frame may still be
        // copied out of `out` (top of the CTA loop), and thread 0 overwrites prev_g / prev_nbytes behind this frame
        if (c == 0) sync();
        bitpos_end = bitpos0 + (c == 0 ? 8 * frame_header_bytes(bs, f) : 0) + subframe_header_bits(0, 0, 0, 32, 0);
        if (t == 0) {
            Pk pk;
            pk_begin(pk, out, bitpos0);
            if (c == 0) emit_frame_header(pk, hot->crc8, bs, f, P.nch);
            emit_subframe_header(pk, 0, 0, 0);
            emit_sample(pk, res[0], 32);
            pk_end(pk, hot->tail_val[c][0], hot->tail_word[c][0]);
        }
        return true;
    }
    int32_t coef1[H];
    {
        const uint32_t qw[6] = {pb.x, pb.y, pb.z, pb.w, pc.x, pc.y};
#pragma unroll
        for (int m = 0; m < H; ++m) coef1[m] = (int32_t)(int16_t)(uint16_t)(qw[m >> 1] >> (16 * (m & 1)));
    }

    // ---- residual pass + estimate, for the LPC candidate first; the fixed predictor only on demand
    const int maxp = P.max_porder;
    const int gsh = 7 - maxp;
    const int part = t >> gsh;
    const bool leader = (t & ((1 << gsh) - 1)) == 0;
    const uint32_t verbatim_bits = (uint32_t)bps * (uint32_t)bs;
    int cand = ok1 ? 1 : (ok0 ? 0 : -1);
    if (cand < 0) return false;
    int order = 0, porder = 0, k = 0, rice2 = 0;
    int32_t cf[H];
    for (int pass = 0;; ++pass) {
        order = cand ? ord1 : ord0;
        const int shift = cand ? shift1 : 0;
        if (cand) {
#pragma unroll
            for (int m = 0; m < H; ++m) cf[m] = coef1[m];
        } else {
            fixed_coefs(ord0, cf, H);
        }
        unsigned long long s = 0;
        bool fit = true;
        if (cand ? wide1 : wide) residual_dispatch<H, true>(res, hot, park, t, wasted, cf, shift, order, s, fit);
        else residual_dispatch<H, false>(res, hot, park, t, wasted, cf, shift, order, s, fit);
        FAB_TICK(3);
        // finest partitions: 2^gsh consecutive threads each; parameters and estimated bits computed redundantly by
        // every thread of the group
        unsigned long long gs = s;
        for (int m = 1; m < (1 << gsh); m <<= 1) gs += shfl_xor64(gs, m);
        const uint32_t npart = (uint32_t)(bs >> maxp) - (part == 0 ? (uint32_t)order : 0u);
        int kf = 0;
        const uint32_t e = rice_estimate(gs, npart, kf);
        {
            const uint32_t bsum = redux_add(leader ? e : 0u);
            const unsigned long long ts = warp_sum_u64(s);
            const uint32_t fl = (ballot(!fit) ? 1u : 0u) | (ballot(kf >= 15) ? 2u : 0u);
            if (ln == 0) { hot->x_bits[pass & 1][wp] = bsum; hot->x_sum[pass & 1][wp] = ts; hot->x_flag[pass & 1][wp] = fl; }
        }
        FAB_TICK(4);
        sync();   // B3: the partials are visible
        FAB_TICK(5);
        // every thread: partition order (maximum or 0) and size of the subframe; all inputs are block-uniform
        uint32_t bits_hi = 0, flag = 0;
        unsigned long long tot = 0;
#pragma unroll
        for (int w = 0; w < kEncWarps; ++w) { bits_hi += hot->x_bits[pass & 1][w]; tot += hot->x_sum[pass & 1][w]; flag |= hot->x_flag[pass & 1][w]; }
        int k0 = 0;
        uint32_t bits_lo = rice_estimate(tot, (uint32_t)(bs - order), k0);
        bits_lo += 6u + (k0 >= 15 ? 1u : 0u);
        bits_hi += 6u + ((flag & 2u) ? (1u << maxp) : 0u);
        const bool use_hi = bits_hi < bits_lo;
        const uint32_t side = (uint32_t)order * (uint32_t)bps + (cand ? 9u + (uint32_t)order * (uint32_t)prec1 : 0u);
        const bool unfit = (flag & 1u) != 0;
        if (cand == 1 && ok0 && (unfit || fixed_bits < side + bits_lo)) {
            // the fixed predictor looks smaller (or the LPC residual does not fit): fetch the samples again and redo
            cand = 0;
            if (t == 0) {
                fence_proxy_async();
                bulk_load(res, park, (uint32_t)(kMaxBs * 4), &hot->mbar);
            }
            mbar_wait(&hot->mbar, X.tma_phase);
            X.tma_phase ^= 1u;
            continue;
        }
        if (unfit || side + (use_hi ? bits_hi : bits_lo) >= verbatim_bits) return false;   // (block-uniform) general path
        porder = use_hi ? maxp : 0;
        k = use_hi ? kf : k0;
        rice2 = use_hi ? ((flag & 2u) ? 1 : 0) : (k0 >= 15 ? 1 : 0);
        break;
    }
    const int plen = rice2 ? 5 : 4;
    const int skip = t == 0 ? order : 0;
    const int ptype = cand == 0 ? 2 : 3;
    const int prec = cand == 0 ? 0 : prec1;
    // ---- this channel's header: the bit string k_enc_design prepared (every thread fetches "its" word of it now and
    //      stores it behind B5); without one, thread 0 emits the fields into hdr_tmp
    const PlanHeader* ph = P.hdrs + ((size_t)(g - P.g_begin) * P.nch + c);
    const uint32_t hn = P.hdrs != nullptr ? (cand ? hot->pf_hdr[slot][c].x : hot->pf_hdr[slot][c].y) : 0u;     // (block-uniform)
    const bool pre = hn != 0;
    const uint32_t* hwords = cand ? ph->lpc : ph->fix;
    const uint32_t hs = (uint32_t)bitpos0 & 31u;
    const int hfull = (int)((hs + hn) >> 5);          // frame words that are complete once the header is in
    uint32_t hval = 0;
    if (pre && t < hfull) {
        const uint32_t b = ldg32(hwords + t), a = t > 0 ? ldg32(hwords + t - 1) : 0u;
        hval = hs ? funnel_r(b, a, hs) : b;
    }
    Pk pk;
    int hdr_words = 0;
    if (t == 0 && !pre) {
        // same accumulator protocol as Pk, words go to hdr_tmp[0 ..); bit offset of the first word kept
        pk_begin(pk, hot->hdr_tmp, bitpos0 & 31);          // word index 0 = frame word (bitpos0 >> 5)
        if (c == 0) emit_frame_header(pk, hot->crc8, bs, f, P.nch);
        emit_subframe_header(pk, ptype, order, wasted);
        for (int j = 0; j < order; ++j) emit_sample(pk, hot->warm[j], bps);
        if (ptype == 3) {
            pk_emit(pk, (uint32_t)(prec1 - 1), 4);
            pk_emit(pk, (uint32_t)shift1 & 31u, 5);
            for (int j = 0; j < order; ++j) {
                int32_t cj = cf[0];
#pragma unroll
                for (int q = 1; q < H; ++q) cj = (q == j) ? cf[q] : cj;
                pk_emit(pk, (uint32_t)cj & ((1u << prec1) - 1u), prec1);
            }
        }
        pk_emit(pk, (uint32_t)rice2, 2);
        pk_emit(pk, (uint32_t)porder, 4);
        hdr_words = pk.word;
    }
    FAB_TICK(6);
    // ---- exact code lengths of the chunk, block scan
    const bool part_start = porder == 0 ? t == 0 : leader;
    uint32_t lens = part_start ? (uint32_t)plen : 0u;
    uint32_t qor = 0;
    const int32_t* rp = res + (t << 2);
#pragma unroll
    for (int q = 0; q < kSpt / 4; ++q) {
        const U4 v = lds128(rp + q * (kEncThreads * 4));
        uint32_t q0 = v.x >> k, q1 = v.y >> k, q2 = v.z >> k, q3 = v.w >> k;
        if (4 * q < H) {      // only the first quads can hold warm-up samples
            q0 = 4 * q + 0 < skip ? 0u : q0; q1 = 4 * q + 1 < skip ? 0u : q1;
            q2 = 4 * q + 2 < skip ? 0u : q2; q3 = 4 * q + 3 < skip ? 0u : q3;
        }
        lens += (q0 + q1) + (q2 + q3);
        qor |= (q0 | q1) | (q2 | q3);
    }
    lens += (uint32_t)(kSpt - skip) * (uint32_t)(k + 1);
    uint32_t inc = lens;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t n = shfl_up(inc, d);
        if (ln >= d) inc += n;
    }
    if (ln == 31) hot->scan[wp] = inc;
    FAB_TICK(7);
    sync();   // B5
    FAB_TICK(8);
    uint32_t wbase = 0, total = 0;
#pragma unroll
    for (int w = 0; w < kEncWarps; ++w) {
        uint32_t x = hot->scan[w];
        if (w < wp) wbase += x;
        total += x;
    }
    const uint32_t excl = wbase + inc - lens;
    const int hdr_bits = subframe_header_bits(ptype, order, wasted, bps, prec);
    if ((uint32_t)hdr_bits + total >= verbatim_bits + 8u) return false;   // VERBATIM is smaller: general path
    const int sub0 = bitpos0 + (c == 0 ? 8 * frame_header_bytes(bs, f) : 0);
    const int body0 = sub0 + hdr_bits;

    // ---- pack: the pending bits sit right-aligned in `lo` (fill < 32 of them between codes; older bits above
    //      them are stale and never read again)
    bitpos_end = body0 + (int)total;
    uint32_t lo = 0, hi = 0;
    int fill, word;
    if (pre) {
        if (t < hfull) out[ow((bitpos0 >> 5) + t)] = hval;
    }
    if (t == 0 && pre) {
        // the header bits behind the last complete word, then the residual coding method and partition order
        fill = (int)((hs + hn) & 31u);
        word = (bitpos0 >> 5) + hfull;
        if (fill) {
            const int kw = (int)((hn - 1u) >> 5), r = (int)((hn - 1u) & 31u) + 1;     // last header word, bits used in it
            const uint64_t x = (((uint64_t)(kw > 0 ? ldg32(hwords + kw - 1) : 0u) << 32) | ldg32(hwords + kw)) >> (32 - r);
            lo = (uint32_t)x & ((1u << fill) - 1u);
        }
        hi = funnel_lc(lo, hi, 6u);
        lo = (lo << 6) | ((uint32_t)rice2 << 4) | (uint32_t)porder;
        fill += 6;
        if (fill >= 32) { fill -= 32; out[ow(word)] = funnel_r(lo, hi, (uint32_t)fill); word++; }
    } else if (t == 0) {
        // move the finished header words into the staged frame and continue the same bit stream there
        const int w0 = bitpos0 >> 5;
        for (int i = 0; i < hdr_words; ++i) out[ow(w0 + i)] = hot->hdr_tmp[ow(i)];
        fill = pk.fill;
        word = w0 + hdr_words;
        lo = fill ? (uint32_t)(pk.acc >> (64 - fill)) : 0u;
    } else {
        const int pos = body0 + (int)excl;
        fill = pos & 31;
        word = pos >> 5;
    }
    if (part_start) {
        hi = funnel_lc(lo, hi, (uint32_t)plen);
        lo = (lo << plen) | (uint32_t)k;
        fill += plen;
        if (fill >= 32) { fill -= 32; out[ow(word)] = funnel_r(lo, hi, (uint32_t)fill); word++; }
    }
    if (qor + (uint32_t)k + 1u <= 32u) {
        // every code of the chunk fits 32 bits: branch-free appends
        const uint32_t kbit = 1u << k, kmask = kbit - 1u;
        const uint32_t k1 = (uint32_t)k + 1u;
        // (a code of length 0 and value 0 is a no-op: that is how thread 0 passes over its warm-up samples)
#define FAB_APPEND_M(uv, msk)                                                          \
        do {                                                                           \
            const uint32_t u_ = (uv);                                                  \
            const uint32_t len_ = ((u_ >> k) + k1) & (msk);                            \
            hi = funnel_lc(lo, hi, len_);                                              \
            lo = funnel_lc(0u, lo, len_) | (((u_ & kmask) | kbit) & (msk));            \
            fill += (int)len_;                                                         \
            if (fill >= 32) { fill -= 32; out[ow(word)] = funnel_r(lo, hi, (uint32_t)fill); word++; } \
        } while (0)
#define FAB_APPEND(uv) FAB_APPEND_M(uv, 0xFFFFFFFFu)
#pragma unroll
        for (int q = 0; q < H / 4; ++q) {       // quads that may hold warm-up samples (thread 0)
            const U4 v = lds128(rp + q * (kEncThreads * 4));
            FAB_APPEND_M(v.x, 4 * q + 0 >= skip ? 0xFFFFFFFFu : 0u);
            FAB_APPEND_M(v.y, 4 * q + 1 >= skip ? 0xFFFFFFFFu : 0u);
            FAB_APPEND_M(v.z, 4 * q + 2 >= skip ? 0xFFFFFFFFu : 0u);
            FAB_APPEND_M(v.w, 4 * q + 3 >= skip ? 0xFFFFFFFFu : 0u);
        }
#pragma unroll 2
        for (int q = H / 4; q < kSpt / 4; ++q) {
            const U4 v = lds128(rp + q * (kEncThreads * 4));
            FAB_APPEND(v.x);
            FAB_APPEND(v.y);
            FAB_APPEND(v.z);
            FAB_APPEND(v.w);
        }
#undef FAB_APPEND
#undef FAB_APPEND_M
        hot->tail_val[c][t] = fill ? (lo << (32 - fill)) : 0u;
        hot->tail_word[c][t] = (uint16_t)word;
    } else {
        Pk pq;
        pq.out = out;
        pq.acc = fill ? ((uint64_t)lo << (64 - fill)) : 0ull;
        pq.fill = fill;
        pq.word = word;
#pragma unroll 1
        for (int j = skip; j < kSpt; ++j) pk_rice(pq, (uint32_t)res[(((j >> 2) * kEncThreads + t) << 2) + (j & 3)], k);
        pk_end(pq, hot->tail_val[c][t], hot->tail_word[c][t]);
    }
    FAB_TICK(9);
    return true;
}

// ------------------------------------------------------------------------------------------------------
// General path: any blocksize <= 4096, any sample width, wasted bits, CONSTANT / VERBATIM / FIXED / LPC.
// ------------------------------------------------------------------------------------------------------
struct GenChunk {                 // thread-local copy of the chunk (local memory: this path is not tuned)
    int32_t x[kMaxOrd + kSpt];    // x[kMaxOrd + j] = sample (32 t + j) >> wasted; history before it
};

FA_D int64_t gen_residual(const GenChunk& G, int j, int order, const int32_t* coef, int shift) {
    int64_t sum = 0;
    for (int m = 0; m < order; ++m) sum += (int64_t)coef[m] * (int64_t)G.x[kMaxOrd + j - 1 - m];
    return (int64_t)G.x[kMaxOrd + j] - (sum >> shift);
}

FA_D void enc_channel_general_body(const EncParams& P, EncCtx& X, const FrameSrc& S, int c, int f, uint32_t g, int bitpos0,
                                   int& bitpos_end) {
    EncShared* sh = X.sh;
    uint32_t* out = X.out;
    retire_full(P, X);
    const int t = tid();
    const int ln = lane(), wp = warp();
    const int bs = S.bs;
    const int i0 = t * kSpt;
    const int nmine = i0 >= bs ? 0 : (bs - i0 < kSpt ? bs - i0 : kSpt);
    GenChunk G;
    for (int j = 0; j < kMaxOrd + kSpt; ++j) {
        int i = i0 - kMaxOrd + j;
        G.x[j] = (i >= 0 && i < bs) ? src_sample(S, c, i) : 0;
    }
    // ---- statistics
    {
        uint32_t orv = 0;
        int32_t mn = 0x7fffffff, mx = (int32_t)0x80000000u;
        for (int j = 0; j < nmine; ++j) {
            int32_t v = G.x[kMaxOrd + j];
            orv |= (uint32_t)v;
            mn = v < mn ? v : mn;
            mx = v > mx ? v : mx;
        }
        uint32_t wor = redux_or(orv);
        int32_t wmn = redux_min(mn), wmx = redux_max(mx);
        if (ln == 0) { sh->w_or[wp] = wor; sh->w_mn[wp] = wmn; sh->w_mx[wp] = wmx; }
    }
    sync();
    uint32_t t_or = 0;
    int32_t t_mn = 0x7fffffff, t_mx = (int32_t)0x80000000u;
    for (int w = 0; w < kEncWarps; ++w) {
        t_or |= sh->w_or[w];
        t_mn = sh->w_mn[w] < t_mn ? sh->w_mn[w] : t_mn;
        t_mx = sh->w_mx[w] > t_mx ? sh->w_mx[w] : t_mx;
    }
    const int wasted = t_or == 0 ? 0 : ctz32(t_or);
    const int bps = 32 - wasted;
    const bool constant = t_mn == t_mx;
    if (wasted)
        for (int j = 0; j < kMaxOrd + kSpt; ++j) G.x[j] >>= wasted;
    const int sub0 = bitpos0 + (c == 0 ? 8 * frame_header_bytes(bs, f) : 0);
    const uint32_t verbatim_bits = (uint32_t)bps * (uint32_t)bs;
    const bool try_pred = !constant && bs > 4;

    int ptype = constant ? 0 : 1;
    int win = -1;
    if (try_pred) {
        // ---- fixed-predictor error sums (64-bit) and windowed autocorrelation
        unsigned long long fe[5] = {0, 0, 0, 0, 0};
        uint32_t bad = 0;
        for (int j = 0; j < nmine; ++j) {
            if (i0 + j < 4) continue;
            int64_t a0 = G.x[kMaxOrd + j], a1 = G.x[kMaxOrd + j - 1], a2 = G.x[kMaxOrd + j - 2], a3 = G.x[kMaxOrd + j - 3],
                    a4 = G.x[kMaxOrd + j - 4];
            int64_t e[5];
            e[0] = a0; e[1] = a0 - a1; e[2] = e[1] - (a1 - a2); e[3] = e[2] - (a1 - 2 * a2 + a3);
            e[4] = e[3] - (a1 - 3 * a2 + 3 * a3 - a4);
            for (int k = 0; k < 5; ++k) {
                if (!fits_res(e[k])) bad |= 1u << k;
                fe[k] += (unsigned long long)(e[k] < 0 ? -e[k] : e[k]);
            }
        }
        int max_order = P.max_lpc_order;
        if (max_order >= bs) max_order = bs - 1;
        double ac[kMaxOrd + 1];
        for (int l = 0; l <= kMaxOrd; ++l) ac[l] = 0.0;
        if (max_order > 0) {
            for (int j = 0; j < nmine; ++j) {
                double w0 = (double)fmul((float)G.x[kMaxOrd + j], P.window[i0 + j]);
                for (int l = 0; l <= max_order; ++l) {
                    int i = i0 + j - l;
                    if (i < 0) break;
                    double wl = (double)fmul((float)G.x[kMaxOrd + j - l], P.window[i]);
                    ac[l] = dfma(w0, wl, ac[l]);
                }
            }
        }
        uint32_t wbad = redux_or(bad);
        for (int k = 0; k < 5; ++k) {
            unsigned long long v = warp_sum_u64(fe[k]);
            if (ln == 0) sh->w_fe[wp][k] = v;
        }
        for (int l = 0; l <= max_order; ++l) {
            double v = warp_sum_d(ac[l]);
            if (ln == 0) sh->w_ac[wp][l] = v;
        }
        if (ln == 0) sh->w_bad[wp] = wbad;
        sync();
        if (t == 0) {
            uint32_t tb = 0;
            for (int w = 0; w < kEncWarps; ++w) tb |= sh->w_bad[w];
            for (int k = 0; k < 5; ++k) {
                unsigned long long v = 0;
                for (int w = 0; w < kEncWarps; ++w) v += sh->w_fe[w][k];
                sh->t_fe[k] = v;
            }
            for (int l = 0; l <= max_order; ++l)
                sh->t_ac[l] = dadd(dadd(sh->w_ac[0][l], sh->w_ac[1][l]), dadd(sh->w_ac[2][l], sh->w_ac[3][l]));
            design_fixed(sh, bs, bps, tb, P.max_porder);
            design_lpc(sh, bs, bps, max_order, P.qlp_precision, P.max_porder, 0u);
        }
        if (t < 2 * kMaxParts) ((unsigned long long*)sh->psum)[t] = 0;
        sync();
        // ---- residual partition sums (shared atomics at partition boundaries only)
        uint32_t resbad = 0;
        for (int cd = 0; cd < 2; ++cd) {
            if (!sh->cand_ok[cd]) continue;   // block-uniform
            const Plan& pl = sh->cand[cd];
            int32_t coef[kMaxOrd];
            if (cd == 0) fixed_coefs(pl.order, coef, kMaxOrd);
            else for (int m = 0; m < kMaxOrd; ++m) coef[m] = pl.qlp[m];
            const int psize = bs >> sh->maxp[cd];
            int j = i0 < pl.order ? pl.order - i0 : 0;
            if (j < nmine) {
                int part = (i0 + j) / psize;
                int next = (part + 1) * psize;
                unsigned long long acc = 0;
                for (; j < nmine; ++j) {
                    if (i0 + j == next) {
                        atom_add_shared64(&sh->psum[cd][part], acc);
                        acc = 0;
                        part++;
                        next += psize;
                    }
                    int64_t rv = gen_residual(G, j, pl.order, coef, pl.shift);
                    if (!fits_res(rv)) resbad |= 1u << cd;
                    acc += (unsigned long long)(rv < 0 ? -rv : rv);
                }
                atom_add_shared64(&sh->psum[cd][part], acc);
            }
        }
        resbad = redux_or(resbad);
        if (ln == 0) sh->w_bad[wp] = resbad;
        sync();
        resbad = sh->w_bad[0] | sh->w_bad[1] | sh->w_bad[2] | sh->w_bad[3];
        if (wp < 2 && sh->cand_ok[wp] && !((resbad >> wp) & 1))
            rice_search_warp(sh, wp, bs, sh->cand[wp].order, sh->maxp[wp]);
        sync();
        {
            uint32_t best = verbatim_bits;
            for (int cd = 0; cd < 2; ++cd) {
                if (!sh->cand_ok[cd] || ((resbad >> cd) & 1)) continue;
                const Plan& pl = sh->cand[cd];
                uint32_t bits = (uint32_t)pl.order * (uint32_t)bps + pl.res_bits +
                                (cd == 1 ? 9u + (uint32_t)pl.order * (uint32_t)pl.prec : 0u);
                if (bits < best) { best = bits; win = cd; }
            }
        }
        if (win >= 0) ptype = win == 0 ? 2 : 3;
    }

    // ---- exact size of the predictive subframe; fall back to VERBATIM if it does not pay
    int order = 0, porder = 0, plen = 4, shift = 0, prec = 0;
    int32_t coef[kMaxOrd];
    for (int m = 0; m < kMaxOrd; ++m) coef[m] = 0;
    uint32_t lens = 0;
    if (ptype >= 2) {
        const Plan& pl = sh->cand[win];
        order = pl.order; porder = pl.porder; plen = pl.rice2 ? 5 : 4; shift = pl.shift; prec = pl.prec;
        if (win == 0) fixed_coefs(order, coef, kMaxOrd);
        else for (int m = 0; m < kMaxOrd; ++m) coef[m] = pl.qlp[m];
        const int psize = bs >> porder;
        const uint8_t* kp = &sh->kpar[win][(1 << porder) - 1];
        int j = i0 < order ? order - i0 : 0;
        if (j < nmine) {
            int part = (i0 + j) / psize;
            int next = (part + 1) * psize;
            int k = kp[part];
            if (i0 + j == (part == 0 ? order : part * psize)) lens += (uint32_t)plen;
            for (; j < nmine; ++j) {
                if (i0 + j == next) { part++; next += psize; k = kp[part]; lens += (uint32_t)plen; }
                int64_t rv = gen_residual(G, j, order, coef, shift);
                uint32_t u = ((uint32_t)rv << 1) ^ (uint32_t)(rv >> 63);
                lens += (u >> k) + 1u + (uint32_t)k;
            }
        }
    }
    uint32_t inc = lens;
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t n = shfl_up(inc, d);
        if (ln >= d) inc += n;
    }
    if (ln == 31) sh->scan[wp] = inc;
    sync();
    uint32_t wbase = 0, total = 0;
    for (int w = 0; w < kEncWarps; ++w) {
        uint32_t x = sh->scan[w];
        if (w < wp) wbase += x;
        total += x;
    }
    const uint32_t excl = wbase + inc - lens;
    if (ptype >= 2 && (uint32_t)subframe_header_bits(ptype, order, 0, bps, prec) + total >= verbatim_bits + 8u) ptype = 1;
    const int hdr_bits = subframe_header_bits(ptype, order, wasted, bps, prec);
    const int body0 = sub0 + hdr_bits;   // for CONSTANT this already includes the value

    // ---- pack
    bitpos_end = ptype == 1 ? body0 + bs * bps : ptype >= 2 ? body0 + (int)total : body0;
    Pk pk;
    bool open = false;
    if (t == 0) {
        pk_begin(pk, out, bitpos0);
        open = true;
        if (c == 0) emit_frame_header(pk, X.hot->crc8, bs, f, P.nch);
        emit_subframe_header(pk, ptype, order, wasted);
        if (ptype == 0) {
            emit_sample(pk, G.x[kMaxOrd], bps);
        } else if (ptype >= 2) {
            for (int j = 0; j < order; ++j) emit_sample(pk, G.x[kMaxOrd + j], bps);
            if (ptype == 3) emit_lpc_params(pk, sh->cand[win]);
            pk_emit(pk, (uint32_t)sh->cand[win].rice2, 2);
            pk_emit(pk, (uint32_t)porder, 4);
        }
    }
    if (ptype == 1) {
        if (nmine > 0) {
            if (!open) { pk_begin(pk, out, body0 + i0 * bps); open = true; }
            for (int j = 0; j < nmine; ++j) emit_sample(pk, G.x[kMaxOrd + j], bps);
        }
    } else if (ptype >= 2) {
        const int psize = bs >> porder;
        const uint8_t* kp = &sh->kpar[win][(1 << porder) - 1];
        int j = i0 < order ? order - i0 : 0;
        if (j < nmine) {
            if (!open) { pk_begin(pk, out, body0 + (int)excl); open = true; }
            int part = (i0 + j) / psize;
            int next = (part + 1) * psize;
            int k = kp[part];
            if (i0 + j == (part == 0 ? order : part * psize)) pk_emit(pk, (uint32_t)k, plen);
            for (; j < nmine; ++j) {
                if (i0 + j == next) { part++; next += psize; k = kp[part]; pk_emit(pk, (uint32_t)k, plen); }
                int64_t rv = gen_residual(G, j, order, coef, shift);
                uint32_t u = ((uint32_t)rv << 1) ^ (uint32_t)(rv >> 63);
                pk_rice(pk, u, k);
            }
        }
    }
    if (open) pk_end(pk, X.hot->tail_val[c][t], X.hot->tail_word[c][t]);
}

FA_DNOINL int enc_channel_general(const EncParams P, EncCtx X, const FrameSrc S, int c, int f, uint32_t g, int bitpos0) {
    int bitpos_end = 0;
    enc_channel_general_body(P, X, S, c, f, g, bitpos0, bitpos_end);
    return bitpos_end;
}

// ------------------------------------------------------------------------------------------------------
// The CTA body: loops over (stream, frame) units.  `smem_raw` >= enc_smem_bytes(nch).
// ------------------------------------------------------------------------------------------------------
// Thread 0: take the next (stream, frame) ticket of the batch and do its index arithmetic one frame ahead.
FA_D void enc_fetch_ticket(const EncParams& P, EncHot* hot, int slot) {
    const uint32_t g = P.g_begin + atom_add_global(P.ticket, 1u);
    const int f = (int)(g % (uint32_t)P.nframes);
    const int64_t left = P.stream_size - (int64_t)f * P.blocksize;
    hot->gq[slot] = g;
    hot->gq_f[slot] = f;
    hot->gq_bs[slot] = (int)(left < P.blocksize ? left : P.blocksize);
}

FA_D void enc_set_ticket(const EncParams& P, EncHot* hot, int slot, uint64_t g64) {
    const uint32_t g = g64 < (uint64_t)P.g_end ? (uint32_t)g64 : P.g_end;
    const int f = (int)(g % (uint32_t)P.nframes);
    const int64_t left = P.stream_size - (int64_t)f * P.blocksize;
    hot->gq[slot] = g;
    hot->gq_f[slot] = f;
    hot->gq_bs[slot] = (int)(left < P.blocksize ? left : P.blocksize);
}

// Thread 0: the plans and the head of the prebuilt headers of the ticket in `slot` -> shared memory (cp.async: no register
// is waited for; completion is collected before the next top-of-loop barrier).
FA_D void enc_prefetch_plans(const EncParams& P, EncHot* hot, int slot) {
    const uint32_t g = hot->gq[slot];
    if (g < P.g_end) {
        for (int c = 0; c < P.nch; ++c) {
            const size_t r = (size_t)(g - P.g_begin) * P.nch + c;
            const unsigned char* pp = (const unsigned char*)(P.plans + r);
            cp_async16(&hot->pf_plan[slot][c][0], pp);
            cp_async16(&hot->pf_plan[slot][c][1], pp + 16);
            cp_async16(&hot->pf_plan[slot][c][2], pp + 32);
            if (P.hdrs != nullptr) cp_async16(&hot->pf_hdr[slot][c], P.hdrs + r);
        }
    }
    cp_async_commit();
}

// Where the samples of (stream, frame) unit g come from (short-frame and general paths; full frames read the
// integers k_enc_analyze parked).
FA_D FrameSrc enc_frame_src(const EncParams& P, uint32_t g, int f, int bs) {
    const int64_t s = (int64_t)(g / (uint32_t)P.nframes);
    FrameSrc S;
    S.dtype = P.dtype; S.bs = bs;
    S.off32 = 0.f; S.gain32 = 0.f; S.off64 = 0.; S.gain64 = 0.;
    if (P.dtype == kF32) { S.off32 = ((const float*)P.offsets)[s]; S.gain32 = ((const float*)P.gains)[s]; }
    if (P.dtype == kF64) { S.off64 = ((const double*)P.offsets)[s]; S.gain64 = ((const double*)P.gains)[s]; }
    const int esize = (P.dtype == kI32 || P.dtype == kF32) ? 4 : 8;
    S.base = (const unsigned char*)P.data + (s * P.stream_size + (int64_t)f * P.blocksize) * esize;
    S.vec = (((uintptr_t)S.base) & 15) == 0;
    return S;
}

// FULLK: the kernel of the full (4096-sample) frames -- persistent CTAs taking tickets over the whole batch and
// passing over the other frames; !FULLK: the kernel of those other frames (last frame of a stream, blocksize-1152
// levels), CTA i starting at frame `first + i * stride`.  Two kernels so that the register-hungry short path does
// not share a register budget (and an instruction cache) with the full-frame path.
template <int H, bool FULLK>
FA_D void encode_frames_cta(const EncParams& P, unsigned char* smem_raw, uint32_t first = 0, uint32_t stride = 1) {
    EncHot* hot = (EncHot*)smem_raw;
    const int t = tid();
    const int nch = P.nch;
    const uint32_t total_frames = P.g_end;
    EncCtx X;
    X.hot = hot;
    X.res = (int32_t*)(smem_raw + kEncHotBytes);       // 128-byte aligned: TMA destination
    X.sh = (EncShared*)X.res;
    X.out = (uint32_t*)(X.res + kMaxBs);
    X.out_words_padded = (int)(enc_out_words(nch) + (enc_out_words(nch) >> 4) + 8);
    X.retired = false;
    X.tma_phase = 0;
#if defined(FAB_PHASE_TIMING) && defined(__CUDACC__)
    for (int k = 0; k < 12; ++k) X.ph[k] = 0;
    X.last = clock64();
#endif

    for (int i = t; i < 256; i += kEncThreads) hot->crc8[i] = P.crc->crc8[i];
    uint64_t g_mine = (uint64_t)first + (uint64_t)blockIdx_x() * stride;      // (!FULLK)
    if (t == 0) {
        mbar_init(&hot->mbar, 1);
        hot->prev_valid2[0] = hot->prev_valid2[1] = 0;
        if (FULLK) { enc_fetch_ticket(P, hot, 0); enc_prefetch_plans(P, hot, 0); }
        else enc_set_ticket(P, hot, 0, g_mine);
    }
    hot->tail_val[0][t] = 0; hot->tail_val[1][t] = 0;

    // Per iteration: [top barrier] start the TMA copy of this frame's samples -> copy the previous frame (packed in
    // `out`) to its slot while that copy is in flight -> residuals, Rice parameters, packing -> [barrier] OR the
    // trailing partial words of the packing sessions into the staged frame.
    for (int iter = 0;; ++iter) {
        const int slot = iter & 1;
        // ---- work assignment: dynamic tickets (any order: every frame has its own output slot)
        FAB_TICK(10);
        if (FULLK && t == 0) cp_async_wait_all();      // this frame's plans (prefetched during the previous iteration)
        sync();   // the previous frame is complete in `out` (packing + tail ORs); nobody reads the sample buffer any more
        FAB_TICK(0);
        const uint32_t g = hot->gq[slot];
        const int f = hot->gq_f[slot], bs = hot->gq_bs[slot];
        const bool mine = g < total_frames && ((bs == kMaxBs) == FULLK) && !(!FULLK && fixed_done(P, g));
        if (FULLK) {
            if (t == 0) {
                if (mine) {
                    fence_proxy_async();
                    bulk_load(X.res, P.slots + (int64_t)(g - P.g_begin) * P.slot_bytes, (uint32_t)(kMaxBs * 4), &hot->mbar);
                }
                enc_fetch_ticket(P, hot, slot ^ 1);     // for the next iteration
                enc_prefetch_plans(P, hot, slot ^ 1);
            }
        } else {
            g_mine += (uint64_t)gridDim_x() * stride;
            if (t == 0) enc_set_ticket(P, hot, slot ^ 1, g_mine);
        }
        if (hot->prev_valid2[slot]) retire_copyout(P, X);
        if (t == 0) hot->prev_valid2[slot ^ 1] = 0;    // (last read one top barrier ago)
        X.retired = true;
        if (g >= total_frames) break;
        if (!mine) continue;      // the other kernel's frame

        int bitpos = 0;
        for (int c = 0; c < nch; ++c) {
            int bend = 0;
            bool done = false;
            if constexpr (FULLK) {
                // planar int32 samples parked by k_enc_analyze in this frame's slot (the compressed frame only
                // replaces them when the frame is retired, one iteration from now)
                const int32_t* park = (const int32_t*)(P.slots + (int64_t)(g - P.g_begin) * P.slot_bytes) + (int64_t)c * kMaxBs;
                done = enc_channel_full<H>(P, X, park, c, f, g, bitpos, bend, slot);
            } else if (bs >= 64) {
                bend = enc_channel_short<H>(P, X, enc_frame_src(P, g, f, bs), c, f, g, bitpos);
                done = bend >= 0;
            }
            if (!done) bend = enc_channel_general(P, X, enc_frame_src(P, g, f, bs), c, f, g, bitpos);
            bitpos = bend;
        }
        // the frame now waits in `out`; it is copied to its slot at the top of the next iteration
        if (t == 0) {
            if (bitpos & 31) X.out[ow(bitpos >> 5)] = 0;   // final partial word: nobody plain-stores it, tails are OR-ed in
            hot->prev_valid2[slot ^ 1] = 1; hot->prev_g = g; hot->prev_nbytes = (bitpos + 7) >> 3;
        }
        sync();   // B6: every plain store of the packing sessions (and the word zeroed above) is in place
        // trailing partial words of the packing sessions
        for (int c = 0; c < nch; ++c) {
            uint32_t tv = hot->tail_val[c][t];
            if (tv) { atom_or_shared(&X.out[ow(hot->tail_word[c][t])], tv); hot->tail_val[c][t] = 0; }
        }
    }
#if defined(FAB_PHASE_TIMING) && defined(__CUDACC__)
    if ((blockIdx.x == 7 || blockIdx.x == 300) && (t == 0 || t == 37 || t == 127 || t == 96))
        printf("cta %d t %d: top %lld | plan %lld tma %lld resid %lld est %lld B3 %lld hdr/copy %lld lens %lld B5 %lld pack %lld rest %lld\n",
               (int)blockIdx.x, t, X.ph[0], X.ph[1], X.ph[2], X.ph[3], X.ph[4], X.ph[5], X.ph[6], X.ph[7], X.ph[8], X.ph[9], X.ph[10]);
#endif
}

}  // namespace fa
