// fa_encode_fixed.h -- the encoder of libFLAC's levels 0..2 (blocksize 1152, FIXED predictors only, Rice partition
// order <= 3): one WARP per frame.
//
// The reference treats every level alike (compress.c:185: FLAC__stream_encoder_set_compression_level); at these
// levels libFLAC never designs an LPC predictor, so a frame needs no autocorrelation, no design stage and no second
// pass: the warp stages the frame's 1152 samples (quantising float input on the way, utils.c:160-243), every lane
// takes 36 consecutive samples into registers, the five fixed-predictor error sums pick the order (libFLAC fixed.c),
// the Rice parameters of partition orders 3..0 come from warp-segment sums (1152 >> 3 = 144 samples = 4 lanes), and
// the lanes write their codes into a zeroed bit string in shared memory at offsets given by a prefix sum over the
// lanes' code lengths (a unary run is just a skip).  The frame goes to its slot; k_enc_compact appends the CRC-16 as
// for every other frame.  The 128-thread kernels of fa_encode.h, whose 32-samples-per-thread layout keeps 36 of 128
// threads busy on such a frame, remain the fallback: a frame this path declines (short last frame, constant or wide
// samples, wasted bits, a subframe that would not beat VERBATIM) keeps fsize == 0 and is picked up by them.
#pragma once
#include "fa_encode.h"

namespace fa {

constexpr int kFxSpl = kFxBs / 32;             // samples per lane: 36
constexpr int kFxWarps = 2;                    // warps (frames in flight) per CTA
constexpr int kFxOutWords = 2 * kFxBs + 64;    // two channels at the VERBATIM size + headers

struct FxShared {                              // per warp
    alignas(16) int32_t stage[kFxBs];          // one channel of the frame as int32
    alignas(16) uint32_t out[kFxOutWords];     // the frame as an MSB-first bit string (zeroed, then OR-ed into)
};

// OR the nb (1..32) bits of v (< 2^nb) into the bit string at bit position pos
FA_D void fx_put(uint32_t* out, uint32_t pos, uint32_t v, int nb) {
    const uint32_t w = pos >> 5, off = pos & 31u;
    const unsigned long long x = (unsigned long long)v << (64 - (int)off - nb);
    atom_or_shared(out + w, (uint32_t)(x >> 32));
    if ((int)off + nb > 32) atom_or_shared(out + w + 1, (uint32_t)x);
}

// One warp: frame g.  false: not handled (no side effect besides scratch).
FA_D bool fixed_frame_warp(const EncParams& P, uint32_t g, FxShared* ws) {
    const int ln = lane();
    const int64_t s = (int64_t)(g / (uint32_t)P.nframes);
    const int f = (int)(g % (uint32_t)P.nframes);
    const int64_t samp0 = (int64_t)f * P.blocksize;
    if (P.blocksize != kFxBs || P.stream_size - samp0 < kFxBs) return false;
    const int bs = kFxBs, bps = 32, nch = P.nch;
    FrameSrc S;
    S.dtype = P.dtype; S.bs = bs; S.vec = false;
    S.off32 = 0.f; S.gain32 = 0.f; S.off64 = 0.; S.gain64 = 0.;
    if (P.dtype == kF32) { S.off32 = ((const float*)P.offsets)[s]; S.gain32 = ((const float*)P.gains)[s]; }
    if (P.dtype == kF64) { S.off64 = ((const double*)P.offsets)[s]; S.gain64 = ((const double*)P.gains)[s]; }
    const int esize = (P.dtype == kI32 || P.dtype == kF32) ? 4 : 8;
    S.base = (const unsigned char*)P.data + (s * P.stream_size + samp0) * esize;

    for (int i = ln; i < kFxOutWords; i += 32) ws->out[i] = 0u;
    syncwarp();
    uint32_t bitpos;
    {
        uint8_t fh[16];
        const int nfh = build_frame_header(fh, P.crc->crc8, bs, f, nch);
        if (ln == 0)
            for (int i = 0; i < nfh; ++i) fx_put(ws->out, 8u * (uint32_t)i, fh[i], 8);
        bitpos = 8u * (uint32_t)nfh;
    }
    const uint32_t verbatim_bits = (uint32_t)bps * (uint32_t)bs;

    for (int c = 0; c < nch; ++c) {
        // ---- stage the channel (coalesced), then 36 consecutive samples per lane + the four before them
        if (P.dtype == kF32) {
            const float* p = (const float*)S.base;
            const bool gain_pos = S.gain32 > 0.0f;
#pragma unroll 12
            for (int j = 0; j < kFxSpl; ++j) ws->stage[ln + 32 * j] = quant_f32_fast(p[ln + 32 * j], S.off32, S.gain32, gain_pos);
        } else if (P.dtype == kI32) {
            const int32_t* p = (const int32_t*)S.base;
#pragma unroll 12
            for (int j = 0; j < kFxSpl; ++j) ws->stage[ln + 32 * j] = p[ln + 32 * j];
        } else {
            for (int j = 0; j < kFxSpl; ++j) ws->stage[ln + 32 * j] = src_sample(S, c, ln + 32 * j);
        }
        syncwarp();
        int32_t x[kFxSpl];
#pragma unroll
        for (int q = 0; q < kFxSpl / 4; ++q) {
            const U4 v = lds128(ws->stage + kFxSpl * ln + 4 * q);
            x[4 * q] = (int32_t)v.x; x[4 * q + 1] = (int32_t)v.y; x[4 * q + 2] = (int32_t)v.z; x[4 * q + 3] = (int32_t)v.w;
        }
        int32_t hm1 = 0, hm2 = 0, hm3 = 0, hm4 = 0;
        if (ln != 0) {
            const U4 v = lds128(ws->stage + kFxSpl * ln - 4);
            hm4 = (int32_t)v.x; hm3 = (int32_t)v.y; hm2 = (int32_t)v.z; hm1 = (int32_t)v.w;
        }
        syncwarp();        // (every lane has its samples and its neighbour's last four: the stage can be overwritten)
        // ---- statistics: libFLAC fixed.c sums |e_k| over i >= 4
        uint32_t orv = 0;
        int32_t mn = 0x7fffffff, mx = (int32_t)0x80000000u;
        uint32_t fe0 = 0, fe1 = 0, fe2 = 0, fe3 = 0, fe4 = 0;
        {
            uint32_t p1 = (uint32_t)hm1 - (uint32_t)hm2;
            const uint32_t p1b = (uint32_t)hm2 - (uint32_t)hm3, p1c = (uint32_t)hm3 - (uint32_t)hm4;
            uint32_t p2 = p1 - p1b;
            uint32_t p3 = p2 - (p1b - p1c);
            int32_t xprev = hm1;
#pragma unroll
            for (int j = 0; j < kFxSpl; ++j) {
                const int32_t a0 = x[j];
                orv |= (uint32_t)a0;
                mn = a0 < mn ? a0 : mn;
                mx = a0 > mx ? a0 : mx;
                const uint32_t d1 = (uint32_t)a0 - (uint32_t)xprev;
                const uint32_t d2 = d1 - p1, d3 = d2 - p2, d4 = d3 - p3;
                p1 = d1; p2 = d2; p3 = d3;
                xprev = a0;
                if (j >= 4 || ln != 0) {
                    fe0 = sad_acc(a0, 0, fe0);
                    fe1 = sad_acc((int32_t)d1, 0, fe1);
                    fe2 = sad_acc((int32_t)d2, 0, fe2);
                    fe3 = sad_acc((int32_t)d3, 0, fe3);
                    fe4 = sad_acc((int32_t)d4, 0, fe4);
                }
            }
        }
        const uint32_t wor = redux_or(orv);
        const int32_t wmn = redux_min(mn), wmx = redux_max(mx);
        // CONSTANT subframes, wasted bits and wide samples (the 32-bit sums above need |x| < 2^22) are the other path's
        if (wmn == wmx || (wor & 1u) == 0u || wmn < -(1 << kNarrowBits) || wmx >= (1 << kNarrowBits)) return false;
        unsigned long long te[5];
        te[0] = warp_sum_u32_wide(fe0); te[1] = warp_sum_u32_wide(fe1); te[2] = warp_sum_u32_wide(fe2);
        te[3] = warp_sum_u32_wide(fe3); te[4] = warp_sum_u32_wide(fe4);
        // ---- order: libFLAC FLAC__fixed_compute_best_predictor (as design_fixed)
        int order;
        {
            const unsigned long long m34 = te[3] < te[4] ? te[3] : te[4];
            const unsigned long long m234 = te[2] < m34 ? te[2] : m34;
            const unsigned long long m1234 = te[1] < m234 ? te[1] : m234;
            if (te[0] < m1234) order = 0;
            else if (te[1] < m234) order = 1;
            else if (te[2] < m34) order = 2;
            else if (te[3] < te[4]) order = 3;
            else order = 4;
            const unsigned long long tsel = order == 0 ? te[0] : order == 1 ? te[1] : order == 2 ? te[2] : order == 3 ? te[3] : te[4];
            if (tsel > 0) {
                const float rb = flog2(0.6931472f * (float)tsel / (float)(bs - 4));
                if (!(rb < (float)bps)) return false;          // no gain expected: VERBATIM (other path)
            }
        }
        int maxp = max_porder_for(bs, order, P.max_porder);
        if (maxp > 3) maxp = 3;
        // ---- residual of that order, zigzag-coded back into the lane's own 36 words of the stage (the samples are not
        //      needed again); lane 0's first `order` samples are the warm-up and count as zero
        const int32_t w0 = x[0], w1 = x[1], w2 = x[2], w3 = x[3];
        unsigned long long lsum;
        {
            uint32_t p1 = (uint32_t)hm1 - (uint32_t)hm2;
            const uint32_t p1b = (uint32_t)hm2 - (uint32_t)hm3, p1c = (uint32_t)hm3 - (uint32_t)hm4;
            uint32_t p2 = p1 - p1b;
            uint32_t p3 = p2 - (p1b - p1c);
            int32_t xprev = hm1;
            uint32_t sa = 0, sb = 0;
#pragma unroll
            for (int q4 = 0; q4 < kFxSpl / 4; ++q4) {
                uint32_t zz[4];
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {
                    const int j = 4 * q4 + jj;
                    const int32_t a0 = x[j];
                    const uint32_t d1 = (uint32_t)a0 - (uint32_t)xprev;
                    const uint32_t d2 = d1 - p1, d3 = d2 - p2, d4 = d3 - p3;
                    p1 = d1; p2 = d2; p3 = d3;
                    xprev = a0;
                    const int32_t e = (int32_t)(order == 0 ? (uint32_t)a0 : order == 1 ? d1 : order == 2 ? d2 : order == 3 ? d3 : d4);
                    uint32_t z = ((uint32_t)e << 1) ^ (uint32_t)(e >> 31);
                    uint32_t ae = (uint32_t)(e < 0 ? -e : e);      // the parameter estimate works on sum |e| (libFLAC)
                    if (ln == 0 && j < order) { z = 0u; ae = 0u; }
                    zz[jj] = z;
                    if (jj & 1) sb += ae; else sa += ae;       // (|e| < 2^27: eighteen of them fit 32 bits)
                }
                U4 v; v.x = zz[0]; v.y = zz[1]; v.z = zz[2]; v.w = zz[3];
                sts128(ws->stage + kFxSpl * ln + 4 * q4, v);
            }
            lsum = (unsigned long long)sa + (unsigned long long)sb;
        }
        // ---- Rice parameters: partition order p has 2^p partitions of 32 >> p lanes
        unsigned long long seg[4];      // seg[p] = sum over this lane's partition at order p
        {
            unsigned long long v = lsum;
            v += shfl_xor64(v, 1); v += shfl_xor64(v, 2);
            seg[3] = v;
            v += shfl_xor64(v, 4);
            seg[2] = v;
            v += shfl_xor64(v, 8);
            seg[1] = v;
            v += shfl_xor64(v, 16);
            seg[0] = v;
        }
        uint32_t best_bits = 0xFFFFFFFFu;
        int best_p = 0, best_k = 0, best_r2 = 0;
#pragma unroll
        for (int p = 3; p >= 0; --p) {
            if (p > maxp) continue;
            const int lanes = 32 >> p;
            const int part = ln / lanes;
            const bool lead = (ln & (lanes - 1)) == 0;
            const uint32_t n = (uint32_t)(bs >> p) - (part == 0 ? (uint32_t)order : 0u);
            int kp;
            const uint32_t pb = rice_estimate(seg[p], n, kp);
            uint32_t bits = redux_add(lead ? pb : 0u) + 6u;
            const int r2 = ballot(kp >= 15) != 0u ? 1 : 0;
            if (r2) bits += (uint32_t)(1 << p);       // 5-bit parameters
            if (bits < best_bits) { best_bits = bits; best_p = p; best_k = kp; best_r2 = r2; }
        }
        const uint32_t hdr_bits = (uint32_t)subframe_header_bits(2, order, 0, bps, 0);
        if (hdr_bits + best_bits >= verbatim_bits + 8u) return false;      // VERBATIM is smaller (other path)
        // ---- exact code lengths, lane offsets
        const int k = best_k;
        const int plen = best_r2 ? 5 : 4;
        const bool leader = (ln & ((32 >> best_p) - 1)) == 0;
        const int skip = ln == 0 ? order : 0;           // warm-up samples: not coded
        uint32_t lbits = (leader ? (uint32_t)plen : 0u) + (uint32_t)(kFxSpl - skip) * (uint32_t)(k + 1);
        uint32_t qmax = 0;
#pragma unroll
        for (int q4 = 0; q4 < kFxSpl / 4; ++q4) {
            const U4 v = lds128(ws->stage + kFxSpl * ln + 4 * q4);
            const uint32_t q0 = v.x >> k, q1 = v.y >> k, q2 = v.z >> k, q3 = v.w >> k;      // (the warm-up slots hold zero)
            lbits += q0 + q1 + q2 + q3;
            qmax = qmax > (q0 | q1 | q2 | q3) ? qmax : (q0 | q1 | q2 | q3);
        }
        if (ballot(qmax > (1u << 16)) != 0u) return false;            // (an outlier the estimate did not see: other path)
        uint32_t incl = lbits;
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t o = shfl_up(incl, d);
            if (ln >= d) incl += o;
        }
        const uint32_t total = shfl(incl, 31);
        const uint32_t sub0 = bitpos;
        const uint32_t res0 = sub0 + hdr_bits;
        // (the exact size: a subframe that does not beat VERBATIM is the other path's -- which also bounds the frame by
        // the slot and the bit string by its buffer)
        if (hdr_bits + total >= verbatim_bits + 8u) return false;
        // ---- subframe header, warm-up, residual header (lane 0); then every lane its parameter and codes
        if (ln == 0) {
            uint32_t pos = sub0;
            fx_put(ws->out, pos, (uint32_t)(8 + order) << 1, 8); pos += 8;
            if (order > 0) { fx_put(ws->out, pos, (uint32_t)w0, 32); pos += 32; }
            if (order > 1) { fx_put(ws->out, pos, (uint32_t)w1, 32); pos += 32; }
            if (order > 2) { fx_put(ws->out, pos, (uint32_t)w2, 32); pos += 32; }
            if (order > 3) { fx_put(ws->out, pos, (uint32_t)w3, 32); pos += 32; }
            fx_put(ws->out, pos, (uint32_t)best_r2, 2); pos += 2;
            fx_put(ws->out, pos, (uint32_t)best_p, 4);
        }
        {
            // the lane's bits start at b0: a sequential packer with the current word in a register; finished words are
            // OR-ed into the string (the first and the last one are shared with the neighbouring lanes) -- one shared
            // atomic per word instead of two per code
            const uint32_t b0 = res0 + (incl - lbits);
            uint32_t pos = b0, cw = 0;
            auto flush = [&](uint32_t w, uint32_t val) { atom_or_shared(ws->out + w, val); };
            auto put = [&](uint32_t v, uint32_t nb) {        // nb in 1..32, v < 2^nb
                const uint32_t end = (pos & 31u) + nb;
                if (end < 32u) {
                    cw |= v << (32u - end);
                } else {
                    const uint32_t r = end - 32u;         // bits that go to the next word
                    flush(pos >> 5, cw | (v >> r));
                    cw = r ? v << (32u - r) : 0u;
                }
                pos += nb;
            };
            if (leader) put((uint32_t)k, (uint32_t)plen);
            const uint32_t kmask = (1u << k) - 1u, stop = 1u << k;
#pragma unroll 1
            for (int q4 = 0; q4 < kFxSpl / 4; ++q4) {
                const U4 v = lds128(ws->stage + kFxSpl * ln + 4 * q4);
                const uint32_t zz[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {
                    if (4 * q4 + jj < skip) continue;
                    const uint32_t npos = pos + (zz[jj] >> k);      // unary zeros: just move on (the string is zeroed)
                    if ((npos >> 5) != (pos >> 5)) { flush(pos >> 5, cw); cw = 0u; }
                    pos = npos;
                    put(stop | (zz[jj] & kmask), (uint32_t)k + 1u);
                }
            }
            if (pos & 31u) flush(pos >> 5, cw);
        }
        bitpos = res0 + total;
        syncwarp();
    }
    // ---- frame end: pad to a byte, copy to the slot (big-endian bit string -> bytes), publish the size
    const uint32_t nbytes = (bitpos + 7u) >> 3;
    uint8_t* slot = P.slots + (int64_t)(g - P.g_begin) * P.slot_bytes;
    for (uint32_t i = (uint32_t)ln; i < (nbytes + 15u) >> 4; i += 32u) {
        U4 v = lds128(ws->out + 4 * i);
        v.x = bswap32(v.x); v.y = bswap32(v.y); v.z = bswap32(v.z); v.w = bswap32(v.w);
        sts128(slot + 16 * i, v);
    }
    if (ln == 0) P.fsize[g - P.g_begin] = nbytes + 2u;
    syncwarp();
    return true;
}

}  // namespace fa
