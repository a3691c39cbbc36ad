// fa_decode_tile.h -- throughput decoder: one warp decodes 32 frames (one per lane) in lock step.
//
// Same role as frame_body() in fa_decode.h (libFLAC frame decode + the write callback
// decompress.c:66-101), restructured for the machine:
//   * compressed bytes stream through a per-lane shared-memory ring filled by cp.async at one
//     warp-uniform point per group of samples (see BitRdC: register prefetch stalls the whole warp);
//   * the bit reader is a CURSOR into that ring: every code is decoded from a 32-bit window fetched at
//     the cursor (two ring words + one funnel shift), so the steady-state loop has no refill branch and
//     no buffer state -- with 32 lanes at 32 different bit positions a "refill if low" test is taken by
//     some lane on almost every sample, i.e. the whole warp pays the refill every time;
//   * predictor history and coefficients live in registers (order <= 12, 32-bit samples), four
//     samples per loop trip so the history "shift" is register renaming;
//   * every lane appends its samples to a [32 lanes][32 samples] shared-memory tile; after 32 samples
//     the warp transposes the tile so that each store instruction writes 128 contiguous bytes of one
//     frame (fully coalesced), optionally restoring int32 -> float32 on the way (utils.c:350-368);
//   * the frame CRC-16 is checked by its own frame-parallel pass (crc_frame_warp, k_dec_crc);
//   * frames this path does not handle (33-bit side channel, order > 12, ...) are flagged and left to
//     the general per-thread decoder.
#pragma once
#include "fa_decode.h"
#include "fa_quant.h"

namespace fa {

constexpr int kTileOrd = 12;
constexpr int kTileStride = 36;   // words per tile row: 16-byte aligned rows, and rows 9 x 16 bytes apart keep 16-byte accesses
                                  // of 8 consecutive lanes (one row each, or one row together) on distinct banks
#ifndef FAB_TILE_WARPS
#define FAB_TILE_WARPS 1          // (CTAs of one warp retire item by item: 3.59 -> 3.53 ms against two-warp CTAs, 3.57 with four)
#endif
constexpr int kTileWarps = FAB_TILE_WARPS;  // warps per CTA

constexpr int kRingChunks = 4;                 // 16-byte chunks per lane in the shared-memory ring
constexpr int kRingWords = kRingChunks * 4;
constexpr int kRingStride = kRingWords + 4;    // words per lane row (16-byte aligned, spreads the banks)

struct TileRow {          // per-lane output description, read by all lanes during the flush
    int32_t* out;         // address of (frame sample 0, channel 0)
    int lo, hi;           // valid sample range inside the frame
    float off, coeff;     // int32 -> float32 restore (when enabled)
};

struct TileShared {       // per warp
    alignas(16) int32_t tile[32 * kTileStride];
    TileRow row[32];
    uint32_t ring[32 * kRingStride];   // compressed bytes in flight: one ring of kRingChunks chunks per lane
};

// Bit reader.  The compressed bytes of every lane's frame stream through a small ring in shared memory
// that is topped up with asynchronous 16-byte copies (cp.async) at ONE warp-uniform point per group of
// samples (brc_service).  A register prefetch queue does not work here: register scoreboards are per
// warp, so whenever one lane consumed its prefetched chunk the whole warp waited for the most recent
// load of ANY lane.  With the ring, loads never target a register.  `pos` is the bit cursor, counted
// from the first byte of the first chunk; ring word (pos >> 5) & 15 holds the bit under the cursor.
struct BitRdC {
    const U4* gp;      // next chunk to copy
    const U4* gend;    // first chunk holding no valid byte
    uint32_t* ring;    // this lane's ring (nullptr: inactive lane)
    uint32_t pos;      // bit cursor
    uint32_t pos0;     // cursor at brc_init
    uint32_t wr;       // chunks issued so far
    uint32_t landed;   // chunks known to be complete in the ring
    int err;
    // steady-state window (tile_next4): the big-endian ring words under the cursor and behind it, plus the byte offset of
    // the latter inside the ring.  Only valid between brc_window_load and the next call of any other reader routine.
    uint32_t cur, nxt, noff;
    int wok;           // the window is valid
};

FA_D U4 u4_zero() { U4 z; z.x = z.y = z.z = z.w = 0; return z; }

// Top the ring up (called at a warp-uniform point; lanes with nothing to do predicate off).
FA_D void brc_service(BitRdC& br) {
    cp_async_wait_all();          // copies issued at the previous service point: a whole sample group old
    br.landed = br.wr;
    // at most two chunks per service point: 8 samples rarely consume more than 32 bytes (a lane that does
    // runs into the wait of brc_ensure, which services again)
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        if (br.ring != nullptr && br.wr - (br.pos >> 7) < (uint32_t)kRingChunks) {
            uint32_t* slot = br.ring + (br.wr & (kRingChunks - 1)) * 4;
            if (br.gp < br.gend) cp_async16(slot, br.gp);
            else sts128(slot, u4_zero());     // past the end of the stream: zeros
            br.gp++;
            br.wr++;
        }
    }
    cp_async_commit();
}

// Make bits [pos, pos + nbits) readable (nbits <= 224: they fit the ring next to the cursor's chunk).
FA_D void brc_ensure(BitRdC& br, uint32_t nbits) {
    const uint32_t need = ((br.pos + nbits - 1u) >> 7) + 1u;     // chunks that must have landed
    if (need > br.landed) {
        // ran ahead of the copies (long codes, or the first words of a frame): wait for what is in flight; if that
        // is not enough, fetch now
        cp_async_wait_all();
        br.landed = br.wr;
        while (need > br.landed) {
            brc_service(br);
            cp_async_wait_all();
            br.landed = br.wr;
        }
    }
}

// the 32 bits under the cursor (the caller has ensured them)
FA_D uint32_t brc_peek(const BitRdC& br) {
    const uint32_t wi = br.pos >> 5;
    const uint32_t w0 = bswap32(br.ring[wi & (kRingWords - 1)]), w1 = bswap32(br.ring[(wi + 1) & (kRingWords - 1)]);
    return funnel_l(w1, w0, br.pos & 31u);
}

// Load the two-word window at the cursor (the caller has ensured >= 64 bits).
FA_D void brc_window_load(BitRdC& br) {
    const uint32_t wi = br.pos >> 5;
    br.cur = bswap32(br.ring[wi & (kRingWords - 1)]);
    br.noff = ((wi + 1) & (kRingWords - 1)) * 4u;
    br.nxt = bswap32(*(const uint32_t*)((const unsigned char*)br.ring + br.noff));
}

// Start reading at byte `start`.
FA_D void brc_init(BitRdC& br, uint32_t* ring, const uint8_t* start, const uint8_t* end) {
    uintptr_t s = (uintptr_t)start;
    br.gp = (const U4*)(s & ~(uintptr_t)15);
    br.gend = (const U4*)(((uintptr_t)end + 15) & ~(uintptr_t)15);
    br.ring = ring;
    br.pos = (uint32_t)(s & 15) * 8u;
    br.pos0 = br.pos;
    br.wr = 0;
    br.landed = 0;
    br.err = 0;
    br.cur = br.nxt = br.noff = 0;
    br.wok = 0;
    brc_service(br);
}

FA_D uint32_t brc_read(BitRdC& br, int nb) {  // nb in [0, 32]
    if (nb == 0) return 0u;
    brc_ensure(br, 64u);
    const uint32_t v = brc_peek(br) >> (32 - nb);
    br.pos += (uint32_t)nb;
    return v;
}
FA_D int32_t brc_read_signed(BitRdC& br, int nb) {  // nb in [0, 32]
    if (nb == 0) return 0;
    uint32_t v = brc_read(br, nb);
    uint32_t sign = 1u << (nb - 1);
    return (int32_t)((v ^ sign) - sign);
}
FA_D uint32_t brc_unary(BitRdC& br) {
    uint32_t q = 0;
    for (;;) {
        brc_ensure(br, 64u);
        const uint32_t w = brc_peek(br);
        if (w != 0) {
            const int z = clz32(w);
            br.pos += (uint32_t)z + 1u;
            return q + (uint32_t)z;
        }
        q += 32u;
        br.pos += 32u;
        if (br.gp > br.gend + 4 + kRingChunks) { br.err = 1; return q; }  // ran off the end of the stream
    }
}
FA_D int32_t unzigzag32(uint32_t u) { return (int32_t)(u >> 1) ^ sext1(u); }
// Rice code with parameter k (< 32): any length.
FA_D int32_t brc_rice(BitRdC& br, int k) {
    brc_ensure(br, 64u);
    const uint32_t w = brc_peek(br);
    const int z = clz32(w);                    // 32 when w == 0
    uint32_t q, low;
    if (z + 1 + k <= 32) {
        q = (uint32_t)z;
        low = k ? ((w << (z + 1)) >> (32 - k)) : 0u;     // (k >= 1 here implies z + 1 <= 31)
        br.pos += (uint32_t)(z + 1 + k);
    } else {
        q = brc_unary(br);
        low = brc_read(br, k);
    }
    return unzigzag32((q << k) | low);
}

// Bits consumed since brc_init.
FA_D int64_t brc_pos_bits(const BitRdC& br) { return (int64_t)(br.pos - br.pos0); }

struct TileLane {
    int mode;       // 0 const, 1 verbatim, 2 predictive
    int lpc;        // predictive: 1 = LPC subframe (parameters follow the warm-up), 0 = fixed predictor
    int order, shift, wasted, bps;
    int raw_left;   // warm-up / verbatim samples still to read
    int need_params;
    int32_t cval;
    int plen, esc, psize, part, nparts, left, k, rawbits;
    int fl;         // residuals of the current partition open to the four-at-a-time path: `left` when k >= 0, else 0
    // 32-bit prediction sums: exact whenever asum * (largest |sample| of the subframe) < 2^31.  `nar` is the lane's guess
    // after the warm-up (the bound holds for samples up to the next power of two above the warm-up's largest magnitude;
    // this library's encoder lowers the coefficient precision of narrow frames until asum * max|x| < 2^30, so the guess is
    // always "yes" for them); mn / mx follow every decoded sample and the subframe is CHECKED at its end -- a subframe
    // that breaks the bound after all goes to the general decoder, which keeps 64-bit sums.
    int32_t mn, mx;
    int asum;       // sum of |coefficient|
    int nar;
    int32_t h[kTileOrd];
    int32_t c[kTileOrd];
};

// Subframe header.  false => this path cannot decode it (br.err tells a bad stream from "unsupported").
FA_D bool tile_subframe_begin(BitRdC& br, int bs, int bps, TileLane& L) {
    if (brc_read(br, 1) != 0) return false;
    int type = (int)brc_read(br, 6);
    int wasted = 0;
    if (brc_read(br, 1)) wasted = (int)brc_unary(br) + 1;
    bps -= wasted;
    if (bps <= 0 || bps > 32 || br.err) return false;
    L.wasted = wasted;
    L.bps = bps;
    L.order = 0;
    L.lpc = 0;
    L.shift = 0;
    L.left = 0;
    L.fl = 0;
    L.part = -1;
    L.nparts = 0;
    L.k = 0;
    L.need_params = 0;
    L.mn = 0; L.mx = 0; L.asum = 0; L.nar = 0;
#pragma unroll
    for (int j = 0; j < kTileOrd; ++j) { L.h[j] = 0; L.c[j] = 0; }
    if (type == 0) {
        L.mode = 0;
        L.raw_left = 0;
        L.cval = brc_read_signed(br, bps);
        return true;
    }
    if (type == 1) {
        L.mode = 1;
        L.raw_left = bs;
        return true;
    }
    bool lpc = type >= 32;
    int order;
    if (lpc) order = (type & 31) + 1;
    else if (type >= 8 && type <= 12) order = type - 8;
    else return false;
    if (order > kTileOrd || order > bs) return false;
    L.mode = 2;
    L.lpc = lpc ? 1 : 0;
    L.order = order;
    L.raw_left = order;
    L.need_params = 1;
    return true;
}

// After the warm-up samples: LPC parameters + residual header.
FA_D bool tile_subframe_params(BitRdC& br, int bs, TileLane& L) {
    const int order = L.order;
    L.need_params = 0;
    if (L.lpc) {
        int prec = (int)brc_read(br, 4) + 1;
        if (prec == 16) return false;
        int sh = (int)brc_read(br, 5);
        if (sh & 16) return false;  // negative shift
        L.shift = sh;
#pragma unroll
        for (int j = 0; j < kTileOrd; ++j)
            if (j < order) L.c[j] = brc_read_signed(br, prec);
    } else {
        const int32_t fx[5][4] = {{0, 0, 0, 0}, {1, 0, 0, 0}, {2, -1, 0, 0}, {3, -3, 1, 0}, {4, -6, 4, -1}};
#pragma unroll
        for (int j = 0; j < 4; ++j) L.c[j] = fx[order][j];
    }
    {
        int a = 0;
#pragma unroll
        for (int j = 0; j < kTileOrd; ++j) a += L.c[j] < 0 ? -L.c[j] : L.c[j];        // < 12 * 2^14
        L.asum = a;
        const int64_t mw = (int64_t)L.mx > -(int64_t)L.mn ? (int64_t)L.mx : -(int64_t)L.mn;     // warm-up magnitude
        const int bits = 64 - clz64((uint64_t)mw);                                    // mw < 2^bits
        L.nar = (bits < 31 && ((uint64_t)a << bits) < (1ull << 31)) ? 1 : 0;
    }
    uint32_t method = brc_read(br, 2);
    if (method > 1) return false;
    L.plen = method == 0 ? 4 : 5;
    L.esc = method == 0 ? 15 : 31;
    int porder = (int)brc_read(br, 4);
    L.psize = bs >> porder;
    L.nparts = 1 << porder;
    if (porder > 0 && (L.psize << porder) != bs) return false;
    if (porder > 0 && L.psize < order) return false;
    L.part = -1;
    L.left = 0;
    L.fl = 0;
    return !br.err;
}

FA_D void tile_open_partition(BitRdC& br, TileLane& L) {
    while (L.left == 0) {
        L.part++;
        if (L.part >= L.nparts) { br.err = 1; L.left = 1 << 30; L.k = 0; L.fl = 0; return; }
        L.left = L.psize - (L.part == 0 ? L.order : 0);
        int k = (int)brc_read(br, L.plen);
        if (k == L.esc) { L.k = -1; L.rawbits = (int)brc_read(br, 5); }
        else L.k = k;
        L.fl = L.k >= 0 ? L.left : 0;
    }
}

// One sample, any mode (slow path: warm-up, verbatim, constant, partition edges, escapes).
template <int ORD>
FA_D int32_t tile_next_sample(BitRdC& br, TileLane& L) {
    int32_t v;
    if (L.mode == 0) {
        v = L.cval;
    } else if (L.raw_left > 0) {
        v = brc_read_signed(br, L.bps);
        L.raw_left--;
    } else {
        if (L.left == 0) tile_open_partition(br, L);
        L.left--;
        L.fl = L.fl > 0 ? L.fl - 1 : 0;
        int32_t r = (L.k >= 0) ? brc_rice(br, L.k) : brc_read_signed(br, L.rawbits);
        int64_t sum = 0;
#pragma unroll
        for (int j = 0; j < ORD; ++j) sum += (int64_t)L.c[j] * (int64_t)L.h[j];
        v = (int32_t)((int64_t)r + (sum >> L.shift));
    }
#pragma unroll
    for (int j = ORD - 1; j > 0; --j) L.h[j] = L.h[j - 1];
    if (ORD > 0) L.h[0] = v;
    L.mn = v < L.mn ? v : L.mn;
    L.mx = v > L.mx ? v : L.mx;
    return (int32_t)((uint32_t)v << L.wasted);
}

// Four residual samples of one partition (k >= 0): the steady-state inner loop.  The caller keeps the two-word window
// (br.cur, br.nxt) valid across consecutive calls.  The four codes are decoded WITHOUT branches on the assumption that
// each is at most 32 bits long: the 32 bits under the cursor come from the window with one funnel shift (no shared-memory
// access on the dependent chain: the word behind the window is fetched, predicated, only when the cursor crosses a word
// boundary), the position of the stop bit gives quotient, remainder shift and code length.  A code longer than 32 bits
// (stop bit not inside the window's first 32 - k bits) sets the sign of `bad`; the group is then decoded again from
// the saved cursor by the general routine -- rare: one code in ~10^4 on detector data.
// narrow (warp-uniform): every lane of the warp guessed that 32-bit prediction sums are exact (TileLane::nar).
template <int ORD>
FA_D void tile_next4(BitRdC& br, TileLane& L, int32_t* out4, const bool narrow) {
    int32_t r[4];
    const int k = L.k;
    brc_ensure(br, 4u * 32u + 64u);
    const uint32_t pos0 = br.pos;
    const uint32_t kmask = (1u << k) - 1u;
    const int n0 = 32 + k;               // code length = n0 - f, f = index of the stop bit in the 32-bit view
    int bad = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const uint32_t sh = br.pos & 31u;
        const uint32_t w = funnel_l(br.nxt, br.cur, sh);
        const int f = 31 - clz32(w);                     // -1 when w == 0
        const int d = f - k;                             // remainder = (w >> d) & kmask; d < 0: the code is longer than 32 bits
        bad |= d;
        const uint32_t u = ((uint32_t)(31 - f) << k) | ((w >> (d & 31)) & kmask);
        r[q] = unzigzag32(u);
        const uint32_t n = (uint32_t)(n0 - f);
        br.pos += n;
        if (sh + n >= 32u) {             // (n <= 33 here, and a group with n > 32 is decoded again: at most one word is crossed)
            br.cur = br.nxt;
            br.noff = (br.noff + 4u) & (kRingWords * 4u - 1u);
            br.nxt = bswap32(*(const uint32_t*)((const unsigned char*)br.ring + br.noff));
        }
    }
    if (bad < 0) {
        br.pos = pos0;
#pragma unroll
        for (int q = 0; q < 4; ++q) r[q] = brc_rice(br, k);      // (unrolled: a rolled loop would index r[] and park it in local memory)
        brc_ensure(br, 64u);
        brc_window_load(br);
    }
    L.left -= 4;
    L.fl -= 4;
    int32_t s[4];
    // history as seen by sample q: s[q-1], .., s[0], h[0], h[1], ...  The terms are added oldest first: the products with
    // the old history do not wait for anything, and only the last multiply-add of sample q waits for sample q - 1
    if (narrow) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            uint32_t sum = 0;
#pragma unroll
            for (int j = ORD - 1; j >= 0; --j) {
                int32_t hv = (j < q) ? s[q - 1 - j] : L.h[j - q];
                sum += (uint32_t)L.c[j] * (uint32_t)hv;
            }
            s[q] = (int32_t)((uint32_t)r[q] + (uint32_t)((int32_t)sum >> L.shift));
        }
    } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            int64_t sum = 0;
#pragma unroll
            for (int j = ORD - 1; j >= 0; --j) {
                int32_t hv = (j < q) ? s[q - 1 - j] : L.h[j - q];
                sum += (int64_t)L.c[j] * (int64_t)hv;
            }
            s[q] = (int32_t)((int64_t)r[q] + (sum >> L.shift));
        }
    }
    {
        const int32_t lo01 = s[0] < s[1] ? s[0] : s[1], hi01 = s[0] > s[1] ? s[0] : s[1];
        const int32_t lo23 = s[2] < s[3] ? s[2] : s[3], hi23 = s[2] > s[3] ? s[2] : s[3];
        const int32_t lo = lo01 < lo23 ? lo01 : lo23, hi = hi01 > hi23 ? hi01 : hi23;
        L.mn = lo < L.mn ? lo : L.mn;
        L.mx = hi > L.mx ? hi : L.mx;
    }
#pragma unroll
    for (int j = ORD - 1; j >= 4; --j) L.h[j] = L.h[j - 4];
#pragma unroll
    for (int q = 0; q < 4; ++q)
        if (3 - q < ORD) L.h[3 - q] = s[q];
    U4 o;
    o.x = (uint32_t)s[0] << L.wasted; o.y = (uint32_t)s[1] << L.wasted; o.z = (uint32_t)s[2] << L.wasted; o.w = (uint32_t)s[3] << L.wasted;
    sts128(out4, o);      // (tile rows are 16-byte aligned, the group starts at a multiple of four samples)
}

struct TileParams {
    DecParams D;
    int64_t j0, nwin;           // frame window (for the hinted blocksize)
    unsigned char* frame_flag;  // [n_sel][nframes_cap]: 1 = leave to the general decoder
    int restore;                // 1: nch == 1 and D.data receives float32 (offsets/gains given)
    const float* offsets;
    const float* gains;
    WinParams W;                // the windows (WIN instantiations only)
};

// Decode + flush all tiles of one channel pass with a compile-time upper bound on the predictor order.
template <int ORD>
FA_D void tile_channel_pass(const TileParams& P, TileShared* ws, BitRdC& br, TileLane& L, bool& run,
                            bool& fail, bool& punt, int bs, uint32_t bsmax, int c, int nch) {
    const int ln = lane();
    int32_t* trow = ws->tile + ln * kTileStride;
    for (uint32_t base = 0; base < bsmax; base += 32) {
        // (once per 32 samples: a lane only makes its guess when it reads its subframe parameters, inside the first block;
        // until every predictive lane has said "yes" the warp keeps the 64-bit loop)
        const bool narrow = ballot(run && L.mode == 2 && (L.need_params != 0 || L.nar == 0)) == 0;
#pragma unroll 1
        for (int s = 0; s < 32; s += 4) {
            int i = (int)base + s;
            if ((s & 4) == 0) brc_service(br);   // warp-uniform refill point of the compressed-byte rings (every 8 samples)
            if (run && i < bs) {
                // (fl >= 4 implies a predictive subframe past its warm-up and parameters, k >= 0, and -- partitions tile the
                // block -- four more samples inside the block)
                const bool fast = L.fl >= 4;
                if (fast) {
                    if (!br.wok) { brc_ensure(br, 64u); brc_window_load(br); br.wok = 1; }
                    tile_next4<ORD>(br, L, trow + s, narrow);
                } else {
                    br.wok = 0;
                    for (int q = 0; q < 4; ++q) {
                        int32_t v = 0;
                        if (run && i + q < bs) {
                            if (L.need_params && L.raw_left == 0) {
                                if (!tile_subframe_params(br, bs, L)) {
                                    run = false;
                                    if (br.err) fail = true; else punt = true;
                                }
                            }
                            if (run) v = tile_next_sample<ORD>(br, L);
                        }
                        trow[s + q] = v;
                    }
                }
            }
        }
        syncwarp();
        // transpose.  Common case (one channel, every active row holds all 32 samples of this block inside
        // its window, 16-byte aligned destination): 8 trips, each lane moves 4 consecutive samples of one
        // row with one 16-byte store (a group of 8 lanes covers a row: 128 contiguous bytes).
        bool vec_ok;
        {
            const TileRow mine = ws->row[ln];
            const bool inactive = mine.hi == 0;
            const bool full = mine.lo <= (int)base && (int)base + 32 <= mine.hi &&
                              ((((uintptr_t)(mine.out + base)) & 15) == 0);
            vec_ok = nch == 1 && ballot(!(inactive || full)) == 0;
        }
        if (vec_ok) {
            const int c4 = (ln & 7) * 4;
#pragma unroll 2
            for (int it = 0; it < 8; ++it) {
                const int r = it * 4 + (ln >> 3);
                const TileRow row = ws->row[r];
                if (row.hi != 0) {
                    const U4 tv = lds128(ws->tile + r * kTileStride + c4);
                    const int32_t v0 = (int32_t)tv.x, v1 = (int32_t)tv.y, v2 = (int32_t)tv.z, v3 = (int32_t)tv.w;
                    U4 q;
                    if (P.restore) {
                        float f0 = restore_f32(v0, row.off, row.coeff), f1 = restore_f32(v1, row.off, row.coeff);
                        float f2 = restore_f32(v2, row.off, row.coeff), f3 = restore_f32(v3, row.off, row.coeff);
                        memcpy(&q.x, &f0, 4); memcpy(&q.y, &f1, 4); memcpy(&q.z, &f2, 4); memcpy(&q.w, &f3, 4);
                    } else {
                        q.x = (uint32_t)v0; q.y = (uint32_t)v1; q.z = (uint32_t)v2; q.w = (uint32_t)v3;
                    }
                    sts128(row.out + base + c4, q);
                }
            }
        } else {
            // general: each iteration stores 32 consecutive samples of one frame (128 B)
            const int i = (int)base + ln;
#pragma unroll 4
            for (int r = 0; r < 32; ++r) {
                const TileRow row = ws->row[r];
                if ((uint32_t)(i - row.lo) < (uint32_t)(row.hi - row.lo)) {
                    int32_t v = ws->tile[r * kTileStride + ln];
                    if (P.restore) ((float*)row.out)[i] = restore_f32(v, row.off, row.coeff);
                    else row.out[(int64_t)i * nch + c] = v;
                }
            }
        }
        syncwarp();
    }
    // the subframe's prediction sums were exact in 32 bits?  (checked whether or not the warp took the 32-bit loop: a lane
    // only ever guesses "yes" wrongly when the signal outgrows its warm-up by more than a power of two)
    if (run && L.mode == 2 && L.nar) {
        const int64_t m = (int64_t)L.mx > -(int64_t)L.mn ? (int64_t)L.mx : -(int64_t)L.mn;
        if ((int64_t)L.asum * m >= (1ll << 31)) { run = false; punt = true; }
    }
}

// One warp: 32 consecutive work items (resolve_item: WIN = false the (stream, frame) pairs of fab_decode, WIN = true
// the frames of the windows of P.W).  `ws` = this warp's shared storage.
template <bool WIN = false>
FA_D void tile_warp_body(const TileParams& P, int64_t item0, TileShared* ws) {
    const DecParams& D = P.D;
    const int ln = lane();
    const int nch = D.nch;
    int64_t idx = item0 + ln;
    const WorkItem it = resolve_item<WIN>(D, P.W, P.nwin, idx);
    const int64_t k = it.k;
    bool active = k >= 0;
    int64_t j = 0;
    int bs_nom = 0, bs = 0;
    const uint8_t* fp = nullptr;
    const uint8_t* end = nullptr;
    long long off = 0, next = -1;
    if (active) {
        if (D.stream_flag[k] != 0) active = false;
    }
    if (active) {
        const StreamMeta m = D.meta[k];
        bs_nom = m.blocksize;
        int64_t jj0 = it.first / bs_nom, jj1 = (it.first + it.n - 1) / bs_nom;
        if (jj1 - jj0 + 1 > it.nwin) {
            if (it.jrel == 0) atom_or_global(&D.stream_flag[k], 1);
            active = false;
        } else {
            j = jj0 + it.jrel;
            if (j > jj1) active = false;
        }
    }
    FrameHdr fh;
    if (active) {
        const long long* fo = D.frame_off + k * (int64_t)(D.nframes_cap + 1);
        off = fo[j];
        next = fo[j + 1];
        if (off < 0) { atom_or_global(&D.stream_flag[k], 2); active = false; }
    }
    if (active) {
        const uint8_t* buf = D.bytes + D.starts[k];
        end = buf + D.nbytes[k];
        fp = buf + off;
        bool ok = parse_frame_header(fp, end - fp, D.crc, fh);
        int bps = ok ? (fh.bps ? fh.bps : D.meta[k].bps) : 0;
        if (!ok || fh.nch != nch || bps != 32 || fh.variable || (int64_t)fh.number != j) {
            atom_or_global(&D.stream_flag[k], 2);
            active = false;
        } else if (fh.ca >= 8) {
            P.frame_flag[k * (int64_t)D.nframes_cap + j] = 1;  // side channel: general decoder
            active = false;
        } else {
            bs = fh.blocksize;
        }
    }
    // publish the row description
    {
        TileRow r;
        r.out = nullptr; r.lo = 0; r.hi = 0; r.off = 0.f; r.coeff = 0.f;
        if (active) {
            int64_t s0 = j * (int64_t)bs_nom;
            r.out = D.data + (it.out + (s0 - it.first)) * nch;
            int64_t lo = it.first - s0, hi = it.first + it.n - s0;
            r.lo = (int)(lo < 0 ? 0 : lo);
            r.hi = (int)(hi > bs ? bs : hi);
            if (P.restore) { r.off = P.offsets[k]; r.coeff = restore_coeff_f32(P.gains[k]); }
        }
        ws->row[ln] = r;
    }
    syncwarp();
    uint32_t bsmax = (uint32_t)(active ? bs : 0);
    for (int m = 16; m >= 1; m >>= 1) { uint32_t o = shfl_xor(bsmax, m); bsmax = o > bsmax ? o : bsmax; }

    BitRdC br;
    if (active) {
        brc_init(br, ws->ring + ln * kRingStride, fp + fh.hdr_bytes, end);
    } else {
        br.gp = br.gend = nullptr; br.ring = nullptr; br.pos = br.pos0 = 0; br.wr = 0; br.landed = 0; br.err = 0;
        br.cur = br.nxt = br.noff = 0; br.wok = 0;
    }
    bool fail = false;      // stream problem -> walker
    bool punt = false;      // unsupported subframe -> general decoder
    TileLane L;
    L.mode = 0; L.order = 0; L.raw_left = 0; L.need_params = 0; L.left = 0; L.fl = 0; L.k = 0; L.wasted = 0; L.shift = 0; L.cval = 0;
    for (int c = 0; c < nch; ++c) {
        if (active && !fail && !punt) {
            if (!tile_subframe_begin(br, bs, 32, L)) {
                if (br.err) fail = true; else punt = true;
            }
        }
        bool run = active && !fail && !punt;
        // warp-uniform bound on the predictor order picks the instantiation of the sample loop
        uint32_t omax = (uint32_t)((run && L.mode == 2) ? L.order : 0);
        for (int m = 16; m >= 1; m >>= 1) { uint32_t o = shfl_xor(omax, m); omax = o > omax ? o : omax; }
        if (omax <= 4) tile_channel_pass<4>(P, ws, br, L, run, fail, punt, bs, bsmax, c, nch);
        else if (omax <= 8) tile_channel_pass<8>(P, ws, br, L, run, fail, punt, bs, bsmax, c, nch);
        else tile_channel_pass<kTileOrd>(P, ws, br, L, run, fail, punt, bs, bsmax, c, nch);
        if (run && br.err) fail = true;
    }
    if (active) {
        if (punt && !fail) {
            P.frame_flag[k * (int64_t)D.nframes_cap + j] = 1;
        } else if (!fail) {
            // frame end: pad to a byte, chain check against the next frame's start (the CRC-16 is k_dec_crc's job)
            int64_t bits = brc_pos_bits(br);               // relative to the body start
            int64_t body_bytes = (bits + 7) >> 3;
            int64_t len = fh.hdr_bytes + body_bytes + 2;
            if (fp + len > end) fail = true;
            if (!fail && next >= 0 && off + len != next) fail = true;
        }
        if (fail) atom_or_global(&D.stream_flag[k], 2);
    }
}

// ------------------------------------------------------------------------------------------------------
// Frame CRC-16 as its own frame-parallel pass (k_dec_crc): one warp per (stream, frame) item of the tile
// decoder's index space.  Inside the tile decoder the CRC was 23 % of the instructions, sitting on the
// serial per-lane chain and doubled by divergence; here the warp reads the frame in coalesced 512-byte rows
// and works in the trinomial domain of fa_bits.h (shifts and XORs only: no tables, no shared memory).  A
// mismatch flags the stream for the sequential walker exactly like a mismatch found by the general decoder.
// ------------------------------------------------------------------------------------------------------
template <bool WIN = false>
FA_D void crc_frame_warp(const TileParams& P, int64_t idx) {
    const DecParams& D = P.D;
    const int ln = lane();
    const WorkItem it = resolve_item<WIN>(D, P.W, P.nwin, idx);
    const int64_t k = it.k;
    if (k < 0) return;
    if (D.stream_flag[k] != 0) return;
    const int bs_nom = D.meta[k].blocksize;
    if (bs_nom <= 0) return;
    const int64_t jj0 = it.first / bs_nom, jj1 = (it.first + it.n - 1) / bs_nom;
    if (jj1 - jj0 + 1 > it.nwin) return;              // (the tile kernel hands this stream to the walker)
    const int64_t j = jj0 + it.jrel;
    if (j > jj1) return;
    const long long* fo = D.frame_off + k * (int64_t)(D.nframes_cap + 1);
    const long long off = fo[j], next = fo[j + 1];
    if (off < 0) return;                              // (flagged by the tile kernel)
    const long long nb = D.nbytes[k];
    const long long len = (next >= 0 ? next : nb) - off;
    if (len < 3 || off + len > nb) { if (ln == 0) atom_or_global(&D.stream_flag[k], 2); return; }
    const uint8_t* fp = D.bytes + D.starts[k] + off;
    const int64_t nbody = len - 2;
    const uint32_t want = ((uint32_t)fp[len - 2] << 8) | fp[len - 1];
    // The frame is cut into `head` bytes up to a 16-byte boundary, n16 aligned 16-byte chunks and a `tail`; the chunks form
    // rows of 32 that the warp loads with one coalesced 512-byte access each, RIGHT-aligned so that the last row is full.
    // Every lane keeps a Horner accumulator over its column in the trinomial domain (fa_bits.h: rows are 512 bytes apart,
    // * t^4096 is four shifts) plus the XOR of its words; the 32 columns are combined by a butterfly with power-of-two
    // shifts, head and tail are added by lane 0, and crct_finish forms the CRC.
    int64_t head = (int64_t)((16 - ((uintptr_t)fp & 15)) & 15);
    if (head > nbody) head = nbody;
    const int n16 = (int)((nbody - head) >> 4);
    const uint8_t* base = fp + head;
    uint32_t c = 0, px = 0;
    if (n16 > 0) {
        const int rows = (n16 + 31) >> 5;
        const int first = (rows << 5) - n16;          // lanes below this have no chunk in row 0
        const U4* cp = (const U4*)base + (ln - first);
        if (ln >= first) {
            const U4 q = ldg128(cp);
            c = crct_fold(crct_chunk(q));
            px = q.x ^ q.y ^ q.z ^ q.w;
        }
        for (int r = 1; r < rows; ++r) {
            cp += 32;
            const U4 q = ldg128(cp);
            c = crct_fold(crct_mulc<0x116u>(c) ^ crct_chunk(q));      // (c < 2^18 -> * t^4096 < 2^26)
            px ^= q.x ^ q.y ^ q.z ^ q.w;
        }
        c = crct_fold(crct_fold(c));
        // lane l's column still has to move 16 * (31 - l) bytes: combine groups of 1, 2, 4, 8, 16 lanes
        {
            uint32_t u;
            u = shfl_xor(c, 1);  if (ln & 1) c = crct_fold(crct_mulc<0x106u>(u)) ^ c;      // * t^128
            u = shfl_xor(c, 2);  if (ln & 2) c = crct_fold(crct_mulc<0x012u>(u)) ^ c;      // * t^256
            u = shfl_xor(c, 4);  if (ln & 4) c = crct_fold(crct_mulc<0x104u>(u)) ^ c;      // * t^512
            u = shfl_xor(c, 8);  if (ln & 8) c = crct_fold(crct_mulc<0x016u>(u)) ^ c;      // * t^1024
            u = shfl_xor(c, 16); if (ln & 16) c = crct_fold(crct_mulc<0x114u>(u)) ^ c;     // * t^2048
        }
        c = shfl(c, 31);
        px = redux_xor(px);
    }
    if (ln == 0) {
        // the head sits n16 * 16 bytes in front of the end of the chunks
        uint32_t h = 0;
        for (int64_t i = 0; i < head; ++i) { h = crct_byte(h, fp[i]); px ^= fp[i]; }
        if (head > 0 && n16 > 0) h = crct_shift_bytes(h, (uint64_t)n16 << 4);
        c ^= h;
        for (int64_t i = head + ((int64_t)n16 << 4); i < nbody; ++i) { c = crct_byte(c, fp[i]); px ^= fp[i]; }
        if (crct_finish(c, px) != want) atom_or_global(&D.stream_flag[k], 2);
    }
}

}  // namespace fa
