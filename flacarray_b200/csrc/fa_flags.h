// fa_flags.h -- per-row ranges of out-of-threshold samples of decoded integer rows.
//
// Input: rows [n_rows][n] of int32 (1-channel streams) or int64 (2-channel streams), the decoder's output layout.  Sample
// i of a row is flagged iff its value lies outside the row's keep range [L, H] (L > H: every sample is flagged).  Integer
// rows take [L, H] as given; float rows take float64 thresholds lo / hi and flag_bounds turns them into [L, H] once per
// row, so that the sample loop is two integer compares.  Flagged samples j1 < j2 that follow each other belong to one
// range iff j2 - j1 <= 2 * pad + 1; a range with first and last flagged samples js, je is reported as
// [max(js - pad, 0), min(je + pad + 1, n)) + sample0.
//
// Three passes over a caller-owned workspace (a per-row bitmask and one FlagPiece per piece of a row):
//   1. flag_scan_warp (one warp per piece): read the piece's samples with 16-byte loads, write its mask words, then
//      summarise them: flagged count, first and last flagged sample, and breaks (gaps > 2 * pad + 1) inside the piece.
//   2. flag_offsets_warp (one warp per row): walk the row's pieces forwards (is a piece's first flagged sample the start
//      of a range?) and backwards (is its last flagged sample the end of one?), giving each piece the index of its first
//      range start and of its first range end, and the row its flagged count and range count.
//   3. flag_write_warp (one warp per piece): read the piece's mask words and write every range start and end it holds
//      into its slot: the start by the piece of the range's first flagged sample, the end by that of its last.
//
// Mask layout.  A row that does not start on a 16-byte boundary (n % 4 != 0 for int32 rows) starts `a` elements past one.
// Bit t of the row's mask stands for sample t - a, so that every 16-byte vector of samples fills E = 16 / sizeof(T)
// consecutive bits of one mask word, and pieces are cut at multiples of `piece` bits (a multiple of 32): no two pieces
// share a mask word and every vector lies in one piece.  Samples outside the row are never read; their bits stay 0.
//
// The same bodies are compiled by nvcc (fab_flag_count, fab_flag_write) and by the host emulator of fa_simt.h
// (tests/hostsim/hostsim_flags.cpp).
#pragma once
#include <type_traits>

#include "fa_bits.h"
#include "fa_quant.h"
#include "fa_simt.h"

namespace fa {

constexpr int kFlagWarps = 8;              // warps per CTA of k_flag_scan / k_flag_offsets / k_flag_write
constexpr int kFlagPieceBytes = 32768;     // decoded bytes one warp scans
constexpr long long kFlagNone = 0x7FFFFFFFFFFFFFFFll;

// one piece of a row: pass 1 fills the first four fields, pass 2 the rest
struct FlagPiece {
    long long cnt, first, last, brk;       // flagged samples, first / last flagged sample of the row, breaks inside
    long long s_off, e_off;                // index (within the row) of the first range start / end the piece writes
    int fs, le;                            // does the first flagged sample start a range, the last one end a range?
    long long unused;
};

struct FlagParams {
    const void* rows;        // [n_rows][n] int32 (is_int64 == 0) or int64
    int is_int64;
    int64_t n_rows, n;
    int64_t piece;           // mask bits per piece, a multiple of 32
    int64_t ppr;             // pieces per row
    int64_t wpr;             // mask words per row
    int64_t pad;             // samples added on both sides of a flagged sample
    int64_t gap;             // min(2 * pad + 1, n): flagged samples further apart than this start a new range
    const void* lo;          // [n_rows] int64 L (integer rows) or float64 threshold (float rows)
    const void* hi;          // [n_rows] int64 H or float64 threshold
    const void* offsets;     // [n_rows] float32 / float64, or null (integer rows); gains likewise
    const void* gains;
    const int* status;       // [n_rows] or null: rows with a non-zero status are skipped
    uint32_t* mask;          // [n_rows][wpr]
    FlagPiece* sum;          // [n_rows][ppr]
    long long* nflag;        // [n_rows] flagged samples (-1 for a skipped row)
    long long* nrange;       // [n_rows] ranges (0 for a skipped row)
    const long long* base;   // [n_rows] first output slot of each row (pass 3)
    int64_t sample0;         // index of a row's sample 0 in its stream
    long long* first_out;    // range starts / ends (pass 3)
    long long* last_out;
};

FA_HD size_t flag_align(size_t v) { return (v + 255) & ~(size_t)255; }

// Geometry of a call on rows [n_rows][n]; piece == 0 is kFlagPieceBytes of samples per piece (the library), the host
// emulator passes smaller pieces.  Returns 0 and fills *P's geometry, or the error bits of bad arguments.
inline int flag_geometry(int64_t n_rows, int64_t n, int is_int64, int64_t pad, FlagParams* P, int64_t piece = 0) {
    if (n_rows <= 0) return kErrZeroNstream;
    if (n <= 0) return kErrZeroStreamsize;
    if (pad < 0 || piece < 0 || piece % 32 != 0) return kErrDecodeSampleRange;
    const int64_t amax = is_int64 ? 1 : 3;              // a row starts at most this many elements past a 16-byte boundary
    P->is_int64 = is_int64 ? 1 : 0;
    P->n_rows = n_rows; P->n = n; P->pad = pad;
    P->gap = pad >= n ? n : (2 * pad + 1 < n ? 2 * pad + 1 : n);
    P->piece = piece > 0 ? piece : kFlagPieceBytes / (is_int64 ? 8 : 4);
    P->ppr = (n + amax + P->piece - 1) / P->piece;
    P->wpr = (n + amax + 31) / 32;
    if ((P->ppr + kFlagWarps - 1) / kFlagWarps > 0x7FFFFFFFll || (n_rows + kFlagWarps - 1) / kFlagWarps > 0x7FFFFFFFll)
        return kErrAlloc;
    return 0;
}

// bytes of the mask and of the piece records (each 256-byte aligned); the records follow the mask
inline size_t flag_mask_bytes(const FlagParams& P) { return flag_align((size_t)P.n_rows * (size_t)P.wpr * 4); }
inline size_t flag_workspace_bytes(const FlagParams& P) {
    return flag_mask_bytes(P) + flag_align((size_t)P.n_rows * (size_t)P.ppr * sizeof(FlagPiece));
}

// ---- the keep range of a float row --------------------------------------------------------------------------------
// The restore of biased integer u (u = x + 2^(B-1) as an unsigned B-bit number, so that u orders like x), widened.
template <bool I64>
FA_D double flag_restore(unsigned long long u, double off, double coeff) {
    if constexpr (I64) return restore_f64((long long)(u ^ 0x8000000000000000ull), off, coeff);
    else return (double)restore_f32((int32_t)((uint32_t)u ^ 0x80000000u), (float)off, (float)coeff);
}

// The largest u with q(u) false, q(u) = ((above ? v > t : v < t) != neg) for v the restore of u, when q is false then
// true as u grows.  Returns false when q(0) is already true.  B + 1 restores.
template <bool I64>
FA_D bool flag_last_false(double off, double coeff, double t, bool above, bool neg, unsigned long long* r) {
    unsigned long long u = 0;
    double v = flag_restore<I64>(u, off, coeff);
    if ((above ? v > t : v < t) != neg) return false;
    for (int b = I64 ? 63 : 31; b >= 0; --b) {
        const unsigned long long c = u | (1ull << b);
        v = flag_restore<I64>(c, off, coeff);
        if ((above ? v > t : v < t) == neg) u = c;
    }
    *r = u;
    return true;
}

// [L, H] of a float row: the restored value v of x (restore_f64, or restore_f32 widened to double, with this row's
// offset and coefficient, float32 values passed as double) satisfies lo <= v <= hi iff L <= x <= H.  The restore is
// monotone in x -- non-decreasing for coeff >= 0 and non-increasing for coeff < 0 -- so the samples it keeps form one
// integer interval, found with two binary searches over the integers.  L > H: no integer is kept (every sample is
// flagged).  lo = -inf / hi = +inf leave that side open.
template <bool I64>
FA_D void flag_bounds(double off, double coeff, double lo, double hi, long long* L, long long* H) {
    const unsigned long long bias = I64 ? 0x8000000000000000ull : 0x80000000ull;
    const unsigned long long top = I64 ? ~0ull : 0xFFFFFFFFull;        // the largest biased integer
    // coeff >= 0: the samples under lo are a prefix of the biased integers and those over hi a suffix; coeff < 0: the
    // samples over hi are the prefix and those under lo the suffix.  The kept biased range is [lo_u, hi_u].
    const bool up = !(coeff < 0.0);
    unsigned long long r, lo_u = 0, hi_u = 0;
    bool none = false;
    if (flag_last_false<I64>(off, coeff, up ? lo : hi, !up, true, &r)) {     // r: the last integer of the prefix
        if (r == top) none = true;
        else lo_u = r + 1;
    }
    if (flag_last_false<I64>(off, coeff, up ? hi : lo, up, false, &r)) hi_u = r;   // r: the last integer kept
    else none = true;
    if (none || lo_u > hi_u) { *L = 1; *H = 0; return; }
    if constexpr (I64) { *L = (long long)(lo_u ^ bias); *H = (long long)(hi_u ^ bias); }
    else { *L = (long long)(int32_t)(uint32_t)(lo_u ^ bias); *H = (long long)(int32_t)(uint32_t)(hi_u ^ bias); }
}

// ---- runs of mask words --------------------------------------------------------------------------------------------
struct FlagRun {
    long long cnt, first, last, brk;
};

// bits of w that have a set bit of w 1 .. g places below them (g < 32)
FA_D uint32_t flag_cover(uint32_t w, long long g) {
    uint32_t r = 0, p = w;                              // p = w | w << 1 | ... | w << (pw - 1)
    int sh = 0;
    for (int pw = 1; pw < 32; pw <<= 1) {
        if (g & pw) { r |= p << sh; sh += pw; }
        p |= p << pw;
    }
    return r << 1;
}

// Summary of mask words [k0, k1) of one row, in order; bit b of word k is sample 32 k + b - a.
FA_D FlagRun flag_run_words(const uint32_t* mw, int64_t k0, int64_t k1, int a, long long g) {
    FlagRun r{0, 0, -1, 0};
    for (int64_t k = k0; k < k1; ++k) {
        const uint32_t w = mw[k];
        if (!w) continue;
        const long long b0 = 32 * k - a;
        const long long f = b0 + ctz32(w), l = b0 + 31 - clz32(w);
        if (r.cnt == 0) r.first = f;
        else if (f - r.last > g) r.brk++;
        if (g < 32) r.brk += popc32(w & ~flag_cover(w, g)) - 1;
        r.last = l;
        r.cnt += popc32(w);
    }
    return r;
}

// r followed by s
FA_D FlagRun flag_join(const FlagRun& r, const FlagRun& s, long long g) {
    if (s.cnt == 0) return r;
    if (r.cnt == 0) return s;
    FlagRun t;
    t.cnt = r.cnt + s.cnt;
    t.first = r.first;
    t.last = s.last;
    t.brk = r.brk + s.brk + (s.first - r.last > g ? 1 : 0);
    return t;
}

FA_D long long shfl_down_ll(long long v, int d) { return (long long)shfl64((unsigned long long)v, lane() + d < 32 ? lane() + d : 31); }
FA_D long long shfl_up_ll(long long v, int d) { return (long long)shfl_up64((unsigned long long)v, d); }
FA_D long long shfl_ll(long long v, int src) { return (long long)shfl64((unsigned long long)v, src); }

// element offset of a row's first sample past the 16-byte boundary below it
template <typename T>
FA_D int flag_row_shift(const T* row_p) { return (int)(((uintptr_t)row_p & 15) / sizeof(T)); }

// mask words [*k0, *k1) of piece pc of a row with shift a, and lane `ln`'s share [*l0, *l1) of them
FA_D void flag_piece_words(const FlagParams& P, int64_t pc, int a, int64_t* k0, int64_t* k1, int64_t* l0, int64_t* l1) {
    const int64_t t0 = pc * P.piece;
    int64_t t1 = t0 + P.piece;
    if (t1 > a + P.n) t1 = a + P.n;
    *k0 = t0 / 32;
    *k1 = t1 > t0 ? (t1 + 31) / 32 : *k0;
    const int64_t per = (*k1 - *k0 + 31) / 32;
    *l0 = *k0 + lane() * per;
    *l1 = *l0 + per < *k1 ? *l0 + per : *k1;
    if (*l0 > *l1) *l0 = *l1;
}

// ---- pass 1 --------------------------------------------------------------------------------------------------------
template <bool I64>
FA_D void flag_scan_warp(const FlagParams& P, int64_t row, int64_t pc) {
    typedef typename std::conditional<I64, long long, int32_t>::type T;
    constexpr int E = 16 / (int)sizeof(T);              // samples per 16-byte vector
    constexpr int LPW = 32 / E;                         // lanes per mask word
    constexpr int U = 4;
    if (P.status && P.status[row] != 0) return;
    const int ln = lane();
    const T* row_p = (const T*)P.rows + row * P.n;
    const int a = flag_row_shift(row_p);
    const uintptr_t vbase = (uintptr_t)row_p - (uintptr_t)a * sizeof(T);     // 16-byte aligned: bit t <-> vbase + t
    T L, H;
    {
        long long l, h;
        if (P.offsets) {
            const double lo = ((const double*)P.lo)[row], hi = ((const double*)P.hi)[row];
            if constexpr (I64)
                flag_bounds<true>(((const double*)P.offsets)[row], restore_coeff_f64(((const double*)P.gains)[row]), lo, hi,
                                  &l, &h);
            else
                flag_bounds<false>((double)((const float*)P.offsets)[row],
                                   (double)restore_coeff_f32(((const float*)P.gains)[row]), lo, hi, &l, &h);
        } else {
            l = ((const long long*)P.lo)[row];
            h = ((const long long*)P.hi)[row];
        }
        if constexpr (!I64) {                           // the same flags with int32 bounds
            if (l > h || l > 0x7FFFFFFFll || h < -0x80000000ll) { l = 1; h = 0; }
            else { l = l < -0x80000000ll ? -0x80000000ll : l; h = h > 0x7FFFFFFFll ? 0x7FFFFFFFll : h; }
        }
        L = (T)l;
        H = (T)h;
    }
    const int64_t t0 = pc * P.piece, tv = a + P.n;      // bits [a, tv) hold samples
    int64_t t1 = t0 + P.piece;
    if (t1 > tv) t1 = tv;
    const int64_t nslot = t1 > t0 ? (t1 - t0 + E - 1) / E : 0;
    uint32_t* mw = P.mask + row * P.wpr + t0 / 32;
    for (int64_t i0 = 0; i0 < nslot; i0 += 32 * U) {
        U4 w[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t i = i0 + 32 * u + ln, t = t0 + E * i;
            if (i < nslot && t >= a && t + E <= tv) w[u] = ldg128((const void*)(vbase + (uintptr_t)t * sizeof(T)));
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (i0 + 32 * u >= nslot) break;            // the same in every lane
            const int64_t i = i0 + 32 * u + ln, t = t0 + E * i;
            uint32_t f = 0;
            if (i < nslot && t >= a && t + E <= tv) {
                if constexpr (I64) {
                    const long long x0 = (long long)(((unsigned long long)w[u].y << 32) | w[u].x);
                    const long long x1 = (long long)(((unsigned long long)w[u].w << 32) | w[u].z);
                    f = (uint32_t)(x0 < L || x0 > H) | (uint32_t)(x1 < L || x1 > H) << 1;
                } else {
                    const int32_t x0 = (int32_t)w[u].x, x1 = (int32_t)w[u].y, x2 = (int32_t)w[u].z, x3 = (int32_t)w[u].w;
                    f = (uint32_t)(x0 < L || x0 > H) | (uint32_t)(x1 < L || x1 > H) << 1 |
                        (uint32_t)(x2 < L || x2 > H) << 2 | (uint32_t)(x3 < L || x3 > H) << 3;
                }
            } else if (i < nslot) {                     // the vector holds bits outside the row: element by element
                for (int e = 0; e < E; ++e) {
                    const int64_t te = t + e;
                    if (te >= a && te < tv) {
                        const T x = row_p[te - a];
                        f |= (uint32_t)(x < L || x > H) << e;
                    }
                }
            }
            uint32_t v = f << (E * (ln % LPW));
#pragma unroll
            for (int m = 1; m < LPW; m <<= 1) v |= shfl_xor(v, m);
            if (ln % LPW == 0 && i < nslot) mw[i / LPW] = v;
        }
    }
    syncwarp();                                         // the piece's words are visible to the whole warp
    int64_t k0, k1, l0, l1;
    flag_piece_words(P, pc, a, &k0, &k1, &l0, &l1);
    const uint32_t* rm = P.mask + row * P.wpr;
    FlagRun r = flag_run_words(rm, l0, l1, a, P.gap);
    for (int d = 1; d < 32; d <<= 1) {                  // ordered reduction: lane i joins lanes [i, i + 2d)
        FlagRun o;
        o.cnt = shfl_down_ll(r.cnt, d); o.first = shfl_down_ll(r.first, d);
        o.last = shfl_down_ll(r.last, d); o.brk = shfl_down_ll(r.brk, d);
        if (ln + d < 32) r = flag_join(r, o, P.gap);
    }
    if (ln == 0) {
        FlagPiece* s = P.sum + row * P.ppr + pc;
        s->cnt = r.cnt; s->first = r.first; s->last = r.last; s->brk = r.brk;
    }
}

// ---- pass 2 --------------------------------------------------------------------------------------------------------
FA_D void flag_offsets_warp(const FlagParams& P, int64_t row) {
    const int ln = lane();
    if (P.status && P.status[row] != 0) {
        if (ln == 0) { P.nflag[row] = -1; P.nrange[row] = 0; }
        return;
    }
    FlagPiece* s = P.sum + row * P.ppr;
    const long long g = P.gap;
    // forwards: the last flagged sample before each piece decides whether its first flagged sample starts a range
    long long carry_last = -1, carry_s = 0, carry_n = 0;
    for (int64_t c0 = 0; c0 < P.ppr; c0 += 32) {
        const int64_t p = c0 + ln;
        long long cnt = 0, first = 0, brk = 0, last = -1;
        if (p < P.ppr) { cnt = s[p].cnt; first = s[p].first; last = s[p].last; brk = s[p].brk; }
        long long mx = cnt ? last : -1, sc, nc = cnt;
        for (int d = 1; d < 32; d <<= 1) {
            const long long o = shfl_up_ll(mx, d);
            if (ln >= d && o > mx) mx = o;
        }
        long long prev = shfl_up_ll(mx, 1);
        if (ln == 0) prev = -1;
        if (carry_last > prev) prev = carry_last;
        const int fs = cnt != 0 && (prev < 0 || first - prev > g);
        const long long st = cnt ? brk + fs : 0;
        sc = st;
        for (int d = 1; d < 32; d <<= 1) {
            const long long o = shfl_up_ll(sc, d), on = shfl_up_ll(nc, d);
            if (ln >= d) { sc += o; nc += on; }
        }
        if (p < P.ppr) { s[p].s_off = carry_s + sc - st; s[p].fs = fs; }
        const long long m31 = shfl_ll(mx, 31);
        carry_last = m31 > carry_last ? m31 : carry_last;
        carry_s += shfl_ll(sc, 31);
        carry_n += shfl_ll(nc, 31);
    }
    // backwards: the first flagged sample after each piece decides whether its last flagged sample ends a range
    long long carry_next = kFlagNone, carry_e = 0;
    for (int64_t c0 = (P.ppr - 1) / 32 * 32; c0 >= 0; c0 -= 32) {
        const int64_t p = c0 + ln;
        long long cnt = 0, first = 0, brk = 0, last = -1;
        if (p < P.ppr) { cnt = s[p].cnt; first = s[p].first; last = s[p].last; brk = s[p].brk; }
        long long mn = cnt ? first : kFlagNone;
        for (int d = 1; d < 32; d <<= 1) {
            const long long o = shfl_down_ll(mn, d);
            if (ln + d < 32 && o < mn) mn = o;
        }
        long long next = shfl_down_ll(mn, 1);
        if (ln == 31) next = kFlagNone;
        if (carry_next < next) next = carry_next;
        const int le = cnt != 0 && (next == kFlagNone || next - last > g);
        const long long en = cnt ? brk + le : 0;
        long long ec = en;
        for (int d = 1; d < 32; d <<= 1) {
            const long long o = shfl_down_ll(ec, d);
            if (ln + d < 32) ec += o;
        }
        if (p < P.ppr) { s[p].e_off = carry_s - carry_e - ec; s[p].le = le; }
        const long long m0 = shfl_ll(mn, 0);
        carry_next = m0 < carry_next ? m0 : carry_next;
        carry_e += shfl_ll(ec, 0);
    }
    if (ln == 0) { P.nflag[row] = carry_n; P.nrange[row] = carry_s; }
}

// ---- pass 3 --------------------------------------------------------------------------------------------------------
FA_D void flag_write_warp(const FlagParams& P, int64_t row, int64_t pc) {
    if (P.status && P.status[row] != 0) return;
    const FlagPiece* sp = P.sum + row * P.ppr + pc;
    if (sp->cnt == 0) return;                           // the same in every lane
    const int ln = lane();
    const int esz = P.is_int64 ? 8 : 4;
    const int a = (int)((((uintptr_t)P.rows + (uintptr_t)(row * P.n * esz)) & 15) / esz);
    int64_t k0, k1, l0, l1;
    flag_piece_words(P, pc, a, &k0, &k1, &l0, &l1);
    const uint32_t* rm = P.mask + row * P.wpr;
    const long long g = P.gap, n = P.n, pad = P.pad;
    const FlagRun r = flag_run_words(rm, l0, l1, a, g);
    long long mx = r.cnt ? r.last : -1, mn = r.cnt ? r.first : kFlagNone;
    for (int d = 1; d < 32; d <<= 1) {
        const long long o = shfl_up_ll(mx, d), q = shfl_down_ll(mn, d);
        if (ln >= d && o > mx) mx = o;
        if (ln + d < 32 && q < mn) mn = q;
    }
    long long prev = shfl_up_ll(mx, 1), next = shfl_down_ll(mn, 1);
    if (ln == 0) prev = -1;
    if (ln == 31) next = kFlagNone;
    const int fs = r.cnt != 0 && (prev >= 0 ? r.first - prev > g : sp->fs != 0);
    const int le = r.cnt != 0 && (next != kFlagNone ? next - r.last > g : sp->le != 0);
    const long long st = r.cnt ? r.brk + fs : 0, en = r.cnt ? r.brk + le : 0;
    long long sc = st, ec = en;
    for (int d = 1; d < 32; d <<= 1) {
        const long long o = shfl_up_ll(sc, d), q = shfl_up_ll(ec, d);
        if (ln >= d) { sc += o; ec += q; }
    }
    const long long b = P.base[row];
    long long* fo = P.first_out + b + sp->s_off + (sc - st);
    long long* eo = P.last_out + b + sp->e_off + (ec - en);
    const long long s0 = P.sample0;
    long long pj = -1;                                  // the previous flagged sample of this lane
    for (int64_t k = l0; k < l1; ++k) {
        uint32_t w = rm[k];
        while (w) {
            const long long j = 32 * k - a + ctz32(w);
            w &= w - 1;
            if (pj < 0) {
                if (fs) *fo++ = s0 + (j > pad ? j - pad : 0);
            } else if (j - pj > g) {
                *eo++ = s0 + (pad < n - pj ? pj + pad + 1 : n);
                *fo++ = s0 + (j > pad ? j - pad : 0);
            }
            pj = j;
        }
    }
    if (pj >= 0 && le) *eo = s0 + (pad < n - pj ? pj + pad + 1 : n);
}

}  // namespace fa
