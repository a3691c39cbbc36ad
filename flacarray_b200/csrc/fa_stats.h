// fa_stats.h -- per-row, per-bin statistics (count, min, max, mean, std) of decoded integer rows, exact in integers.
//
// Input: rows [n_rows][n] of int32 (1-channel streams) or int64 (2-channel streams), the decoder's output layout.  A row
// is split into bins of `bin` samples (the last one may be shorter) and every bin into pieces of at most `piece`
// samples.  One warp reduces one piece to an exact partial (S = sum x, Q = sum x^2, min, max); the partials of a bin are
// merged by plain integer addition, so the result does not depend on how the bin was cut or in which order the pieces
// are added.  The finisher forms n*Q - S^2 exactly in 256 bits, converts S and n*Q - S^2 to double with round to
// nearest even, and then uses plain IEEE double operations (no FMA):
//     mean_i = dbl(S) / n,   std_i = sqrt(dbl(n*Q - S^2)) / n
// Float arrays map these through the restore's own offset and coefficient (fa_quant.h): mean = off + coeff * mean_i,
// std = |coeff| * std_i, and min / max are the restored integer min / max (the restore is monotone).
//
// Widths: |x| <= 2^63 and a bin holds at most 2^32 - 1 samples, so |S| < 2^95 (two words) and Q < 2^158 (three words);
// n*Q and S^2 are below 2^190 and fit the 256-bit finisher.  The same bodies are compiled by nvcc (fab_row_stats) and by
// the host emulator of fa_simt.h (tests/hostsim/hostsim_stats.cpp).
#pragma once
#include <type_traits>

#include "fa_quant.h"
#include "fa_simt.h"

#if !defined(__CUDACC__)
#include <cmath>
#endif

namespace fa {

typedef unsigned __int128 u128;
typedef __int128 i128;

constexpr int kStatsWarps = 8;              // warps per CTA of k_row_stats / k_row_stats_merge
constexpr int kStatsPieceBytes = 32768;     // decoded bytes one warp reduces into one partial
constexpr int64_t kStatsMaxBin = 0xFFFFFFFFll;

// exact partial of one piece: S in two's complement (s0 low word), Q in q0:q1:q2, min and max widened to int64
struct StatPart {
    unsigned long long s0, s1, q0, q1, q2;
    long long mn, mx;
};

struct StatsParams {
    const void* rows;        // [n_rows][n] int32 (is_int64 == 0) or int64
    int is_int64;
    int64_t n_rows, n;
    int64_t bin;             // samples per bin (>= 1)
    int64_t nbins;           // ceil(n / bin)
    int64_t piece;           // samples per piece (>= 1)
    int64_t ppb;             // pieces per bin: ceil(bin / piece); 1 = the reducer finishes the bin itself
    StatPart* part;          // [n_rows][nbins][ppb] when ppb > 1
    const void* offsets;     // [n_rows] float32 / float64, or null (integer output); gains likewise
    const void* gains;
    const int* status;       // [n_rows] or null: rows with a non-zero status are filled
    long long* count;        // [n_rows][nbins] outputs
    void* mn;                // array dtype: int32 / int64 / float32 / float64
    void* mx;
    double* mean;
    double* std;
};

#if defined(__CUDACC__)
FA_D double bits_to_double(unsigned long long b) { return __longlong_as_double((long long)b); }
FA_D double dsqrt(double v) { return __dsqrt_rn(v); }
#else
inline double bits_to_double(unsigned long long b) { double d; memcpy(&d, &b, 8); return d; }
inline double dsqrt(double v) { return std::sqrt(v); }
#endif

FA_D unsigned long long lo64(u128 v) { return (unsigned long long)v; }
FA_D unsigned long long hi64(u128 v) { return (unsigned long long)(v >> 64); }

// ---- 256-bit helpers of the finisher -------------------------------------------------------------------------------
struct U256 { unsigned long long w[4]; };

FA_D U256 mul_128x128(u128 a, u128 b) {
    const u128 p00 = (u128)lo64(a) * lo64(b), p01 = (u128)lo64(a) * hi64(b);
    const u128 p10 = (u128)hi64(a) * lo64(b), p11 = (u128)hi64(a) * hi64(b);
    const u128 mid = (u128)hi64(p00) + lo64(p01) + lo64(p10);
    const u128 high = (u128)hi64(mid) + hi64(p01) + hi64(p10) + lo64(p11);
    U256 r;
    r.w[0] = lo64(p00); r.w[1] = lo64(mid); r.w[2] = lo64(high); r.w[3] = hi64(p11) + hi64(high);
    return r;
}

// q (192 bits) * n (64 bits)
FA_D U256 mul_192x64(unsigned long long q0, unsigned long long q1, unsigned long long q2, unsigned long long n) {
    U256 r;
    u128 t = (u128)q0 * n;
    r.w[0] = lo64(t);
    t = (u128)q1 * n + hi64(t);
    r.w[1] = lo64(t);
    t = (u128)q2 * n + hi64(t);
    r.w[2] = lo64(t);
    r.w[3] = hi64(t);
    return r;
}

FA_D U256 sub_256(const U256& a, const U256& b) {
    U256 r;
    unsigned long long borrow = 0;
    for (int i = 0; i < 4; ++i) {
        const unsigned long long d = a.w[i] - b.w[i];
        const unsigned long long bo = (a.w[i] < b.w[i]) | (d < borrow);
        r.w[i] = d - borrow;
        borrow = bo;
    }
    return r;
}

// bits [s, s + 64) of v (zero beyond the top)
FA_D unsigned long long bits_at(const U256& v, int s) {
    const int k = s >> 6, o = s & 63;
    const unsigned long long lo = k < 4 ? v.w[k] : 0ull, hi = k + 1 < 4 ? v.w[k + 1] : 0ull;
    return o ? (lo >> o) | (hi << (64 - o)) : lo;
}

// is any bit below position s set?
FA_D bool low_bits_set(const U256& v, int s) {
    for (int i = 0; i < 4; ++i) {
        if (s >= 64 * (i + 1)) { if (v.w[i]) return true; }
        else if (s > 64 * i) { if (v.w[i] & ((1ull << (s - 64 * i)) - 1)) return true; }
    }
    return false;
}

// the double nearest to v, ties to even (what Python's float(int) returns)
FA_D double dbl_u256(const U256& v) {
    int k = 3;
    while (k > 0 && v.w[k] == 0) --k;
    if (v.w[k] == 0) return 0.0;
    int p = 64 * k + 63 - clz64(v.w[k]);          // position of the top bit
    if (p < 53) return (double)v.w[0];           // exact
    unsigned long long m = bits_at(v, p - 52) & ((1ull << 53) - 1);
    const bool half = (bits_at(v, p - 53) & 1ull) != 0;
    if (half && (low_bits_set(v, p - 53) || (m & 1ull))) ++m;
    if (m >> 53) { m >>= 1; ++p; }
    return bits_to_double(((unsigned long long)(p + 1023) << 52) | (m & ((1ull << 52) - 1)));
}

FA_D double dbl_i128(unsigned long long s0, unsigned long long s1) {
    const bool neg = (long long)s1 < 0;
    const u128 s = ((u128)s1 << 64) | s0;
    const u128 a = neg ? (u128)0 - s : s;
    U256 v;
    v.w[0] = lo64(a); v.w[1] = hi64(a); v.w[2] = 0; v.w[3] = 0;
    const double d = dbl_u256(v);
    return neg ? -d : d;
}

// ---- partials -------------------------------------------------------------------------------------------------------
FA_D StatPart stat_identity() {
    StatPart p;
    p.s0 = p.s1 = p.q0 = p.q1 = p.q2 = 0;
    p.mn = (long long)0x7FFFFFFFFFFFFFFFull;
    p.mx = (long long)0x8000000000000000ull;
    return p;
}

FA_D void stat_add(StatPart& a, const StatPart& b) {
    const u128 s = (((u128)a.s1 << 64) | a.s0) + (((u128)b.s1 << 64) | b.s0);
    a.s0 = lo64(s); a.s1 = hi64(s);
    const u128 q = (((u128)a.q1 << 64) | a.q0) + (((u128)b.q1 << 64) | b.q0);
    a.q2 += b.q2 + (q < (((u128)b.q1 << 64) | b.q0) ? 1ull : 0ull);
    a.q0 = lo64(q); a.q1 = hi64(q);
    a.mn = b.mn < a.mn ? b.mn : a.mn;
    a.mx = b.mx > a.mx ? b.mx : a.mx;
}

FA_D unsigned long long shfl_xor64(unsigned long long v, int m) {
    const uint32_t lo = shfl_xor((uint32_t)v, m), hi = shfl_xor((uint32_t)(v >> 32), m);
    return ((unsigned long long)hi << 32) | lo;
}

FA_D void stat_warp_reduce(StatPart& p) {
    for (int m = 16; m >= 1; m >>= 1) {
        StatPart o;
        o.s0 = shfl_xor64(p.s0, m); o.s1 = shfl_xor64(p.s1, m);
        o.q0 = shfl_xor64(p.q0, m); o.q1 = shfl_xor64(p.q1, m); o.q2 = shfl_xor64(p.q2, m);
        o.mn = (long long)shfl_xor64((unsigned long long)p.mn, m);
        o.mx = (long long)shfl_xor64((unsigned long long)p.mx, m);
        stat_add(p, o);
    }
}

// per-lane accumulators: int32 rows keep S in 64 bits and Q in 128 (a lane adds at most piece / 32 samples of < 2^62)
struct LaneAcc32 {
    long long s = 0;
    u128 q = 0;
    int32_t mn = 0x7FFFFFFF, mx = (int32_t)0x80000000;
    FA_D void add(int32_t x) {
        s += x;
        q += (unsigned long long)((long long)x * x);
        mn = x < mn ? x : mn;
        mx = x > mx ? x : mx;
    }
    FA_D StatPart part() const {
        StatPart p;
        p.s0 = (unsigned long long)s; p.s1 = s < 0 ? ~0ull : 0ull;
        p.q0 = lo64(q); p.q1 = hi64(q); p.q2 = 0;
        p.mn = mn; p.mx = mx;
        return p;
    }
};

// int64 rows: with |x| = h 2^32 + l, x^2 = l^2 + 2 h l 2^32 + h^2 2^64, and each of the three products is one 32 x 32 -> 64
// multiply added into its own 128-bit sum; S is the sum of x read as unsigned, less 2^64 per negative x.  So the
// per-sample carry chains are two words long.  (Exact for up to 2^32 samples per lane.)
struct LaneAcc64 {
    u128 su = 0, a = 0, b = 0, c = 0;          // sum of (uint64)x; sums of l^2, h l, h^2
    unsigned long long neg = 0;                // number of negative x
    long long mn = (long long)0x7FFFFFFFFFFFFFFFull, mx = (long long)0x8000000000000000ull;
    FA_D void add(long long x) {
        su += (unsigned long long)x;
        neg += (unsigned long long)x >> 63;
        const unsigned long long ax = x < 0 ? 0ull - (unsigned long long)x : (unsigned long long)x;
        const unsigned long long h = ax >> 32, l = ax & 0xFFFFFFFFull;
        a += l * l;
        b += h * l;
        c += h * h;
        mn = x < mn ? x : mn;
        mx = x > mx ? x : mx;
    }
    FA_D StatPart part() const {
        StatPart p;
        p.s0 = lo64(su); p.s1 = hi64(su) - neg;
        const u128 b33 = b << 33;                      // b < 2^95
        u128 q = a + b33;
        unsigned long long q2 = q < b33 ? 1ull : 0ull;
        const u128 t = q + ((u128)lo64(c) << 64);
        q2 += (t < q ? 1ull : 0ull) + hi64(c);
        p.q0 = lo64(t); p.q1 = hi64(t); p.q2 = q2;
        p.mn = mn; p.mx = mx;
        return p;
    }
};

// samples of bin b: [b * bin, min((b + 1) * bin, n))
FA_D int64_t stats_bin_len(const StatsParams& P, int64_t b) {
    const int64_t lo = b * P.bin;
    return (lo + P.bin < P.n ? lo + P.bin : P.n) - lo;
}

// One finished (row, bin): the exact sums -> count, min, max, mean, std, or the fill of a failed row.
FA_D void stats_finish(const StatsParams& P, int64_t row, int64_t b, const StatPart& t) {
    const int64_t o = row * P.nbins + b;
    const bool flt = P.offsets != nullptr;
    if (P.status && P.status[row] != 0) {
        const double qnan = bits_to_double(0x7FF8000000000000ull);
        P.count[o] = 0;
        P.mean[o] = qnan;
        P.std[o] = qnan;
        if (P.is_int64) {
            const unsigned long long f = flt ? 0x7FF8000000000000ull : 0ull;
            ((unsigned long long*)P.mn)[o] = f;
            ((unsigned long long*)P.mx)[o] = f;
        } else {
            const uint32_t f = flt ? 0x7FC00000u : 0u;
            ((uint32_t*)P.mn)[o] = f;
            ((uint32_t*)P.mx)[o] = f;
        }
        return;
    }
    const int64_t n = stats_bin_len(P, b);
    const double dn = (double)n;
    // n*Q - S^2 >= 0 exactly (Cauchy-Schwarz), in 256 bits
    const u128 s = ((u128)t.s1 << 64) | t.s0;
    const u128 as = (long long)t.s1 < 0 ? (u128)0 - s : s;
    const U256 d = sub_256(mul_192x64(t.q0, t.q1, t.q2, (unsigned long long)n), mul_128x128(as, as));
    const double mean_i = ddiv(dbl_i128(t.s0, t.s1), dn);
    const double std_i = ddiv(dsqrt(dbl_u256(d)), dn);
    P.count[o] = n;
    if (!flt) {
        P.mean[o] = mean_i;
        P.std[o] = std_i;
        if (P.is_int64) {
            ((long long*)P.mn)[o] = t.mn;
            ((long long*)P.mx)[o] = t.mx;
        } else {
            ((int32_t*)P.mn)[o] = (int32_t)t.mn;
            ((int32_t*)P.mx)[o] = (int32_t)t.mx;
        }
    } else if (P.is_int64) {
        const double off = ((const double*)P.offsets)[row], coeff = restore_coeff_f64(((const double*)P.gains)[row]);
        P.mean[o] = dadd(off, dmul(coeff, mean_i));
        P.std[o] = dmul(coeff < 0.0 ? -coeff : coeff, std_i);
        const double a = restore_f64(t.mn, off, coeff), c = restore_f64(t.mx, off, coeff);
        ((double*)P.mn)[o] = a < c ? a : c;
        ((double*)P.mx)[o] = a < c ? c : a;
    } else {
        const float off = ((const float*)P.offsets)[row], coeff = restore_coeff_f32(((const float*)P.gains)[row]);
        const double doff = (double)off, dcoeff = (double)coeff;
        P.mean[o] = dadd(doff, dmul(dcoeff, mean_i));
        P.std[o] = dmul(dcoeff < 0.0 ? -dcoeff : dcoeff, std_i);
        const float a = restore_f32((int32_t)t.mn, off, coeff), c = restore_f32((int32_t)t.mx, off, coeff);
        ((float*)P.mn)[o] = a < c ? a : c;
        ((float*)P.mx)[o] = a < c ? c : a;
    }
}

// Chunk reducer: one warp reduces piece `idx` (bin idx / ppb, piece idx % ppb) of `row`.  The 16-byte aligned blocks
// inside the piece are read with 16-byte loads, four in flight per lane; the at most three elements before the first
// and after the last such block go through scalar loads.  No byte outside the piece is read.  With ppb == 1 lane 0
// finishes the bin, else it stores the partial for k_row_stats_merge.
template <bool I64>
FA_D void stats_piece_warp(const StatsParams& P, int64_t row, int64_t idx) {
    typedef typename std::conditional<I64, long long, int32_t>::type T;
    const int64_t b = idx / P.ppb, pc = idx - b * P.ppb;
    const int64_t bin_lo = b * P.bin, bin_hi = bin_lo + stats_bin_len(P, b);
    int64_t e0 = bin_lo + pc * P.piece, e1 = e0 + P.piece;
    if (e1 > bin_hi) e1 = bin_hi;
    if (e0 > e1) e0 = e1;                         // a piece past the end of a short last bin: empty
    const T* row_p = (const T*)P.rows + row * P.n;
    const uintptr_t a0 = (uintptr_t)(row_p + e0), a1 = (uintptr_t)(row_p + e1);
    const uintptr_t v0 = (a0 + 15) & ~(uintptr_t)15, v1 = a1 & ~(uintptr_t)15;
    const uintptr_t head_end = v0 < a1 ? v0 : a1, tail_beg = v1 > head_end ? v1 : head_end;
    const int n_head = (int)((head_end - a0) / sizeof(T)), n_tail = (int)((a1 - tail_beg) / sizeof(T));
    const int ln = lane();
    typename std::conditional<I64, LaneAcc64, LaneAcc32>::type acc;
    if (ln < n_head) acc.add(((const T*)a0)[ln]);
    else if (ln < n_head + n_tail) acc.add(((const T*)tail_beg)[ln - n_head]);
    if (v0 < v1) {
        const int64_t nv = (int64_t)((v1 - v0) >> 4);
        const unsigned char* vb = (const unsigned char*)v0;
        constexpr int U = 4;
        for (int64_t i = ln; i < nv; i += 32 * U) {
            U4 w[U];
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (i + 32 * u < nv) w[u] = ldg128(vb + (i + 32 * u) * 16);
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (i + 32 * u >= nv) break;
                if constexpr (I64) {
                    acc.add((long long)(((unsigned long long)w[u].y << 32) | w[u].x));
                    acc.add((long long)(((unsigned long long)w[u].w << 32) | w[u].z));
                } else {
                    acc.add((int32_t)w[u].x);
                    acc.add((int32_t)w[u].y);
                    acc.add((int32_t)w[u].z);
                    acc.add((int32_t)w[u].w);
                }
            }
        }
    }
    StatPart p = acc.part();
    stat_warp_reduce(p);
    if (ln != 0) return;
    if (P.ppb == 1) stats_finish(P, row, b, p);
    else P.part[(row * P.nbins + b) * P.ppb + pc] = p;
}

// Per-bin merge: one warp adds the ppb partials of (row, b) -- integer addition, so the order does not matter -- and
// lane 0 finishes the bin.
FA_D void stats_merge_warp(const StatsParams& P, int64_t row, int64_t b) {
    const StatPart* src = P.part + (row * P.nbins + b) * P.ppb;
    StatPart t = stat_identity();
    for (int64_t i = lane(); i < P.ppb; i += 32) stat_add(t, src[i]);
    stat_warp_reduce(t);
    if (lane() == 0) stats_finish(P, row, b, t);
}

}  // namespace fa
