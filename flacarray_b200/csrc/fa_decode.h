// fa_decode.h -- FLAC stream/frame decoding bodies (one CUDA thread decodes one frame).
//
// Replaces the libFLAC decoder that the reference drives through decompress.c:194-313 and the
// write callback decompress.c:66-101 (interleave channels, clip to [first, first + n_decode)).
// Parallel unit = (selected stream, frame): frames are found either through this library's own
// frame-size table (APPLICATION block "faB2") or, for foreign streams such as libFLAC's, by a
// parallel sync-code scan validated with CRC-8 + frame number + block size; the decode then
// verifies that every frame ends exactly where the next one begins.
#pragma once
#include "fa_bits.h"

namespace fa {

constexpr int kMaxLpcOrder = 32;

// Per-stream metadata extracted by k_parse_meta.
struct StreamMeta {
    int64_t first_frame;   // byte offset of the first frame inside the stream window, -1 = invalid
    int64_t table_off;     // byte offset of the faB2 frame-size table payload, -1 = none
    int32_t blocksize;     // nominal (STREAMINFO min == max), 0 if variable
    int32_t channels;
    int32_t bps;
    int32_t table_entries;
};

// ---- metadata chain ---------------------------------------------------------------------------
FA_D void parse_stream_meta(const uint8_t* buf, int64_t nbytes, StreamMeta& m) {
    m.first_frame = -1;
    m.table_off = -1;
    m.blocksize = 0;
    m.channels = 0;
    m.bps = 0;
    m.table_entries = 0;
    if (nbytes < 8 + 34) return;
    if (buf[0] != 'f' || buf[1] != 'L' || buf[2] != 'a' || buf[3] != 'C') return;
    int64_t pos = 4;
    bool have_si = false;
    for (;;) {
        if (pos + 4 > nbytes) return;
        int last = buf[pos] >> 7, type = buf[pos] & 0x7F;
        int64_t len = ((int64_t)buf[pos + 1] << 16) | ((int64_t)buf[pos + 2] << 8) | buf[pos + 3];
        pos += 4;
        if (pos + len > nbytes) return;
        if (type == 0 && len >= 34) {
            const uint8_t* s = buf + pos;
            int minb = (s[0] << 8) | s[1], maxb = (s[2] << 8) | s[3];
            m.blocksize = (minb == maxb) ? minb : 0;
            m.channels = ((s[12] >> 1) & 7) + 1;
            m.bps = (((s[12] & 1) << 4) | (s[13] >> 4)) + 1;
            have_si = true;
        } else if (type == 2 && len >= 8 && buf[pos] == 'f' && buf[pos + 1] == 'a' && buf[pos + 2] == 'B' &&
                   buf[pos + 3] == '2') {
            // application block written by this library: u32 entry count, then 3 bytes per frame
            int64_t cnt = ((int64_t)buf[pos + 4] << 24) | ((int64_t)buf[pos + 5] << 16) | ((int64_t)buf[pos + 6] << 8) |
                          buf[pos + 7];
            if (8 + 3 * cnt <= len) {
                m.table_off = pos + 8;
                m.table_entries = (int32_t)cnt;
            }
        }
        pos += len;
        if (last) break;
    }
    if (have_si) m.first_frame = pos;
}

// ---- residual + prediction, general path --------------------------------------------------------
struct Residual {
    int plen;       // 4 or 5
    int esc;        // 15 or 31
    int porder;
    int psize;      // blocksize >> porder
    int part;       // index of the current partition
    int left;       // samples left in the current partition
    int k;          // Rice parameter of the current partition, or -1 = escaped
    int rawbits;
};

FA_D bool residual_begin(BitRd& br, int bs, int order, Residual& rs) {
    uint32_t method = br_read(br, 2);
    if (method > 1) return false;
    rs.plen = method == 0 ? 4 : 5;
    rs.esc = method == 0 ? 15 : 31;
    rs.porder = (int)br_read(br, 4);
    rs.psize = bs >> rs.porder;
    if (rs.porder > 0 && (rs.psize << rs.porder) != bs) return false;
    if (rs.psize < order && rs.porder > 0) return false;
    rs.part = -1;
    rs.left = 0;
    rs.k = 0;
    rs.rawbits = 0;
    return true;
}

FA_D int64_t residual_next(BitRd& br, int order, Residual& rs) {
    while (rs.left == 0) {  // open the next partition (a partition may be empty: psize == order)
        rs.part++;
        if (rs.part >= (1 << rs.porder)) { br.err = 1; return 0; }
        rs.left = rs.psize - (rs.part == 0 ? order : 0);
        int k = (int)br_read(br, rs.plen);
        if (k == rs.esc) {
            rs.k = -1;
            rs.rawbits = (int)br_read(br, 5);
        } else {
            rs.k = k;
        }
    }
    rs.left--;
    if (rs.k < 0) return br_read_signed(br, rs.rawbits);
    uint32_t q = br_unary(br);
    uint32_t low = br_read(br, rs.k);
    uint64_t u = ((uint64_t)q << rs.k) | low;
    return (int64_t)(u >> 1) ^ -(int64_t)(u & 1);
}

// Destination of decoded samples of one frame: out[(i - lo_base) * nch + c] for i in [lo, hi).
struct FrameOut {
    int32_t* base;  // address of (frame sample 0, channel 0); only dereferenced for i in [lo, hi)
    int nch;
    int lo, hi;
};

// Store sample i of subframe `c` applying the stereo reconstruction of channel assignment `ca`
// (RFC 9639 4.2).  Channel 0 is always written before channel 1 by the same thread.
FA_D void store_sample(const FrameOut& fo, int ca, int c, int i, int64_t v) {
    if (i < fo.lo || i >= fo.hi) return;
    int32_t* p = fo.base + (int64_t)i * fo.nch;
    if (c == 0) {
        p[0] = (int32_t)v;  // for side/right this keeps the low 32 bits of the 33-bit side
        return;
    }
    if (ca == 8) {          // left/side: right = left - side
        p[1] = (int32_t)((int64_t)p[0] - v);
    } else if (ca == 9) {   // side/right: left = side + right (mod 2^32 arithmetic is exact here)
        p[0] = (int32_t)((uint32_t)p[0] + (uint32_t)v);
        p[1] = (int32_t)v;
    } else if (ca == 10) {  // mid/side
        int64_t m = (int64_t)((uint64_t)(int64_t)p[0] << 1) | (v & 1);
        p[0] = (int32_t)((m + v) >> 1);
        p[1] = (int32_t)((m - v) >> 1);
    } else {
        p[c] = (int32_t)v;
    }
}

// Decode one subframe of `bps` bits (33 for a side channel), general path: any order, any width.
FA_D bool decode_subframe_general(BitRd& br, int bs, int bps, const FrameOut& fo, int ca, int c) {
    if (br_read(br, 1) != 0) return false;
    int type = (int)br_read(br, 6);
    int wasted = 0;
    if (br_read(br, 1)) wasted = (int)br_unary(br) + 1;
    bps -= wasted;
    if (bps <= 0 || br.err) return false;
    if (type == 0) {
        int64_t v = (int64_t)((uint64_t)br_read_signed(br, bps) << wasted);
        for (int i = fo.lo; i < fo.hi; ++i) store_sample(fo, ca, c, i, v);
        return !br.err;
    }
    if (type == 1) {
        for (int i = 0; i < bs; ++i) {
            int64_t v = (int64_t)((uint64_t)br_read_signed(br, bps) << wasted);
            store_sample(fo, ca, c, i, v);
        }
        return !br.err;
    }
    int order, shift = 0;
    int32_t coef[kMaxLpcOrder];
    int64_t hist[kMaxLpcOrder];  // circular: sample i lives at hist[i & 31]
    bool lpc = type >= 32;
    if (lpc) order = (type & 31) + 1;
    else if (type >= 8 && type <= 12) order = type - 8;
    else return false;
    if (order > bs) return false;
    for (int i = 0; i < order; ++i) {
        int64_t v = br_read_signed(br, bps);
        hist[i & 31] = v;
        store_sample(fo, ca, c, i, (int64_t)((uint64_t)v << wasted));
    }
    if (lpc) {
        int prec = (int)br_read(br, 4) + 1;
        if (prec == 16) return false;
        shift = (int)br_read_signed(br, 5);
        if (shift < 0) return false;
        for (int j = 0; j < order; ++j) coef[j] = (int32_t)br_read_signed(br, prec);
    } else {
        const int32_t fx[5][4] = {{0, 0, 0, 0}, {1, 0, 0, 0}, {2, -1, 0, 0}, {3, -3, 1, 0}, {4, -6, 4, -1}};
        for (int j = 0; j < order; ++j) coef[j] = fx[order][j];
    }
    Residual rs;
    if (!residual_begin(br, bs, order, rs)) return false;
    for (int i = order; i < bs; ++i) {
        int64_t r = residual_next(br, order, rs);
        // (wrapping arithmetic: a valid stream keeps |sum| < 2^53, but a damaged one can feed any history, and signed
        // overflow is undefined behaviour; such a frame fails its CRC-16 anyway)
        uint64_t sum = 0;
        for (int j = 0; j < order; ++j) sum += (uint64_t)(int64_t)coef[j] * (uint64_t)hist[(i - 1 - j) & 31];
        int64_t v = (int64_t)((uint64_t)r + (uint64_t)((int64_t)sum >> shift));
        hist[i & 31] = v;
        store_sample(fo, ca, c, i, (int64_t)((uint64_t)v << wasted));
        if (br.err) return false;
    }
    return !br.err;
}

// Running CRC-16 over [p, p + n) (byte-wise; used by the verifying / fallback paths only).
FA_D uint32_t crc16_bytes(const CrcTables* t, const uint8_t* p, int64_t n) {
    uint32_t c = 0;
    for (int64_t i = 0; i < n; ++i) c = crc16_byte(t, c, p[i]);
    return c;
}

// Decode the frame at `p` (window end `end`).  Returns the frame length in bytes, or -1.
// expect_nch / expect_bps: what the stream must carry (flacarray: 1|2 channels, 32 bps).  Samples [lo, hi) of the frame are
// stored from out_base on; an empty range (discard mode: out_base may be null) decodes and checks the whole frame all the
// same.
FA_D int64_t decode_frame_general(const uint8_t* p, const uint8_t* end, const CrcTables* t, int si_bps, int expect_nch,
                                  FrameHdr& fh, int32_t* out_base, int lo, int hi, bool check_crc16) {
    if (!parse_frame_header(p, end - p, t, fh)) return -1;
    int bps = fh.bps ? fh.bps : si_bps;
    if (fh.nch != expect_nch || bps != 32) return -1;
    BitRd br;
    br_init(br, p + fh.hdr_bytes, end);
    FrameOut fo;
    fo.base = out_base;
    fo.nch = fh.nch;
    fo.lo = lo < 0 ? 0 : lo;
    fo.hi = hi > fh.blocksize ? fh.blocksize : hi;
    int ca = fh.ca;
    int bps0 = bps + (ca == 9 ? 1 : 0);
    int bps1 = bps + ((ca == 8 || ca == 10) ? 1 : 0);
    if (!decode_subframe_general(br, fh.blocksize, bps0, fo, ca, 0)) return -1;
    if (fh.nch == 2 && !decode_subframe_general(br, fh.blocksize, bps1, fo, ca, 1)) return -1;
    int64_t bits = br_pos(br);
    int64_t len = fh.hdr_bytes + ((bits + 7) >> 3) + 2;
    if (p + len > end) return -1;
    if (check_crc16) {
        uint32_t want = ((uint32_t)p[len - 2] << 8) | p[len - 1];
        if (crc16_bytes(t, p, len - 2) != want) return -1;
    }
    return len;
}

}  // namespace fa

// =================================================================================================
// Kernel bodies (thin __global__ wrappers in fa_api.cu map thread indices onto these).
// =================================================================================================
namespace fa {

struct DecParams {
    const uint8_t* bytes;
    const long long* starts;   // [n_sel] byte offset of every selected stream
    const long long* nbytes;   // [n_sel]
    int64_t n_sel, stream_size;
    int nch;
    int64_t first, n_decode;   // sample window [first, first + n_decode)
    int32_t* data;             // [n_sel][n_decode][nch]
    const CrcTables* crc;
    StreamMeta* meta;          // [n_sel]
    long long* frame_off;      // [n_sel][nframes_cap + 1] byte offsets relative to the stream start, -1 = unknown
    int nframes_cap;
    int* stream_flag;          // [n_sel] 0 = ok, !=0 = needs the sequential walker
    int* err;
    int verify_crc16;
    const unsigned char* frame_flag;  // optional [n_sel][nframes_cap]: when set, frame_body only decodes flagged frames
    // optional [n_sel] (fab_decode_isolated, fab_verify): when set, a stream that cannot be decoded reports its
    // ERROR_DECODE_INIT / ERROR_DECODE_PROCESS bit here instead of in *err; meta writes every entry, the walker its failures
    int* status = nullptr;
};

// a stream-fatal error of stream k: its own status entry, or the call's error mask
FA_D void stream_failed(const DecParams& P, int64_t k, int bit) {
    if (P.status) P.status[k] = bit;
    else atom_or_global(P.err, bit);
}

// number of frames / size of frame j for a fixed-blocksize stream
FA_D int64_t frames_in_stream(int64_t stream_size, int bs) { return (stream_size + bs - 1) / bs; }

// ---- host-side sizing of a decode call ------------------------------------------------------------------------------
// The blocksize hint: STREAMINFO's min blocksize of the call's first stream, 0 when its bytes do not start with one.
inline int stream_blocksize_hint(const uint8_t* s, int64_t nbytes) {
    return nbytes >= 12 && memcmp(s, "fLaC", 4) == 0 ? (s[8] << 8) | s[9] : 0;
}

// The hinted blocksize *bsh (4096 without a hint, at least 16: the smallest legal blocksize) and the frame-table rows of a
// stream slot *cap.  The item space of a call has the frames of the hinted blocksize; a stream whose blocksize needs more
// frames than that goes to the walker.  Returns kErrAlloc for a table of more than 2^26 frames per stream.
inline int dec_frames_cap(int64_t stream_size, int blocksize_hint, int* bsh, int* cap) {
    int b = blocksize_hint > 0 ? blocksize_hint : 4096;
    if (b < 16) b = 16;
    const int64_t c = (stream_size + b - 1) / b;
    if (c > (1 << 26)) return kErrAlloc;
    *bsh = b;
    *cap = (int)c;
    return 0;
}

// Per-window sample ranges (fab_decode_windows).  Window w reads samples [first[w], last[w]) of stream slot stream[w] and
// writes them from output element out[w] on.  Its work items are the frames the window overlaps for the hinted
// blocksize `bsh`; item0 is the exclusive prefix of those counts, so an item finds its window by a binary search and
// windows of any length share warps.  Records that fail win_valid have no items.
struct WinParams {
    const long long* stream;   // [n_win] stream slot u in [0, n_sel)
    const long long* first;    // [n_win]
    const long long* last;     // [n_win]
    const long long* out;      // [n_win] output element of the window's first sample
    const long long* item0;    // [n_win + 1] first work item of every window; item0[n_win] = number of items
    int64_t n_win;
    int bsh;
};

FA_D bool win_valid(const WinParams& W, int64_t w, int64_t n_sel, int64_t stream_size) {
    const long long u = W.stream[w], a = W.first[w], b = W.last[w];
    return u >= 0 && u < n_sel && a >= 0 && b <= stream_size && a <= b;
}

// frames of [first, first + n) for blocksize bs (0 for an empty window)
FA_D int64_t frames_in_window(int64_t first, int64_t n, int64_t bs) {
    return n > 0 ? (first + n - 1) / bs - first / bs + 1 : 0;
}

// Window records -> item space (k_win_prep), one CTA of NT threads: a record that names a stream slot outside [0, n_sel)
// or a range outside the stream sets ERROR_DECODE_SAMPLE_RANGE and gets no items; W.item0 = exclusive prefix of the frame
// counts (hinted blocksize), W.item0[n_win] = the number of items.  Chunks of NT windows with a running carry.
// wpre[NT / 32], ctot: shared.
template <int NT>
FA_D void win_prep_cta(const WinParams& W, int64_t n_sel, int64_t stream_size, int* err, long long* wpre, long long* ctot) {
    long long* item0 = const_cast<long long*>(W.item0);
    const int ln = lane(), wp = warp();
    long long carry = 0;
    for (int64_t w0 = 0; w0 < W.n_win; w0 += NT) {
        const int64_t w = w0 + tid();
        long long cnt = 0;
        if (w < W.n_win) {
            if (win_valid(W, w, n_sel, stream_size)) cnt = frames_in_window(W.first[w], W.last[w] - W.first[w], W.bsh);
            else atom_or_global(err, kErrDecodeSampleRange);
        }
        long long inc = cnt;       // inclusive scan inside the warp, then over the warps' totals
        for (int d = 1; d < 32; d <<= 1) {
            long long v = (long long)shfl_up64((unsigned long long)inc, d);
            if (ln >= d) inc += v;
        }
        if (ln == 31) wpre[wp] = inc;
        sync();
        if (wp == 0) {
            const long long t = ln < NT / 32 ? wpre[ln] : 0;
            long long ti = t;
            for (int d = 1; d < 32; d <<= 1) {
                long long v = (long long)shfl_up64((unsigned long long)ti, d);
                if (ln >= d) ti += v;
            }
            if (ln < NT / 32) wpre[ln] = ti - t;
            if (ln == 31) *ctot = ti;
        }
        sync();
        if (w < W.n_win) item0[w] = carry + wpre[wp] + inc - cnt;
        carry += *ctot;
        sync();                    // (wpre / ctot are rewritten by the next chunk)
    }
    if (tid() == 0) item0[W.n_win] = carry;
}

// One work item of the decoder's index space: frame `jrel` (counted from the window's first frame) of the window
// [first, first + n) of stream slot k, whose sample `first` goes to output element `out`.  k < 0: no item.
struct WorkItem {
    int64_t k, jrel, first, n, out, nwin;
};

// WIN = false: fab_decode's uniform case, every selected stream with the same window and nwin items each, packed rows.
// WIN = true: the windows of W.
template <bool WIN>
FA_D WorkItem resolve_item(const DecParams& D, const WinParams& W, int64_t nwin, int64_t idx) {
    WorkItem it;
    if constexpr (!WIN) {
        it.k = idx / nwin;
        it.jrel = idx % nwin;
        it.first = D.first;
        it.n = D.n_decode;
        it.out = it.k * D.n_decode;
        it.nwin = nwin;
        if (it.k >= D.n_sel) it.k = -1;
    } else {
        it.k = -1;
        it.jrel = it.first = it.n = it.out = it.nwin = 0;
        if (idx >= W.item0[W.n_win]) return it;
        int64_t lo = 0, hi = W.n_win - 1;      // last window whose first item is <= idx (empty windows share it with the next)
        while (lo < hi) {
            const int64_t mid = (lo + hi + 1) >> 1;
            if (W.item0[mid] <= idx) lo = mid;
            else hi = mid - 1;
        }
        it.k = W.stream[lo];
        it.jrel = idx - W.item0[lo];
        it.first = W.first[lo];
        it.n = W.last[lo] - it.first;
        it.out = W.out[lo];
        it.nwin = W.item0[lo + 1] - W.item0[lo];
    }
    return it;
}

// ---- stage 1: one thread per selected stream: metadata + (if present) the faB2 frame-size table ----
FA_D void meta_body(const DecParams& P, int64_t k) {
    const uint8_t* buf = P.bytes + P.starts[k];
    StreamMeta m;
    parse_stream_meta(buf, P.nbytes[k], m);
    P.meta[k] = m;
    long long* fo = P.frame_off + k * (int64_t)(P.nframes_cap + 1);
    int flag = 0;
    if (P.status) P.status[k] = 0;
    if (m.first_frame < 0 || m.channels != P.nch || m.bps != 32) {
        stream_failed(P, k, kErrDecodeInit);
        flag = 4;  // undecodable
    } else if (m.blocksize <= 0) {
        flag = 1;  // variable blocksize: sequential walker
    } else {
        int64_t nf = frames_in_stream(P.stream_size, m.blocksize);
        if (nf > P.nframes_cap) {
            flag = 1;
        } else if (m.table_off >= 0 && m.table_entries == nf) {
            long long pos = m.first_frame;
            const uint8_t* tb = buf + m.table_off;
            for (int64_t j = 0; j < nf; ++j) {
                fo[j] = pos;
                pos += ((long long)tb[3 * j] << 16) | ((long long)tb[3 * j + 1] << 8) | tb[3 * j + 2];
            }
            fo[nf] = pos;
            if (pos != P.nbytes[k]) flag = 1;
        } else {
            for (int64_t j = 0; j <= nf; ++j) fo[j] = -1;
            fo[nf] = P.nbytes[k];
            flag = 0;
        }
    }
    P.stream_flag[k] = flag;
}

// ---- stage 1 as the product runs it (k_dec_meta): one warp per stream.  Lane 0 walks the (short) metadata chain; the
// frame-size table of streams written by this library is then turned into frame offsets by the whole warp (coalesced
// 3-byte reads, warp scan) instead of a serial loop per stream.  Same results as meta_body, the reference for the rules.
FA_D void meta_warp(const DecParams& P, int64_t k) {
    const int ln = lane();
    const uint8_t* buf = P.bytes + P.starts[k];
    const long long nb = P.nbytes[k];
    StreamMeta m;
    if (ln == 0) {
        parse_stream_meta(buf, nb, m);
        P.meta[k] = m;
    }
    m.first_frame = (int64_t)shfl64((unsigned long long)m.first_frame, 0);
    m.table_off = (int64_t)shfl64((unsigned long long)m.table_off, 0);
    m.blocksize = (int32_t)shfl((uint32_t)m.blocksize, 0);
    m.channels = (int32_t)shfl((uint32_t)m.channels, 0);
    m.bps = (int32_t)shfl((uint32_t)m.bps, 0);
    m.table_entries = (int32_t)shfl((uint32_t)m.table_entries, 0);
    long long* fo = P.frame_off + k * (int64_t)(P.nframes_cap + 1);
    int flag = 0;
    if (m.first_frame < 0 || m.channels != P.nch || m.bps != 32) {
        if (ln == 0) stream_failed(P, k, kErrDecodeInit);
        flag = 4;  // undecodable
    } else if (m.blocksize <= 0) {
        flag = 1;  // variable blocksize: sequential walker
    } else {
        const int64_t nf = frames_in_stream(P.stream_size, m.blocksize);
        if (nf > P.nframes_cap) {
            flag = 1;
        } else if (m.table_off >= 0 && m.table_entries == nf) {
            const uint8_t* tb = buf + m.table_off;
            long long pos = m.first_frame;      // offset of frame j0 (warp-uniform carry)
            for (int64_t j0 = 0; j0 < nf; j0 += 32) {
                const int64_t j = j0 + ln;
                long long len = 0;
                if (j < nf) len = ((long long)tb[3 * j] << 16) | ((long long)tb[3 * j + 1] << 8) | tb[3 * j + 2];
                long long inc = len;
                for (int d = 1; d < 32; d <<= 1) {
                    long long v = (long long)shfl_up64((unsigned long long)inc, d);
                    if (ln >= d) inc += v;
                }
                if (j < nf) fo[j] = pos + inc - len;
                pos += (long long)shfl64((unsigned long long)inc, 31);
            }
            if (ln == 0) fo[nf] = pos;
            if (pos != nb) flag = 1;
        } else {
            for (int64_t j = ln; j < nf; j += 32) fo[j] = -1;
            if (ln == 0) fo[nf] = nb;
        }
    }
    if (ln == 0) {
        P.stream_flag[k] = flag;
        if (P.status && flag != 4) P.status[k] = 0;
    }
}

// ---- stage 2 (foreign streams only): test byte position p of stream k for a frame header -----------
FA_D void sync_body(const DecParams& P, int64_t k, int64_t p) {
    const StreamMeta m = P.meta[k];
    if (P.stream_flag[k] != 0 || m.table_off >= 0) return;
    const uint8_t* buf = P.bytes + P.starts[k];
    int64_t nb = P.nbytes[k];
    if (p < m.first_frame || p + 6 > nb) return;
    if (buf[p] != 0xFF || (buf[p + 1] & 0xFF) != 0xF8) return;  // fixed-blocksize sync code
    FrameHdr fh;
    if (!parse_frame_header(buf + p, nb - p, P.crc, fh)) return;
    int64_t nf = frames_in_stream(P.stream_size, m.blocksize);
    if ((int64_t)fh.number >= nf || fh.nch != P.nch) return;
    int bps = fh.bps ? fh.bps : m.bps;
    if (bps != 32) return;
    int64_t want_bs = ((int64_t)fh.number == nf - 1) ? (P.stream_size - (nf - 1) * m.blocksize) : m.blocksize;
    if (fh.blocksize != want_bs) return;
    long long* fo = P.frame_off + k * (int64_t)(P.nframes_cap + 1);
    long long prev = atom_cas_global64(&fo[fh.number], -1, p);
    if (prev != -1 && prev != p) atom_or_global(&P.stream_flag[k], 2);  // two candidates for one frame
}

// The scan itself, warp-cooperative: warp `w` of `nw` takes rows of 32 aligned 16-byte chunks of stream k (one
// coalesced 512-byte load per row), every lane finds the positions of the byte pair FF F8 inside its chunk with
// branch-free byte-parallel arithmetic (exact zero-byte masks of ~w and w ^ F8F8F8F8, the second shifted down one
// byte through a funnel shift that pulls in the first byte of the next word / next lane's chunk) and hands the
// candidates -- one per frame plus ~one false hit per 64 KB -- to sync_body.  ~3 instructions per byte.
FA_D uint32_t zero_bytes(uint32_t v) {      // 0x80 in every byte of v that is zero (exact)
    const uint32_t t = (v & 0x7F7F7F7Fu) + 0x7F7F7F7Fu;
    return ~(t | v | 0x7F7F7F7Fu);
}
FA_D void sync_scan_warp(const DecParams& P, int64_t k, int64_t w, int64_t nw) {
    if (P.stream_flag[k] != 0 || P.meta[k].table_off >= 0) return;
    const int ln = lane();
    const int64_t nb = P.nbytes[k];
    const uint8_t* buf = P.bytes + P.starts[k];
    const int64_t head = (int64_t)((uintptr_t)buf & 15);
    const uint8_t* abase = buf - head;                    // (aligned chunks: the first / last one may hold a neighbour's bytes)
    const int64_t n16 = (head + nb + 15) >> 4;
    for (int64_t row = w; (row << 5) < n16; row += nw) {
        const int64_t ci = (row << 5) + ln;
        U4 q; q.x = q.y = q.z = q.w = 0;
        if (ci < n16) q = ldg128(abase + (ci << 4));
        uint32_t nxt = shfl_down(q.x, 1);                 // first word of the chunk behind this one
        if (ln == 31) nxt = ci + 1 < n16 ? (uint32_t)abase[(ci + 1) << 4] : 0u;
        const uint32_t f0 = zero_bytes(~q.x), f1 = zero_bytes(~q.y), f2 = zero_bytes(~q.z), f3 = zero_bytes(~q.w);
        const uint32_t e0 = zero_bytes(q.x ^ 0xF8F8F8F8u), e1 = zero_bytes(q.y ^ 0xF8F8F8F8u),
                       e2 = zero_bytes(q.z ^ 0xF8F8F8F8u), e3 = zero_bytes(q.w ^ 0xF8F8F8F8u);
        const uint32_t e4 = zero_bytes((nxt & 0xFFu) ^ 0xF8u) & 0x80u;
        // byte i is FF and byte i + 1 is F8 (little-endian words: the next byte sits 8 bits higher)
        uint32_t c[4];
        c[0] = f0 & funnel_r(e0, e1, 8);
        c[1] = f1 & funnel_r(e1, e2, 8);
        c[2] = f2 & funnel_r(e2, e3, 8);
        c[3] = f3 & funnel_r(e3, e4, 8);
        if ((c[0] | c[1] | c[2] | c[3]) != 0) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                uint32_t m = c[j];
                while (m) {
                    const int b = (31 - clz32(m)) >> 3;       // byte index inside the word
                    m &= ~(0x80u << (8 * b));
                    sync_body(P, k, (ci << 4) + 4 * j + b - head);
                }
            }
        }
    }
}

// ---- stage 3: one thread per (selected stream, frame overlapping the sample window) ---------------
// (frame j of stream k for the window [first, first + n) that starts at output element `out`)
FA_D void frame_body(const DecParams& P, int64_t k, int64_t j, int64_t first, int64_t n, int64_t out) {
    if (P.stream_flag[k] != 0) return;
    if (P.frame_flag && !P.frame_flag[k * (int64_t)P.nframes_cap + j]) return;
    const StreamMeta m = P.meta[k];
    const long long* fo = P.frame_off + k * (int64_t)(P.nframes_cap + 1);
    long long off = fo[j], next = fo[j + 1];
    if (off < 0) { atom_or_global(&P.stream_flag[k], 2); return; }
    const uint8_t* buf = P.bytes + P.starts[k];
    const uint8_t* end = buf + P.nbytes[k];
    int64_t s0 = j * (int64_t)m.blocksize;  // first sample of the frame
    int32_t* base = P.data + (P.data ? (out + (s0 - first)) * P.nch : 0);
    int64_t lo = first - s0, hi = first + n - s0;
    if (!P.data) hi = lo;                   // discard mode (fab_verify): decode and check, store nothing
    FrameHdr fh;
    int64_t len = decode_frame_general(buf + off, end, P.crc, m.bps, P.nch, fh, base,
                                       (int)(lo < 0 ? 0 : lo), (int)(hi > m.blocksize ? m.blocksize : hi),
                                       P.verify_crc16 != 0);
    bool ok = len > 0 && (int64_t)fh.number == j && !fh.variable;
    if (ok && next >= 0 && off + len != next) ok = false;
    if (!ok) atom_or_global(&P.stream_flag[k], 2);
}
FA_D void frame_body(const DecParams& P, int64_t k, int64_t j) { frame_body(P, k, j, P.first, P.n_decode, k * P.n_decode); }

// Work item idx of the call's index space (resolve_item) through the general decoder (k_dec_frames, after the tile path:
// P.frame_flag set, so only the frames it flagged are decoded).
template <bool WIN>
FA_D void frames_item(const DecParams& P, const WinParams& W, int64_t nwin, int64_t idx) {
    const WorkItem it = resolve_item<WIN>(P, W, nwin, idx);
    const int64_t k = it.k;
    if (k < 0) return;
    if (P.stream_flag[k] != 0) return;
    int bs = P.meta[k].blocksize;
    int64_t j0 = it.first / bs, j1 = (it.first + it.n - 1) / bs;
    if (j1 - j0 + 1 > it.nwin) {  // blocksize differs from the host's hint: leave the stream to the walker
        if (it.jrel == 0) atom_or_global(&P.stream_flag[k], 1);
        return;
    }
    int64_t j = j0 + it.jrel;
    if (j > j1) return;
    frame_body(P, k, j, it.first, it.n, it.out);
}

// (a template: the stores of fab_decode's walker stay what they were; register allocation there is sensitive to them)
template <bool ISO>
FA_D void walker_failed(const DecParams& P, int64_t k) {
    if constexpr (ISO) P.status[k] = kErrDecodeProcess;
    else atom_or_global(P.err, kErrDecodeProcess);
}

// ---- stage 4: sequential walker for streams the parallel path could not index -----------------------
// (variable blocksize, ambiguous sync candidates, failed chain check).  Always verifies CRC-16.
// Decodes the window [first, first + n) of stream k to output element `out` on.  ISO (fab_decode_isolated, fab_verify;
// P.status set): a failure goes to the stream's status entry instead of the call's error mask, and P.data may be null
// (discard mode: decode and check, store nothing).  ISO = false is fab_decode's and fab_decode_windows' walker.
template <bool ISO = false>
FA_D void walker_body(const DecParams& P, int64_t k, int64_t first, int64_t n, int64_t out) {
    int flag = P.stream_flag[k];
    if (flag == 0 || flag == 4) return;
    const StreamMeta m = P.meta[k];
    const uint8_t* buf = P.bytes + P.starts[k];
    const uint8_t* end = buf + P.nbytes[k];
    int64_t pos = m.first_frame, sample = 0, last = first + n;
    uint64_t expect = 0;
    while (sample < last) {
        if (pos >= P.nbytes[k]) { walker_failed<ISO>(P, k); return; }
        FrameHdr fh;
        int32_t* base = nullptr;
        int64_t lo = first - sample, hi = last - sample;
        if (!ISO || P.data) base = P.data + (out + (sample - first)) * P.nch;
        else hi = lo;                       // discard mode
        int64_t len = decode_frame_general(buf + pos, end, P.crc, m.bps, P.nch, fh, base, (int)(lo < 0 ? 0 : lo),
                                           (int)(hi > 65536 ? 65536 : hi), true);
        if (len < 0) { walker_failed<ISO>(P, k); return; }
        if (fh.variable ? ((int64_t)fh.number != sample) : (fh.number != expect)) {
            walker_failed<ISO>(P, k);
            return;
        }
        expect++;
        sample += fh.blocksize;
        pos += len;
    }
}
template <bool ISO = false>
FA_D void walker_body(const DecParams& P, int64_t k) { walker_body<ISO>(P, k, P.first, P.n_decode, k * P.n_decode); }

// fab_decode_windows' walker (k_dec_walker_win): window w of a stream the parallel path left to it
FA_D void walker_win(const DecParams& P, const WinParams& W, int64_t w) {
    if (!win_valid(W, w, P.n_sel, P.stream_size)) return;
    const long long first = W.first[w], n = W.last[w] - first;
    if (n > 0) walker_body(P, W.stream[w], first, n, W.out[w]);
}

// fab_decode_isolated, after the walker and the restore (k_dec_fill_failed): elements i0, i0 + stride, ... of the output row
// of stream s are overwritten with `fill` when its status is not 0.  W is the output element (uint32_t for int32 / float32,
// unsigned long long for int64 / float64).
template <typename W>
FA_D void fill_failed(const int* FA_RESTRICT status, W* out, int64_t n_per_stream, W fill, int64_t s, int64_t i0,
                      int64_t stride) {
    if (status[s] == 0) return;
    W* o = out + s * n_per_stream;
    for (int64_t i = i0; i < n_per_stream; i += stride) o[i] = fill;
}

}  // namespace fa
