"""A strict reader of the streams this library's encoder writes.  TEST INFRASTRUCTURE ONLY.

`read_stream(buf, level, stream_size, nch)` parses one stream and returns its syntax as records (STREAMINFO, the faB2
frame-size table, and per frame the header fields and per subframe every syntax element, the residuals and the decoded
samples).  On the first violation it raises `StrictError` naming the stream, the frame, the channel and the field.

It checks what RFC 9639 demands, what libFLAC's decoder refuses (a residual or a sample outside the subframe's bit
depth, an LPC shift outside 0..15, a coefficient precision of 16) and what the library itself documents (DESIGN.md
section 3: STREAMINFO fields, the faB2 table, fixed blocking, independent channels, frame and subframe sizes).  The
encoder's own documented rules for its choices (Rice parameters, partition orders, fixed orders) are checked by
`check_choices` on the records.

It shares no code with oracle/flac_oracle.c, oracle/flac_writer.py or flacarray_b200/csrc: a bug in either cannot hide
one in the encoder.  Plain Python with numpy for the vector parts; the Rice decoder is a per-sample loop.
"""
from dataclasses import dataclass, field

import numpy as np

# level -> (blocksize, max LPC order, max partition order, LPC coefficient precision): fa_encode.h level_preset and the
# precision rule of fab_encode (13 / 14 / 15 bits for blocksizes <= 384 / <= 1152 / larger)
PRESETS = {0: (1152, 0, 3, 14), 1: (1152, 0, 3, 14), 2: (1152, 0, 3, 14), 3: (4096, 6, 4, 15), 4: (4096, 8, 4, 15),
           5: (4096, 8, 5, 15), 6: (4096, 8, 6, 15), 7: (4096, 12, 6, 15), 8: (4096, 12, 6, 15)}
NARROW = 1 << 22          # fa_encode.h kNarrowBits: the 32-bit datapath's sample range
FIXED_COEFS = ((), (1,), (2, -1), (3, -3, 1), (4, -6, 4, -1))
_BS_CODE = {192: 1, 576: 2, 1152: 3, 2304: 4, 4608: 5, 256: 8, 512: 9, 1024: 10, 2048: 11, 4096: 12, 8192: 13,
            16384: 14, 32768: 15}


class StrictError(AssertionError):
    pass


def _tables():
    t8, t16 = [], []
    for i in range(256):
        c = i
        for _ in range(8):
            c = ((c << 1) ^ 0x07) & 0xFF if c & 0x80 else (c << 1) & 0xFF
        t8.append(c)
        c = i << 8
        for _ in range(8):
            c = ((c << 1) ^ 0x8005) & 0xFFFF if c & 0x8000 else (c << 1) & 0xFFFF
        t16.append(c)
    return t8, t16


_T8, _T16 = _tables()


def crc8(b):
    c = 0
    for x in b:
        c = _T8[c ^ x]
    return c


def crc16(b):
    c = 0
    for x in b:
        c = ((c << 8) & 0xFFFF) ^ _T16[(c >> 8) ^ x]
    return c


def stream_header_bytes(nframes):
    return 4 + 4 + 34 + 4 + 8 + 3 * nframes


def slot_bytes(bs, nch):
    """The worst-case frame the encoder reserves (fab_encode_bound, the slot size of fa_api.cu)."""
    return 16 + 2 + nch * (4 * bs + 8)


def rice_param(s, n):
    """The encoder's Rice parameter of a partition of n residuals with sum |r| = s (fa_encode.h rice_estimate,
    rice_search_warp): the smallest k in 0..30 with n * 2^k >= s."""
    k = 0
    while k < 30 and (n << k) < s:
        k += 1
    return k


def rice_bits(s, n):
    """The encoder's size estimate of such a partition (libFLAC set_partitioned_rice_ estimate mode), capped at 2^25."""
    k = rice_param(s, n)
    pb = 4 + (1 + k) * n + ((s >> (k - 1)) if k else (s << 1)) - (n >> 1)
    return min(pb, 1 << 25), k


def fixed_order(fe, bad=0):
    """libFLAC FLAC__fixed_compute_best_predictor's choice from the five error sums (fa_encode.h design_fixed); orders
    in `bad` are excluded."""
    te = [(1 << 64) - 1 if (bad >> k) & 1 else int(fe[k]) for k in range(5)]
    m34 = min(te[3], te[4])
    m234 = min(te[2], m34)
    m1234 = min(te[1], m234)
    if te[0] < m1234:
        return 0
    if te[1] < m234:
        return 1
    if te[2] < m34:
        return 2
    if te[3] < te[4]:
        return 3
    return 4


@dataclass
class Subframe:
    kind: str                 # "constant", "verbatim", "fixed", "lpc"
    order: int = 0
    wasted: int = 0
    warmup: tuple = ()
    precision: int = 0
    shift: int = 0
    coefs: tuple = ()
    method: int = -1          # residual coding method (0 RICE, 1 RICE2), -1 for CONSTANT / VERBATIM
    porder: int = -1
    params: list = field(default_factory=list)     # per partition: Rice parameter, or ("esc", width)
    residual: np.ndarray = None                     # int64, the coded residuals (after the warm-up)
    samples: np.ndarray = None                      # int64, the decoded samples (wasted bits restored)
    nbits: int = 0


@dataclass
class Frame:
    number: int
    offset: int               # byte offset in the stream
    nbytes: int
    blocksize: int
    bs_code: int
    subframes: list
    narrow_mac: list          # per channel: sum|q| * max|x| of a narrow LPC subframe, else None


@dataclass
class Stream:
    blocksize: int
    nch: int
    total_samples: int
    fab2: list
    header_bytes: int
    frames: list

    def samples(self):
        """Decoded samples [nch, n] int64."""
        return np.stack([np.concatenate([f.subframes[c].samples for f in self.frames]) for c in range(self.nch)])


class _Bits:
    """MSB-first reader over a string of '0' / '1' characters (the Rice loop then uses str.find and int(s, 2))."""

    def __init__(self, b):
        self.s = bin(int.from_bytes(b, "big") | (1 << (8 * len(b))))[3:] if len(b) else ""
        self.p = 0

    def u(self, n, err):
        if n == 0:
            return 0
        if self.p + n > len(self.s):
            err("read past the end of the frame")
        v = int(self.s[self.p:self.p + n], 2)
        self.p += n
        return v

    def s_(self, n, err):
        v = self.u(n, err)
        return v - (1 << n) if n and v >> (n - 1) else v

    def unary(self, err):
        i = self.s.find("1", self.p)
        if i < 0:
            err("unary code runs past the end of the frame")
        q = i - self.p
        self.p = i + 1
        return q


def _int_range(bits):
    return -(1 << (bits - 1)), (1 << (bits - 1)) - 1


def read_stream(buf, level, stream_size, nch, name="stream", expect=None):
    """Parse and check one stream.  buf: its bytes (exactly nbytes of them); expect: optional int array [nch, stream_size]
    of the samples the encoder was given (the low and high words of int64 as two channels, float input quantised)."""
    buf = bytes(np.asarray(buf, np.uint8).tobytes()) if not isinstance(buf, (bytes, bytearray)) else bytes(buf)
    bs_nom, max_lpc, max_porder, _ = PRESETS[level]
    where = [name, None, None]

    def err(msg, fieldname=None):
        loc = where[0]
        if where[1] is not None:
            loc += f", frame {where[1]}"
        if where[2] is not None:
            loc += f", channel {where[2]}"
        raise StrictError(f"{loc}: {fieldname + ': ' if fieldname else ''}{msg}")

    def need(cond, fieldname, msg):
        if not cond:
            err(msg, fieldname)

    nframes = -(-stream_size // bs_nom)
    need(len(buf) >= stream_header_bytes(0), "header", f"{len(buf)} bytes cannot hold the stream header")
    need(buf[:4] == b"fLaC", "magic", f"{buf[:4]!r} != b'fLaC'")
    # ---- STREAMINFO (not last), then APPLICATION faB2 (last)
    need(buf[4] == 0x00, "STREAMINFO block header", f"type / last flag byte {buf[4]:#04x} != 0x00")
    need(int.from_bytes(buf[5:8], "big") == 34, "STREAMINFO length", f"{int.from_bytes(buf[5:8], 'big')} != 34")
    si = buf[8:42]
    min_bs, max_bs = int.from_bytes(si[0:2], "big"), int.from_bytes(si[2:4], "big")
    need(min_bs == bs_nom and max_bs == bs_nom, "STREAMINFO blocksize", f"min {min_bs} max {max_bs} != {bs_nom}")
    min_fs, max_fs = int.from_bytes(si[4:7], "big"), int.from_bytes(si[7:10], "big")
    v = int.from_bytes(si[10:18], "big")
    rate, si_nch, si_bps, total = v >> 44, ((v >> 41) & 7) + 1, ((v >> 36) & 31) + 1, v & ((1 << 36) - 1)
    need(rate == 44100, "STREAMINFO sample rate", f"{rate} != 44100")
    need(si_nch == nch, "STREAMINFO channels", f"{si_nch} != {nch}")
    need(si_bps == 32, "STREAMINFO bits per sample", f"{si_bps} != 32")
    need(total == (stream_size if stream_size < (1 << 36) else 0), "STREAMINFO total samples", f"{total} != {stream_size}")
    need(si[18:34] == bytes(16), "STREAMINFO MD5", "not zero")
    need(buf[42] == 0x82, "APPLICATION block header", f"type / last flag byte {buf[42]:#04x} != 0x82")
    alen = int.from_bytes(buf[43:46], "big")
    need(alen == 8 + 3 * nframes, "APPLICATION length", f"{alen} != {8 + 3 * nframes}")
    need(buf[46:50] == b"faB2", "APPLICATION id", f"{buf[46:50]!r} != b'faB2'")
    nf_tab = int.from_bytes(buf[50:54], "big")
    need(nf_tab == nframes, "faB2 frame count", f"{nf_tab} != {nframes}")
    hdr = stream_header_bytes(nframes)
    need(len(buf) >= hdr, "faB2 table", "truncated")
    fab2 = [int.from_bytes(buf[54 + 3 * j:57 + 3 * j], "big") for j in range(nframes)]
    # ---- frames
    frames = []
    pos = hdr
    sample = 0
    for j in range(nframes):
        where[1], where[2] = j, None
        need(pos < len(buf), "frame", f"missing: the stream ends after {j} of {nframes} frames")
        fr = _read_frame(buf, pos, j, bs_nom, max_lpc, max_porder, nch, stream_size - sample, err, need, where,
                         None if expect is None else np.asarray(expect)[:, sample:sample + bs_nom])
        need(fab2[j] == fr.nbytes, "faB2 frame size", f"{fab2[j]} != the frame's {fr.nbytes} bytes")
        frames.append(fr)
        pos += fr.nbytes
        sample += fr.blocksize
    where[1] = None
    need(sample == stream_size, "block sizes", f"sum {sample} != {stream_size}")
    need(pos == len(buf), "stream end", f"{len(buf) - pos} bytes after the last frame")
    if min_fs or max_fs:
        sizes = [f.nbytes for f in frames]
        need(min_fs == min(sizes) and max_fs == max(sizes), "STREAMINFO frame size", f"{min_fs}/{max_fs} != frames")
    return Stream(bs_nom, nch, total, fab2, hdr, frames)


def _read_frame(buf, pos, j, bs_nom, max_lpc, max_porder, nch, remaining, err, need, where, expect):
    # ---- header
    h0 = pos
    need(pos + 6 <= len(buf), "frame header", "truncated")
    need(buf[pos] == 0xFF and buf[pos + 1] == 0xF8, "sync / blocking", f"{buf[pos]:#04x} {buf[pos + 1]:#04x} != 0xff 0xf8")
    bs_code, sr_code = buf[pos + 2] >> 4, buf[pos + 2] & 15
    ca, ss_code, rsv = buf[pos + 3] >> 4, (buf[pos + 3] >> 1) & 7, buf[pos + 3] & 1
    need(sr_code == 9, "sample rate code", f"{sr_code} != 9 (44.1 kHz)")
    need(ss_code == 7, "sample size code", f"{ss_code} != 7 (32 bps)")
    need(rsv == 0, "frame header reserved bit", "set")
    need(ca == (0 if nch == 1 else 1), "channel assignment", f"{ca} is not independent {nch}-channel")
    p = pos + 4
    lead = buf[p]
    n = 1 if lead < 0x80 else 8 - (~lead & 0xFF).bit_length() if lead != 0xFE else 7
    need(lead < 0x80 or 2 <= n <= 7, "frame number", f"bad lead byte {lead:#04x}")
    num = lead if n == 1 else (lead & (0x7F >> n) if n < 7 else 0)
    for i in range(1, n):
        c = buf[p + i]
        need(c & 0xC0 == 0x80, "frame number", f"bad continuation byte {c:#04x}")
        num = (num << 6) | (c & 0x3F)
    need(num == j, "frame number", f"{num} != {j}")
    shortest = 1 if num < 0x80 else next(k for k, lim in ((2, 1 << 11), (3, 1 << 16), (4, 1 << 21), (5, 1 << 26),
                                                          (6, 1 << 31), (7, 1 << 36)) if num < lim)
    need(n == shortest, "frame number", f"coded in {n} bytes, not the shortest {shortest}")
    p += n
    if bs_code == 6:
        bs = buf[p] + 1
        p += 1
    elif bs_code == 7:
        bs = int.from_bytes(buf[p:p + 2], "big") + 1
        p += 2
    elif bs_code == 1:
        bs = 192
    elif 2 <= bs_code <= 5:
        bs = 576 << (bs_code - 2)
    elif bs_code >= 8:
        bs = 256 << (bs_code - 8)
    else:
        err(f"reserved code {bs_code}", "blocksize code")
    want_bs = min(bs_nom, remaining)
    need(bs == want_bs, "blocksize", f"{bs} != {want_bs}" + (" (only the last frame may be short)" if bs < want_bs else ""))
    want_code = _BS_CODE.get(bs, 6 if bs <= 256 else 7)
    need(bs_code == want_code, "blocksize code", f"{bs_code} != {want_code}, the code the encoder documents for {bs}")
    need(buf[p] == crc8(buf[h0:p]), "CRC-8", f"{buf[p]:#04x} != {crc8(buf[h0:p]):#04x}")
    p += 1
    # ---- subframes: the frame ends at the first byte boundary after them plus the CRC-16
    bits = _Bits(buf[p:])
    subs, macs = [], []
    for c in range(nch):
        where[2] = c
        x0 = bits.p
        sf = _read_subframe(bits, bs, max_lpc, max_porder, err, need,
                            None if expect is None else np.asarray(expect[c], np.int64))
        sf.nbits = bits.p - x0
        # no subframe larger than VERBATIM of the same samples plus its header (fab_encode_bound relies on it)
        verb = 8 + sf.wasted + bs * (32 - sf.wasted)
        need(sf.nbits <= verb, "subframe size", f"{sf.nbits} bits > VERBATIM's {verb}")
        if expect is not None:
            need(np.array_equal(sf.samples, np.asarray(expect[c], np.int64)), "samples",
                 f"decoded samples differ from the input from sample {int(np.argmax(sf.samples != expect[c]))}")
        xs = sf.samples >> sf.wasted
        mac = None
        if sf.kind == "lpc" and int(xs.min()) >= -NARROW and int(xs.max()) < NARROW:
            mac = sum(abs(q) for q in sf.coefs) * max(abs(int(xs.min())), abs(int(xs.max())))
        macs.append(mac)
        subs.append(sf)
    where[2] = None
    pad = (-bits.p) % 8
    need(bits.u(pad, err) == 0 if pad else True, "padding", "nonzero bits before the CRC-16")
    end = p + bits.p // 8
    need(end + 2 <= len(buf), "CRC-16", "the stream ends inside the frame")
    got = int.from_bytes(buf[end:end + 2], "big")
    need(got == crc16(buf[h0:end]), "CRC-16", f"{got:#06x} != {crc16(buf[h0:end]):#06x}")
    nbytes = end + 2 - h0
    need(nbytes <= slot_bytes(bs_nom, nch), "frame size", f"{nbytes} > the worst-case slot {slot_bytes(bs_nom, nch)}")
    return Frame(j, h0, nbytes, bs, bs_code, subs, macs)


def _read_subframe(bits, bs, max_lpc, max_porder, err, need, expect):
    need(bits.u(1, err) == 0, "subframe padding bit", "set")
    t = bits.u(6, err)
    wasted = 0
    if bits.u(1, err):
        wasted = bits.unary(err) + 1
    need(wasted < 32, "wasted bits", f"{wasted} >= bps 32")
    b = 32 - wasted
    lo, hi = _int_range(b)
    if t == 0:
        v = bits.s_(b, err)
        return Subframe("constant", wasted=wasted, samples=np.full(bs, v << wasted, np.int64))
    if t == 1:
        x = np.array([bits.s_(b, err) for _ in range(bs)], np.int64)
        return Subframe("verbatim", wasted=wasted, samples=x << wasted)
    if 8 <= t <= 12:
        kind, order = "fixed", t - 8
    elif t >= 32:
        kind, order = "lpc", t - 31
    else:
        err(f"reserved subframe type {t}", "subframe type")
    need(order <= (4 if kind == "fixed" else max_lpc), "predictor order",
         f"{kind} order {order} > {4 if kind == 'fixed' else max_lpc}")
    need(order <= bs, "predictor order", f"{order} > blocksize {bs}")
    warm = tuple(bits.s_(b, err) for _ in range(order))
    sf = Subframe(kind, order=order, wasted=wasted, warmup=warm)
    if kind == "lpc":
        pc = bits.u(4, err)
        need(pc != 15, "LPC precision", "code 15 (precision 16) is invalid")
        sf.precision = pc + 1
        sf.shift = bits.s_(5, err)
        need(0 <= sf.shift <= 15, "LPC shift", f"{sf.shift} outside 0..15")
        sf.coefs = tuple(bits.s_(sf.precision, err) for _ in range(order))
        coefs = sf.coefs
    else:
        coefs = FIXED_COEFS[order]
    # ---- residual
    sf.method = bits.u(2, err)
    need(sf.method in (0, 1), "residual method", f"reserved method {sf.method}")
    sf.porder = bits.u(4, err)
    need(sf.porder <= max_porder, "partition order", f"{sf.porder} > {max_porder}")
    need(bs % (1 << sf.porder) == 0, "partition order", f"2^{sf.porder} does not divide the blocksize {bs}")
    psize = bs >> sf.porder
    need(psize >= order, "partition order", f"first partition of {psize} samples < predictor order {order}")
    plen, esc = (4, 15) if sf.method == 0 else (5, 31)
    res = []
    for part in range(1 << sf.porder):
        n = psize - (order if part == 0 else 0)
        k = bits.u(plen, err)
        if k == esc:
            w = bits.u(5, err)
            sf.params.append(("esc", w))
            res.extend(bits.s_(w, err) for _ in range(n))
            continue
        need(k <= 30, "Rice parameter", f"{k} > 30 in partition {part}")
        sf.params.append(k)
        s = bits.s
        p = bits.p
        for _ in range(n):
            i = s.find("1", p)
            if i < 0 or i + 1 + k > len(s):
                err(f"partition {part} runs past the end of the frame", "residual")
            u = ((i - p) << k) | (int(s[i + 1:i + 1 + k], 2) if k else 0)
            res.append((u >> 1) ^ -(u & 1))
            p = i + 1 + k
        bits.p = p
    ks = [k for k in sf.params if not isinstance(k, tuple)]
    need(sf.method == 0 or any(k >= 15 for k in ks), "residual method", "RICE2 where every parameter fits 4 bits")
    r = np.array(res, np.int64)
    sf.residual = r
    if r.size:
        bad = np.flatnonzero((r < -(1 << 31)) | (r > (1 << 31) - 1))
        if bad.size:
            err(f"sample {order + int(bad[0])}: {int(r[bad[0]])} outside int32", "residual")
    # ---- reconstruction: prediction sums exactly (int64 holds |q| < 2^15 x |x| < 2^31 x 32 terms; no wrap)
    if expect is not None and order < bs:
        x = expect >> wasted
        need(np.array_equal(x << wasted, expect), "wasted bits", "the input is not a multiple of 2^wasted")
        need(tuple(int(v) for v in x[:order]) == warm, "warm-up", "differs from the input")
        pred = np.zeros(bs - order, np.int64)
        for m, cm in enumerate(coefs):
            pred += np.int64(cm) * x[order - 1 - m:bs - 1 - m]
        if kind == "lpc":
            pred >>= sf.shift
        want = x[order:] - pred
        if not np.array_equal(want, r):
            i = int(np.argmax(want != r))
            err(f"sample {order + i}: decodes to {int(pred[i]) + int(r[i])}, the input is {int(x[order + i])}", "samples")
        xs = x
    else:
        xs = list(warm)
        cl = list(coefs)
        for i in range(bs - order):
            acc = 0
            for m, cm in enumerate(cl):
                acc += cm * xs[order + i - 1 - m]
            if kind == "lpc":
                acc >>= sf.shift
            xs.append(acc + int(r[i]))
        xs = np.array(xs, np.int64) if max(map(abs, xs or [0])) < (1 << 62) else np.array(xs, object)
    if len(xs):
        mn, mx = int(np.min(xs)), int(np.max(xs))
        if mn < lo or mx > hi:
            i = int(np.argmax((np.asarray(xs) < lo) | (np.asarray(xs) > hi)))
            err(f"sample {i} = {int(xs[i])} outside {b} bits", "samples")
    sf.samples = np.asarray(xs, np.int64) << wasted
    return sf


def check_choices(st, level, records=None, name="stream"):
    """The encoder's documented rules for its choices, on a stream `st` read by read_stream (fa_encode.h,
    fa_encode_fixed.h); raises StrictError naming the stream, frame, channel and rule.  records: optional (stats
    [nframes, nch], plans [nframes, nch], fixed [nframes]) from the emulator, for the rules that refer to the plan."""
    prec_max = PRESETS[level][3]
    for j, fr in enumerate(st.frames):
        for c, sf in enumerate(fr.subframes):
            loc = f"{name}, frame {j}, channel {c}"
            if sf.kind in ("constant", "verbatim"):
                continue
            bs, order = fr.blocksize, sf.order
            # no escaped partitions; the Rice parameter of every partition from the exact sum |r| of that partition
            if any(isinstance(k, tuple) for k in sf.params):
                raise StrictError(f"{loc}: partition escape codes are never written")
            psize = bs >> sf.porder
            sums, ns = [], []
            i = 0
            for part in range(1 << sf.porder):
                n = psize - (order if part == 0 else 0)
                sums.append(int(np.abs(sf.residual[i:i + n]).sum()))
                ns.append(n)
                i += n
            for part, (s, n, k) in enumerate(zip(sums, ns, sf.params)):
                if k != rice_param(s, n):
                    raise StrictError(f"{loc}: Rice parameter of partition {part} is {k}, the rule gives "
                                      f"{rice_param(s, n)} (sum |r| = {s}, n = {n})")
            # the partition order: one of the orders the paths that can take this frame choose (see _porder_choices)
            allowed = _porder_choices(sf.residual, bs, order, level)
            if sf.porder not in allowed:
                raise StrictError(f"{loc}: partition order {sf.porder}, the rules give {sorted(allowed)}")
            # a FIXED subframe has libFLAC's order for the exact error sums of its samples
            if sf.kind == "fixed":
                fe, bad = fixed_sums(sf.samples >> sf.wasted)
                want = fixed_order(fe, bad)
                if order != want:
                    raise StrictError(f"{loc}: FIXED order {order}, the error sums {fe} give {want}")
            if sf.kind == "lpc" and sf.precision > prec_max:
                raise StrictError(f"{loc}: LPC precision {sf.precision} > the level's {prec_max}")
            # the narrow datapath's condition: a lowered precision is only ever chosen to make it hold
            mac = fr.narrow_mac[c]
            if mac is not None and sf.precision < prec_max and mac >= (1 << 30):
                raise StrictError(f"{loc}: precision lowered to {sf.precision} but sum|q| * max|x| = {mac} >= 2^30")
            if records is not None:
                stats, plans, fixed = records
                if not fixed[j] and plans[j, c]["mode"] >= 2 and plans[j, c]["wasted"] == sf.wasted:
                    pl = plans[j, c]
                    if sf.kind == "fixed" and pl["ok0"] and order != pl["ord0"]:
                        raise StrictError(f"{loc}: FIXED order {order} != the plan's {pl['ord0']}")
                    if pl["ok1"] and not pl["wide1"] and mac is not None and mac >= (1 << 30):
                        raise StrictError(f"{loc}: narrow plan with sum|q| * max|x| = {mac} >= 2^30")


def fixed_sums(x):
    """libFLAC FLAC__fixed_compute_best_predictor(_wide): sum over i >= 4 of |order-k difference|, and the orders whose
    difference leaves -(2^31 - 1) .. 2^31 - 1 somewhere (fa_encode.h fits_res)."""
    x = [int(v) for v in x]
    fe, bad = [0] * 5, 0
    if len(x) <= 4:
        return fe, bad
    d = [np.asarray(x, object)]
    for k in range(1, 5):
        d.append(d[-1][1:] - d[-1][:-1])
    for k in range(5):
        e = d[k][4 - k:]
        fe[k] = int(sum(abs(v) for v in e))
        if any(v < -((1 << 31) - 1) or v > (1 << 31) - 1 for v in e):
            bad |= 1 << k
    return fe, bad


def porder_estimate(res, bs, order, p):
    """The encoder's size estimate of the residual at partition order p: per-partition rice_bits + 6, plus one bit per
    partition when any parameter needs RICE2 (fa_encode.h rice_search_warp, enc_channel_full)."""
    psize = bs >> p
    bits, big, i = 0, False, 0
    for part in range(1 << p):
        n = psize - (order if part == 0 else 0)
        b, k = rice_bits(int(np.abs(res[i:i + n]).sum()), n)
        i += n
        bits += b
        big = big or k >= 15
    return bits + 6 + ((1 << p) if big else 0)


def max_porder_for(bs, order, level_max):
    p = 0
    while p < level_max and not (bs >> p) & 1:
        p += 1
    while p > 0 and (bs >> p) <= order:
        p -= 1
    return p


def _porder_choices(res, bs, order, level):
    """Partition orders the encoder's paths can choose for this residual:
      full 4096-sample frames (k_encode full path): the level's maximum if its estimate is strictly smaller than order
        0's, else 0;
      short frames (short path), the general path and k_enc_fixed: the order of least estimate over 0..maxp, the
        largest such order on ties, with maxp = max_porder_for(bs, order, cap) where cap is the level's maximum (general
        path, k_enc_fixed: at most 3 at levels 0..2, which is their maximum) or, on the short path, also at most
        log2(bs) - 5 (partitions of whole 32-sample thread chunks)."""
    level_max = PRESETS[level][2]
    est = {}

    def e(p):
        if p not in est:
            est[p] = porder_estimate(res, bs, order, p)
        return est[p]

    out = set()
    if bs == 4096:
        out.add(level_max if e(level_max) < e(0) else 0)
    z = (bs & -bs).bit_length() - 1
    caps = {level_max, min(level_max, max(z - 5, 0))}
    for cap in caps:
        mp = max_porder_for(bs, order, cap)
        best, bp = None, mp
        for p in range(mp, -1, -1):
            if best is None or e(p) < best:
                best, bp = e(p), p
        out.add(bp)
    return out
