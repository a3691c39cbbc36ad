"""A FLAC writer driven by explicit syntax.  TEST INFRASTRUCTURE ONLY.

The caller states every syntax element -- subframe type, order, coefficients, precision, shift, wasted bits, residual
coding method, partition order, one Rice parameter or escape width per partition, frame header codes, metadata blocks --
and the writer emits exactly that.  It makes no encoder decisions.  It shares no code with oracle/flac_oracle.c or with
flacarray_b200/csrc: being independent of both is its purpose, so that the decoder can be fed syntax neither encoder
ever writes (escaped partitions, LPC orders above 12, variable blocking, every header code, ...).

Residuals are computed exactly from the samples asked for (int64 arithmetic: |coef| < 2^15, |x| < 2^33 and at most 32
terms keep every prediction sum below 2^53).  The writer refuses a residual of magnitude >= 2^31 and an escape whose raw
width cannot hold its partition.  Bits are packed with numpy; CRCs are table driven.

Syntax the decoder must reject is written through `Sub.bad`, see Sub.
"""
from dataclasses import dataclass, field

import numpy as np

# ---- CRC (RFC 9639: CRC-8 poly 0x07 over the frame header, CRC-16 poly 0x8005 over the whole frame) ----------------


def _crc8_table():
    t = []
    for i in range(256):
        c = i
        for _ in range(8):
            c = ((c << 1) ^ 0x07) & 0xFF if c & 0x80 else (c << 1) & 0xFF
        t.append(c)
    return t


def _crc16_table():
    t = []
    for i in range(256):
        c = i << 8
        for _ in range(8):
            c = ((c << 1) ^ 0x8005) & 0xFFFF if c & 0x8000 else (c << 1) & 0xFFFF
        t.append(c)
    return t


_CRC8 = _crc8_table()
_CRC16 = _crc16_table()


def crc8(b):
    c = 0
    for x in bytes(b):
        c = _CRC8[c ^ x]
    return c


def crc16(b):
    c = 0
    t = _CRC16
    for x in bytes(b):
        c = ((c << 8) & 0xFFFF) ^ t[(c >> 8) ^ x]
    return c


# ---- bit packing ---------------------------------------------------------------------------------------------------


class BitWriter:
    """MSB-first bit fields, packed once at the end.  Fields are (value, width) with width <= 64; longer runs of zero
    bits are split.  Arrays of fields are appended whole, so a partition costs a few numpy calls."""

    def __init__(self):
        self._v = []
        self._n = []
        self.nbits = 0

    def put(self, value, width):
        if width == 0:
            return
        assert 0 < width <= 64 and 0 <= value < (1 << width), (value, width)
        self._v.append(np.array([value], np.uint64))
        self._n.append(np.array([width], np.int64))
        self.nbits += width

    def put_signed(self, value, width):
        assert -(1 << (width - 1)) <= value < (1 << (width - 1)) if width else value == 0, (value, width)
        self.put(value & ((1 << width) - 1), width)

    def put_array(self, values, widths):
        values = np.asarray(values, np.uint64)
        widths = np.asarray(widths, np.int64)
        keep = widths > 0
        self._v.append(values[keep])
        self._n.append(widths[keep])
        self.nbits += int(widths.sum())

    def zeros(self, n):
        while n > 0:
            w = min(n, 64)
            self.put(0, w)
            n -= w

    def pad_to_byte(self):
        self.zeros(-self.nbits % 8)

    def to_bytes(self):
        assert self.nbits % 8 == 0
        if not self._v:
            return b""
        v = np.concatenate(self._v)
        n = np.concatenate(self._n)
        start = np.cumsum(n) - n
        total = int(n.sum())
        pos = np.arange(total, dtype=np.int64) - np.repeat(start, n)
        shift = (np.repeat(n, n) - 1 - pos).astype(np.uint64)
        bits = ((np.repeat(v, n) >> shift) & np.uint64(1)).astype(np.uint8)
        return np.packbits(bits).tobytes()


# ---- syntax --------------------------------------------------------------------------------------------------------

FIXED_COEFS = ([], [1], [2, -1], [3, -3, 1], [4, -6, 4, -1])


@dataclass
class Rice:
    """Residual coding: method 0 (RICE, 4-bit parameters) or 1 (RICE2, 5-bit), partition order, and one entry per
    partition: an int Rice parameter, or ("esc", raw_bits) for an escaped partition."""
    method: int = 0
    porder: int = 0
    params: list = field(default_factory=lambda: [0])


@dataclass
class Sub:
    """One subframe.  kind: "constant", "verbatim", "fixed" (order 0-4) or "lpc" (order 1-32 with `coefs`, `precision`
    1-15 and `shift` 0-15).  `wasted` bits are shifted out of the samples first (they must be multiples of 2^wasted).

    `bad` writes syntax the decoder must reject, then `filler` bytes of arbitrary bits in place of the rest:
      ("type", code)        reserved subframe type code (2-7, 13-31)
      ("shift", s)          LPC shift s < 0
      ("precision_code", 15)
      ("method", m)         residual method 2 or 3
      ("porder", p)         partition order p written as is (one that does not divide the block, or whose first
                            partition is shorter than the order)
    """
    kind: str
    order: int = 0
    coefs: tuple = ()
    precision: int = 15
    shift: int = 0
    wasted: int = 0
    rice: Rice = None
    bad: tuple = None
    filler: int = 64


def _zigzag(r):
    return np.where(r >= 0, 2 * r, -2 * r - 1).astype(np.uint64)


def _write_residual(bw, res, order, bs, rice):
    bw.put(rice.method, 2)
    bw.put(rice.porder, 4)
    nparts = 1 << rice.porder
    assert len(rice.params) == nparts, (len(rice.params), nparts)
    psize = bs >> rice.porder
    assert psize << rice.porder == bs and psize >= order, "partition order does not fit the block"
    plen, esc = (4, 15) if rice.method == 0 else (5, 31)
    i = 0
    for p, par in enumerate(rice.params):
        n = psize - (order if p == 0 else 0)
        r = res[i:i + n]
        i += n
        if isinstance(par, tuple):
            assert par[0] == "esc"
            raw = par[1]
            assert 0 <= raw <= 31
            bw.put(esc, plen)
            bw.put(raw, 5)
            if raw == 0:
                assert not r.any(), "escape with 0 raw bits holds non-zero residuals"
            else:
                lim = 1 << (raw - 1)
                assert r.size == 0 or (int(r.min()) >= -lim and int(r.max()) < lim), "escape raw width too small"
                bw.put_array((r & ((1 << raw) - 1)).astype(np.uint64), np.full(r.size, raw))
            continue
        k = int(par)
        assert 0 <= k < esc
        bw.put(k, plen)
        if n == 0:
            continue
        u = _zigzag(r)
        q = (u >> np.uint64(k)).astype(np.int64)
        low = u & np.uint64((1 << k) - 1)
        short = q + 1 + k <= 64
        if short.all():
            bw.put_array((np.uint64(1) << np.uint64(k)) | low, q + 1 + k)
        else:
            for qq, lo in zip(q.tolist(), low.tolist()):
                if qq + 1 + k <= 64:
                    bw.put((1 << k) | lo, qq + 1 + k)
                else:
                    bw.zeros(qq)
                    bw.put((1 << k) | lo, 1 + k)


def predict_residual(x, kind, order, coefs=(), shift=0):
    """Exact FLAC residual of samples x (int64) for a FIXED or LPC predictor."""
    x = np.asarray(x, np.int64)
    c = FIXED_COEFS[order] if kind == "fixed" else list(coefs)
    assert len(c) == order
    pred = np.zeros(x.size - order, np.int64)
    for j, cj in enumerate(c):
        pred += np.int64(cj) * x[order - 1 - j:x.size - 1 - j]
    if kind == "lpc":
        pred >>= shift
    return x[order:] - pred


def write_subframe(bw, x, bps, sub, bs):
    """Subframe of the samples x (int64, already channel-decorrelated) at `bps` bits (33 for a side channel)."""
    x = np.asarray(x, np.int64)
    assert x.size == bs
    w = sub.wasted
    if w:
        assert not (x & ((1 << w) - 1)).any(), "samples are not multiples of 2^wasted"
        x = x >> w
    b = bps - w
    assert b >= 1 and int(x.min()) >= -(1 << (b - 1)) and int(x.max()) < (1 << (b - 1)), "samples exceed the width"
    bad = sub.bad or (None, None)
    type_code = {"constant": 0, "verbatim": 1}.get(sub.kind)
    if sub.kind == "fixed":
        type_code = 8 + sub.order
    elif sub.kind == "lpc":
        type_code = 32 + sub.order - 1
    if bad[0] == "type":
        type_code = bad[1]
    bw.put(0, 1)
    bw.put(type_code, 6)
    if w:
        bw.put(1, 1)
        bw.zeros(w - 1)
        bw.put(1, 1)
    else:
        bw.put(0, 1)
    if bad[0] == "type":
        return _filler(bw, sub)
    if sub.kind == "constant":
        assert (x == x[0]).all()
        bw.put_signed(int(x[0]), b)
        return
    if sub.kind == "verbatim":
        bw.put_array((x & ((1 << b) - 1)).astype(np.uint64), np.full(bs, b))
        return
    order = sub.order
    assert 0 <= order <= (4 if sub.kind == "fixed" else 32) and order <= bs
    bw.put_array((x[:order] & ((1 << b) - 1)).astype(np.uint64), np.full(order, b))
    if sub.kind == "lpc":
        assert 1 <= order
        if bad[0] == "precision_code":
            bw.put(bad[1], 4)
            return _filler(bw, sub)
        p = sub.precision
        assert 1 <= p <= 15
        bw.put(p - 1, 4)
        if bad[0] == "shift":
            bw.put_signed(bad[1], 5)
            return _filler(bw, sub)
        assert 0 <= sub.shift <= 15
        bw.put_signed(sub.shift, 5)
        for cj in sub.coefs:
            bw.put_signed(int(cj), p)
    if bad[0] == "method":
        bw.put(bad[1], 2)
        return _filler(bw, sub)
    if bad[0] == "porder":
        bw.put(sub.rice.method if sub.rice else 0, 2)
        bw.put(bad[1], 4)
        return _filler(bw, sub)
    res = predict_residual(x, sub.kind, order, sub.coefs, sub.shift)
    assert res.size == 0 or int(np.abs(res).max()) < (1 << 31), "residual of magnitude >= 2^31"
    _write_residual(bw, res, order, bs, sub.rice)


def _filler(bw, sub):
    rng = np.random.default_rng(sub.filler)
    bw.put_array(rng.integers(0, 256, sub.filler, dtype=np.int64).astype(np.uint64), np.full(sub.filler, 8))


# ---- frame header --------------------------------------------------------------------------------------------------

_BS_FIXED = {192: 1, 576: 2, 1152: 3, 2304: 4, 4608: 5, 256: 8, 512: 9, 1024: 10, 2048: 11, 4096: 12, 8192: 13,
             16384: 14, 32768: 15}


def utf8_number(v):
    """FLAC's extended UTF-8 coding of a frame or sample number (up to 36 bits, 7 bytes)."""
    assert 0 <= v < (1 << 36)
    if v < 0x80:
        return bytes([v])
    for n, lim in ((2, 1 << 11), (3, 1 << 16), (4, 1 << 21), (5, 1 << 26), (6, 1 << 31), (7, 1 << 36)):
        if v < lim:
            break
    out = []
    for _ in range(n - 1):
        out.append(0x80 | (v & 0x3F))
        v >>= 6
    lead = (0xFF00 >> n) & 0xFF if n < 7 else 0xFE
    return bytes([lead | v] + out[::-1])


def frame_header(bs, number, nch_code, variable=False, bs_code=None, sr_code=9, ss_code=7, sr_value=None):
    """Frame header bytes up to and including CRC-8.  bs_code None: the table code when bs has one, else 6 / 7.
    sr_value: the trailing value of sample-rate codes 12 (kHz), 13 (Hz), 14 (tens of Hz)."""
    if bs_code is None:
        bs_code = _BS_FIXED.get(bs, 6 if bs <= 256 else 7)
    h = bytearray([0xFF, 0xF8 | (1 if variable else 0), (bs_code << 4) | sr_code, (nch_code << 4) | (ss_code << 1)])
    h += utf8_number(number)
    if bs_code == 6:
        assert 1 <= bs <= 256
        h.append(bs - 1)
    elif bs_code == 7:
        assert 1 <= bs <= 65536
        h += (bs - 1).to_bytes(2, "big")
    elif bs_code == 1:
        assert bs == 192
    elif 2 <= bs_code <= 5:
        assert bs == 576 << (bs_code - 2)
    else:
        assert 8 <= bs_code <= 15 and bs == 256 << (bs_code - 8)
    if sr_code == 12:
        h.append(sr_value if sr_value is not None else 48)
    elif sr_code in (13, 14):
        h += (sr_value if sr_value is not None else 44100 // (10 if sr_code == 14 else 1)).to_bytes(2, "big")
    h.append(crc8(h))
    return bytes(h)


@dataclass
class Frame:
    """One frame of `samples` (int64 [bs] mono, or [bs, 2] left/right) with channel assignment `ca` (0 mono, 1
    independent stereo, 8 left/side, 9 side/right, 10 mid/side) and one Sub per subframe."""
    samples: np.ndarray
    subs: list
    ca: int = 0
    number: int = None     # frame number (fixed) / first sample number (variable); None: filled in by Stream
    variable: bool = False
    bs_code: int = None
    sr_code: int = 9
    ss_code: int = 7
    sr_value: int = None


def channel_signals(samples, ca):
    """The subframe signals and their widths for channel assignment `ca` (RFC 9639 section 4.2)."""
    s = np.asarray(samples, np.int64)
    if ca == 0:
        return [s.reshape(-1)], [32]
    L, R = s[:, 0], s[:, 1]
    if ca == 1:
        return [L, R], [32, 32]
    if ca == 8:
        return [L, L - R], [32, 33]
    if ca == 9:
        return [L - R, R], [33, 32]
    assert ca == 10
    return [(L + R) >> 1, L - R], [32, 33]


def write_frame(fr):
    s = np.asarray(fr.samples, np.int64)
    bs = s.shape[0]
    sigs, widths = channel_signals(s, fr.ca)
    assert len(fr.subs) == len(sigs)
    hdr = frame_header(bs, fr.number, fr.ca, fr.variable, fr.bs_code, fr.sr_code, fr.ss_code, fr.sr_value)
    bw = BitWriter()
    for x, b, sub in zip(sigs, widths, fr.subs):
        write_subframe(bw, x, b, sub, bs)
    bw.pad_to_byte()
    body = hdr + bw.to_bytes()
    return body + crc16(body).to_bytes(2, "big")


# ---- streams -------------------------------------------------------------------------------------------------------


def streaminfo(nch, min_bs, max_bs, total_samples, sample_rate=44100, bps=32, min_fs=0, max_fs=0):
    si = bytearray()
    si += min_bs.to_bytes(2, "big") + max_bs.to_bytes(2, "big")
    si += min_fs.to_bytes(3, "big") + max_fs.to_bytes(3, "big")
    v = (sample_rate << 44) | ((nch - 1) << 41) | ((bps - 1) << 36) | total_samples
    si += v.to_bytes(8, "big")
    si += bytes(16)
    return bytes(si)


def block(type_, payload):
    return bytes([type_]) + len(payload).to_bytes(3, "big") + payload


def padding(n):
    return block(1, bytes(n))


def application(app_id, data):
    return block(2, app_id + data)


def seektable(points):
    return block(3, b"".join(s.to_bytes(8, "big") + o.to_bytes(8, "big") + n.to_bytes(2, "big") for s, o, n in points))


def vorbis_comment(vendor, comments):
    p = len(vendor).to_bytes(4, "little") + vendor + len(comments).to_bytes(4, "little")
    for c in comments:
        p += len(c).to_bytes(4, "little") + c
    return block(4, p)


def fab2_table(frame_sizes, count=None):
    """This library's frame-size APPLICATION block; `count` overrides the entry count (a bogus table)."""
    n = len(frame_sizes) if count is None else count
    return application(b"faB2", n.to_bytes(4, "big") + b"".join(int(v).to_bytes(3, "big") for v in frame_sizes))


def write_stream(frames, nch, min_bs=None, max_bs=None, total_samples=None, blocks=(), number_frames=True):
    """fLaC + STREAMINFO + `blocks` (already framed metadata blocks) + frames.  Returns (stream bytes, frame bytes).
    Frame numbers default to the frame index (fixed) or first sample (variable)."""
    out = []
    sample = 0
    for j, fr in enumerate(frames):
        if fr.number is None and number_frames:
            fr.number = sample if fr.variable else j
        out.append(write_frame(fr))
        sample += np.asarray(fr.samples).shape[0]
    sizes = [np.asarray(f.samples).shape[0] for f in frames]
    min_bs = min(sizes[:-1] or sizes) if min_bs is None else min_bs      # (the last frame of a fixed stream may be short)
    max_bs = max(sizes) if max_bs is None else max_bs
    total_samples = sample if total_samples is None else total_samples
    blocks = list(blocks)
    si = bytes([0x00 if blocks else 0x80]) + (34).to_bytes(3, "big") + streaminfo(nch, min_bs, max_bs, total_samples)
    meta = b""
    for i, b in enumerate(blocks):
        meta += bytes([b[0] | (0x80 if i == len(blocks) - 1 else 0)]) + b[1:]
    return b"fLaC" + si + meta + b"".join(out), out
