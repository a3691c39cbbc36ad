"""Conformance corpus: FLAC streams written syntax element by syntax element (oracle/flac_writer.py), each with the
integers it must decode to or the error it must raise, and the decoder path it is built to reach.

Shared by tests/test_conformance.py (host emulation of the kernel bodies) and tests/test_gpu_conformance.py (the CUDA
library).  Every case is rebuilt from fixed seeds, so a failure reproduces exactly.

Paths, as the throughput decode reports them (hostsim mode 2: info = streams walked + 1000 * frames left to the
general decoder):
  "tile"     every frame decoded by the warp-tile decoder: info == 0
  "general"  some frames left to the general per-thread decoder (LPC order > 12, side channels, a missed 32-bit
             guess): info == 1000 * that many frames, nothing walked
  "walker"   whole streams left to the sequential walker (variable blocking, STREAMINFO min != max, a blocksize that
             needs more frames than the hint allows, duplicate sync candidates, a bad frame-size table)
  "error"    the decode must fail
"""
import functools
from dataclasses import dataclass, field

import numpy as np

from oracle import flac_writer as W
from oracle.flac_writer import Frame, Rice, Sub

I32_MIN, I32_MAX = -2 ** 31, 2 ** 31 - 1
BS = 4096


@dataclass
class Case:
    name: str
    streams: list                  # complete FLAC streams (bytes)
    stream_size: int
    nch: int
    expect: np.ndarray = None      # [n_stream, stream_size] int32 (mono) / int64 (stereo: L low word, R high word)
    path: str = "tile"
    info: int = 0                  # hostsim mode 2 info of the full decode
    frames: list = None            # per stream: the frame bytes (FFmpeg self-check)
    gaps: list = None              # bytes placed in front of each stream in the buffer
    tail: bytes = b""              # bytes behind the last stream
    full: bool = True              # False: too long to decode whole, only `windows` are checked
    windows: list = field(default_factory=list)     # [(stream, first, last)]
    win_expect: list = None        # expected samples of `windows` when not `full`
    ffmpeg: bool = True            # the frames carry explicit sample-rate and sample-size codes

    @property
    def valid(self):
        return self.path != "error"

    @property
    def is_int64(self):
        return self.nch == 2

    def buffer(self):
        """(compressed uint8, starts int64, nbytes int64) with the streams back to back behind their gaps."""
        gaps = self.gaps or [b""] * len(self.streams)
        parts, starts, pos = [], [], 0
        for g, s in zip(gaps, self.streams):
            parts += [g, s]
            pos += len(g)
            starts.append(pos)
            pos += len(s)
        parts.append(self.tail)
        return (np.frombuffer(b"".join(parts), np.uint8).copy(), np.array(starts, np.int64),
                np.array([len(s) for s in self.streams], np.int64))

    def window_expect(self, i):
        if self.win_expect is not None:
            return self.win_expect[i]
        s, a, b = self.windows[i]
        return self.expect[s, a:b]

    def hint(self):
        """The blocksize hint of a decode call: the first stream's STREAMINFO min blocksize, 4096 without one, >= 16."""
        s = self.streams[0]
        h = (s[8] << 8) | s[9] if len(s) >= 12 and s[:4] == b"fLaC" else 0
        return max(16, h or 4096)


# ---- helpers -------------------------------------------------------------------------------------------------------

def walk(rng, n, step, start=0):
    return (start + np.cumsum(rng.integers(-step, step + 1, n))).astype(np.int64)


def _kfor(res, kmax):
    if res.size == 0:
        return 0
    u = np.where(res >= 0, 2 * res, -2 * res - 1).astype(np.float64)
    m = float(u.mean())
    return int(min(kmax, max(0, np.floor(np.log2(m + 1.0)))))


def rice_for(x, kind, order, coefs=(), shift=0, wasted=0, porder=0, method=0, override=None):
    """Rice parameters chosen from the mean residual of every partition; override {partition: param or ("esc", w)}."""
    xs = np.asarray(x, np.int64) >> wasted
    res = np.concatenate([np.zeros(order, np.int64), W.predict_residual(xs, kind, order, coefs, shift)])
    psize = xs.size >> porder
    kmax = 14 if method == 0 else 30
    params = []
    for p in range(1 << porder):
        seg = res[p * psize + (order if p == 0 else 0):(p + 1) * psize]
        params.append(_kfor(seg, kmax))
    for p, v in (override or {}).items():
        params[p] = v
    return Rice(method, porder, params)


def sub_fixed(x, order, porder=0, method=0, wasted=0, override=None):
    return Sub("fixed", order=order, wasted=wasted,
               rice=rice_for(x, "fixed", order, wasted=wasted, porder=porder, method=method, override=override))


def sub_lpc(x, coefs, precision, shift, porder=0, method=0, wasted=0, override=None):
    order = len(coefs)
    return Sub("lpc", order=order, coefs=tuple(int(c) for c in coefs), precision=precision, shift=shift, wasted=wasted,
               rice=rice_for(x, "lpc", order, coefs, shift, wasted, porder, method, override))


def concat(frames):
    return np.concatenate([np.asarray(f.samples, np.int64) for f in frames])


def as_i64(lr):
    """[n, 2] left/right -> the int64 the decoder returns (left in the low word)."""
    return np.ascontiguousarray(np.asarray(lr, np.int64).astype(np.int32)).view(np.int64).reshape(-1)


def edge_windows(sizes, n, s=0):
    """Three windows of stream s across frame edges: around the first edge, over the middle, the tail."""
    b0 = sizes[0]
    w = [(s, max(0, b0 - 3), min(n, b0 + 5)), (s, n // 3, max(n // 3 + 1, (2 * n) // 3)), (s, max(0, n - 7), n)]
    return [x for x in w if x[1] < x[2]]


def single(name, frames, nch=1, path="tile", info=0, blocks=(), ffmpeg=True, **kw):
    data, fb = W.write_stream(frames, nch, blocks=blocks, **kw)
    samples = concat(frames)
    n = samples.shape[0]
    expect = (as_i64(samples) if nch == 2 else samples.astype(np.int32)).reshape(1, -1)
    sizes = [np.asarray(f.samples).shape[0] for f in frames]
    return Case(name, [data], n, nch, expect, path, info, [fb], windows=edge_windows(sizes, n), ffmpeg=ffmpeg)


# ---- valid cases ---------------------------------------------------------------------------------------------------

def _subframe_cases():
    rng = np.random.default_rng(1001)
    out = []
    fr = [Frame(np.full(BS, v, np.int64), [Sub("constant")]) for v in (I32_MIN, I32_MAX, 0, -1)]
    out.append(single("constant_extremes", fr))
    x = rng.integers(I32_MIN, I32_MAX + 1, 2 * BS, dtype=np.int64)
    x[:4] = [I32_MIN, I32_MAX, 0, -1]
    out.append(single("verbatim_full_range", [Frame(x[:BS], [Sub("verbatim")]), Frame(x[BS:], [Sub("verbatim")])]))
    frs = []
    for order in range(5):
        for method in (0, 1):
            x = walk(rng, BS, 300, 1000 * order)
            frs.append(Frame(x, [sub_fixed(x, order, porder=2 + order, method=method)]))
    out.append(single("fixed_orders", frs))
    # orders 1..32 in one stream = one warp of the tile decoder: 4/5, 8/9 and 12/13 side by side; small samples (the
    # 32-bit guess holds) and large ones (64-bit sums)
    streams, fbs, exp = [], [], []
    for amp in (8, 20):
        frs = []
        for order in range(1, 33):
            x = walk(rng, BS, 2 ** (amp - 6), 0 if amp < 16 else 3 << (amp - 2))
            x = np.clip(x, -2 ** amp, 2 ** amp)
            coefs = rng.integers(-2 ** 11, 2 ** 11, order)
            frs.append(Frame(x, [sub_lpc(x, coefs, 12, 9, porder=order % 5, method=order % 2)]))
        d, fb = W.write_stream(frs, 1)
        streams.append(d); fbs.append(fb); exp.append(concat(frs).astype(np.int32))
    out.append(Case("lpc_orders_1_32", streams, 32 * BS, 1, np.array(exp), "general", 1000 * 2 * 20, fbs,
                    windows=edge_windows([BS], 32 * BS) + [(1, 12 * BS - 5, 13 * BS + 9)]))
    frs = []
    for p in range(1, 16):
        x = walk(rng, BS, 3, 0)
        lo, hi = -2 ** (p - 1), 2 ** (p - 1) - 1
        coefs = [lo if j % 2 == 0 else hi for j in range(8)]
        frs.append(Frame(x, [sub_lpc(x, coefs, p, min(15, p + 2), porder=3)]))
    out.append(single("lpc_coefficient_extremes", frs))
    frs = []
    for w in range(1, 32):
        lim = min(2 ** (31 - w), 200)                                # samples >> w fit 32 - w bits
        for kind in ("constant", "verbatim", "fixed", "lpc"):
            base = walk(rng, BS, 3, 0) if lim > 8 else rng.integers(-lim, lim, BS)
            base = np.clip(base, -lim, lim - 1)
            if kind == "constant":
                base = np.full(BS, base[0])
            x = base << w
            if kind in ("constant", "verbatim"):
                sub = Sub(kind, wasted=w)
            elif kind == "fixed":
                sub = sub_fixed(x, 2, porder=1, wasted=w)
            else:
                sub = sub_lpc(x, [3, -2, 1, -1], 6, 1, porder=2, wasted=w)
            frs.append(Frame(x, [sub]))
    out.append(single("wasted_bits_1_31", frs))
    return out


def _residual_cases():
    rng = np.random.default_rng(1002)
    out = []
    # FIXED order 0: the residual is the sample.  RICE params 0..14 (+ an escape), RICE2 0..30 (+ an escape)
    frs = []
    for method, porder, kmax in ((0, 4, 14), (1, 5, 30)):
        psize = BS >> porder
        parts, params = [], []
        for p in range(1 << porder):
            k = min(p, kmax)
            if p == (1 << porder) - 1:
                parts.append(rng.integers(-2 ** 16, 2 ** 16, psize)); params.append(("esc", 17))
            else:
                parts.append(rng.integers(-2 ** k, 2 ** k, psize)); params.append(k)
        x = np.concatenate(parts).astype(np.int64)
        frs.append(Frame(x, [Sub("fixed", order=0, rice=Rice(method, porder, params))]))
    out.append(single("rice_parameters", frs))
    # escapes with 0, 1, 17 and 31 raw bits in the first and in middle partitions, in frames that share a warp with
    # fast-path frames
    frs = []
    widths = (0, 1, 17, 31)
    for j in range(32):
        if j % 2:
            x = walk(rng, BS, 500)
            frs.append(Frame(x, [sub_fixed(x, 2, porder=3, method=j % 4 // 2)]))
            continue
        w0, w1 = widths[(j // 2) % 4], widths[(j // 2 + 1) % 4]
        porder, psize = 3, BS >> 3
        if j % 4 == 0:
            # FIXED order 0: partitions of exactly representable raw values
            parts = []
            for p in range(8):
                w = w0 if p == 0 else w1 if p == 4 else None
                if w is None:
                    parts.append(rng.integers(-300, 300, psize))
                elif w == 0:
                    parts.append(np.zeros(psize, np.int64))
                else:
                    parts.append(rng.integers(-2 ** (w - 1), 2 ** (w - 1), psize))
            x = np.concatenate(parts).astype(np.int64)
            ov = {0: ("esc", w0), 4: ("esc", w1)}
            frs.append(Frame(x, [sub_fixed(x, 0, porder=porder, method=(j // 4) % 2, override=ov)]))
        else:
            x = walk(rng, BS, 200)
            ov = {0: ("esc", 31), 3: ("esc", 17), 7: ("esc", 31)}
            frs.append(Frame(x, [sub_lpc(x, [2, -1, 1, -1, 0, 1, -1, 0], 4, 1, porder=porder, method=1, override=ov)]))
    out.append(single("escaped_partitions", frs))
    # empty first partition (psize == order)
    x1, x2 = walk(rng, BS, 100), walk(rng, BS, 100)
    frs = [Frame(x1, [sub_fixed(x1, 1, porder=12)]),
           Frame(x2, [sub_lpc(x2, [1, 1, -1, 0, 0, 0, 1, -1], 3, 1, porder=9, method=1)])]
    out.append(single("empty_first_partition", frs))
    x = walk(rng, 2 * 32768, 1000)
    frs = [Frame(x[:32768], [sub_fixed(x[:32768], 1, porder=15)]), Frame(x[32768:], [sub_fixed(x[32768:], 0, porder=15)])]
    out.append(single("partition_order_15_bs32768", frs))
    # residuals of +-(2^31 - 1) and long unary runs: 33, 64, 225, ~10000 zero bits (k = 0), 2^18 zero bits (k = 14)
    x = rng.integers(-50, 50, BS).astype(np.int64)
    x[[5, 1600, 2100]] = [I32_MAX, -I32_MAX, I32_MAX]                  # partitions with k = 30
    x[[600, 601, 602, 603, 2700]] = [-17, 32, -113, 5000, -5000]       # k = 0: q = 33, 64, 225, 10000, 9999
    params = [30, 0, 0, 30, 30, 0, 0, 0]
    frs = [Frame(x, [Sub("fixed", order=0, rice=Rice(1, 3, params))])]
    y = rng.integers(-50, 50, BS).astype(np.int64)
    y[[10, 2000]] = [I32_MAX, -I32_MAX]
    y[[2500, 2501]] = [5000, -113]
    frs.append(Frame(y, [Sub("fixed", order=0, rice=Rice(0, 1, [14, 0]))]))
    out.append(single("residual_extremes_long_unary", frs))
    return out


def _guess_cases():
    """The tile decoder's 32-bit prediction guess: sum|coef| * max|x| == 2^31 - 1 stays on the tile path, == 2^31 is
    handed to the general decoder."""
    n = BS
    ramp_up = np.round(np.linspace(0, I32_MAX, n)).astype(np.int64)          # max |x| = 2^31 - 1
    ramp_up[-1] = I32_MAX
    ramp_dn = -ramp_up - 1                                                     # max |x| = 2^31 (INT32_MIN)
    ramp_dn[0] = 0
    half = np.round(np.linspace(0, 2 ** 30, n)).astype(np.int64)               # max |x| = 2^30
    ok = [Frame(ramp_up, [sub_lpc(ramp_up, [1], 2, 0, porder=2)]),
          Frame(ramp_up, [sub_lpc(ramp_up, [0, 1, 0], 2, 0, porder=2)]),
          Frame(-ramp_up, [sub_lpc(-ramp_up, [1], 2, 0, porder=2, method=1)])]
    miss = [Frame(ramp_dn, [sub_lpc(ramp_dn, [1], 2, 0, porder=2)]),
            Frame(half, [sub_lpc(half, [1, 1], 2, 0, porder=2, method=1)]),
            Frame(half, [sub_lpc(half, [2], 3, 0, porder=2, method=1)])]
    for fr in ok + miss:
        fr.samples = np.asarray(fr.samples)
    return [single("guess_product_2p31_minus_1", ok), single("guess_product_2p31", miss, path="general", info=3000)]


def _stereo_cases():
    rng = np.random.default_rng(1004)
    out = []
    frs, side = [], 0
    for j, ca in enumerate((1, 8, 1, 9, 1, 10, 1, 1)):
        L = walk(rng, BS, 400)
        R = L + rng.integers(-30, 31, BS)
        lr = np.stack([L, R], 1)
        sigs, _ = W.channel_signals(lr, ca)
        subs = [sub_fixed(sigs[0], 2, porder=2), sub_lpc(sigs[1], [2, -1, 1, -1], 5, 1, porder=3, method=1)]
        frs.append(Frame(lr, subs, ca=ca))
        side += ca >= 8
    out.append(single("stereo_assignments", frs, nch=2, path="general", info=1000 * side))
    # the 33-bit side channel at the extremes
    frs = []
    c = np.stack([np.full(BS, I32_MIN), np.full(BS, I32_MAX)], 1).astype(np.int64)
    for ca in (8, 9, 10):
        frs.append(Frame(c, [Sub("constant"), Sub("constant")], ca=ca))
    v = np.stack([rng.integers(I32_MIN, I32_MIN + 1000, BS), rng.integers(I32_MAX - 1000, I32_MAX + 1, BS)], 1)
    v[:2] = [[I32_MIN, I32_MAX], [I32_MAX, I32_MIN]]
    for ca in (8, 9, 10):
        frs.append(Frame(v, [Sub("verbatim"), Sub("verbatim")], ca=ca))
    f = np.stack([I32_MIN + np.abs(walk(rng, BS, 50)), I32_MAX - np.abs(walk(rng, BS, 50))], 1)
    for ca in (8, 9, 10):
        sigs, _ = W.channel_signals(f, ca)
        frs.append(Frame(f, [sub_fixed(sigs[0], 1, porder=2), sub_fixed(sigs[1], 2, porder=2)], ca=ca))
    w = 3
    g = np.stack([I32_MIN + (np.abs(walk(rng, BS, 20)) << w), I32_MAX + 1 - ((1 + np.abs(walk(rng, BS, 20))) << w)], 1)
    for ca in (8, 9, 10):
        sigs, _ = W.channel_signals(g, ca)
        coefs = [16] + [3, -3, 2, -2, 1, -1] + [0] * 13             # (sum 2^shift: predicts the level)
        w0 = w if ca != 10 else 0
        frs.append(Frame(g, [sub_lpc(sigs[0], coefs, 8, 4, porder=2, wasted=w0),
                             sub_lpc(sigs[1], coefs, 8, 4, porder=2, wasted=w, method=1)], ca=ca))
    out.append(single("stereo_side_channel_extremes", frs, nch=2, path="general", info=1000 * len(frs)))
    return out


def _blocksize_frames(rng, bs, n, bs_code=None):
    """Fixed-blocksize frames of a walk of n samples; bs_code for the full frames (the last one's code is chosen)."""
    x = walk(rng, n, 700)
    frs = []
    for j, a in enumerate(range(0, n, bs)):
        seg = x[a:a + bs]
        po = 2 if seg.size % 4 == 0 and seg.size >= 16 else 0
        frs.append(Frame(seg, [sub_fixed(seg, 2 if seg.size > 2 else 0, porder=po)],
                         bs_code=bs_code if seg.size == bs else None))
    return frs


def _header_cases():
    rng = np.random.default_rng(1005)
    out = []
    table = [(1, 192), (2, 576), (3, 1152), (4, 2304), (5, 4608)] + [(c, 256 << (c - 8)) for c in range(8, 16)]
    table += [(6, 16), (6, 17), (6, 256), (7, 16), (7, 4095), (7, 65535)]
    for code, bs in table:
        n = 2 * bs + bs // 3 + 1
        out.append(single(f"blocksize_code_{code}_{bs}", _blocksize_frames(rng, bs, n, code)))
    # sample-rate codes 0..14 and sample-size codes 0 / 7, frame by frame
    frs = []
    for j in range(15):
        x = walk(rng, 1152, 100)
        sv = {12: 96, 13: 44100, 14: 4410}.get(j)
        frs.append(Frame(x, [sub_fixed(x, 2, porder=1)], sr_code=j, ss_code=0 if j % 2 else 7, sr_value=sv))
    out.append(single("sample_rate_and_size_codes", frs, ffmpeg=False))
    frs = []
    for j in range(1, 15):
        x = walk(rng, 1152, 100)
        frs.append(Frame(x, [sub_fixed(x, 1, porder=0)], sr_code=j, sr_value={12: 192, 13: 8000, 14: 9600}.get(j)))
    out.append(single("sample_rate_codes_explicit", frs))
    out.append(_utf8_frame_numbers())
    out.append(_variable_sample_numbers())
    # variable blocking with every kind of blocksize, in one stream
    sizes = [16, 17, 192, 4095, 576, 65535, 256, 4096, 1000, 32768, 4608, 16]
    x = walk(rng, sum(sizes), 500)
    frs, a = [], 0
    for bs in sizes:
        seg = x[a:a + bs]
        a += bs
        frs.append(Frame(seg, [sub_fixed(seg, 1, porder=0)], variable=True))
    out.append(single("variable_blocksizes", frs, path="walker", info=1))
    return out


@functools.lru_cache(maxsize=None)
def _utf8_frame_numbers():
    """Fixed blocking at blocksize 16: frame numbers of 1, 2, 3 and 4 UTF-8 bytes (frame 65536 on)."""
    nf = 65536 + 4
    vals = (np.arange(nf, dtype=np.int64) * 2654435761) % (2 ** 32) - 2 ** 31
    frs = [Frame(np.full(16, v), [Sub("constant")]) for v in vals.tolist()]
    data, fb = W.write_stream(frs, 1)
    n = 16 * nf
    expect = np.repeat(vals, 16).astype(np.int32).reshape(1, -1)
    w = [(0, 16 * 127 - 3, 16 * 129 + 2), (0, 16 * 2047 - 1, 16 * 2049), (0, 16 * 65535 - 5, 16 * 65537 + 3), (0, n - 40, n)]
    return Case("frame_numbers_utf8_1_to_4_bytes", [data], n, 1, expect, "tile", 0, [fb], windows=w)


@functools.lru_cache(maxsize=None)
def _variable_sample_numbers():
    """Variable blocking, 65535-sample CONSTANT frames: sample numbers up to the 6-byte UTF-8 form (>= 2^26)."""
    nf = 1026
    frs = [Frame(np.full(65535, (j * 7919) % 65536 - 32768), [Sub("constant")], variable=True) for j in range(nf)]
    for fr in frs:
        fr.samples = np.broadcast_to(fr.samples, (65535,))
    data, fb = W.write_stream(frs, 1)
    n = 65535 * nf
    val = lambda j: (j * 7919) % 65536 - 32768                       # noqa: E731
    w = [(0, 65535 * 1024 - 3, 65535 * 1024 + 4), (0, 65535 * 1025 - 2, 65535 * 1025 + 6), (0, n - 9, n),
         (0, 2 ** 26 - 1, 2 ** 26 + 1)]
    we = []
    for s, a, b in w:
        i = np.arange(a, b)
        we.append(np.array([val(k) for k in (i // 65535).tolist()], np.int32))
    return Case("variable_sample_numbers_6_bytes", [data], n, 1, None, "walker", 1, [fb], full=False, windows=w,
                win_expect=we)


def _stream_cases():
    rng = np.random.default_rng(1006)
    out = []
    frs = _blocksize_frames(rng, BS, 3 * BS + 77)
    blocks = [W.padding(100000), W.seektable([(0, 0, BS), (BS, 1234, BS), (2 ** 64 - 1, 0, 0)]),
              W.vorbis_comment(b"flac_writer", [b"TITLE=conformance", b"X=" + bytes(3000)]),
              W.application(b"abcd", bytes(range(256)) * 4)]
    out.append(single("metadata_blocks", frs, blocks=blocks))
    # frame-size tables (APPLICATION "faB2") that do not describe the stream
    streams, fbs, exp = [], [], []
    n = 3 * BS + 500
    for kind in ("count_too_big", "sizes_wrong", "count_too_small"):
        frs = _blocksize_frames(rng, BS, n)
        for j, f in enumerate(frs):
            f.number = j
        sizes = [len(W.write_frame(f)) for f in frs]
        if kind == "count_too_big":
            blk = W.fab2_table(sizes, count=len(sizes) + 5)
        elif kind == "sizes_wrong":
            blk = W.fab2_table([s + 1 for s in sizes])
        else:
            blk = W.fab2_table(sizes[:-1])
        d, fb = W.write_stream(frs, 1, blocks=[blk])
        streams.append(d); fbs.append(fb); exp.append(concat(frs).astype(np.int32))
    # (a table whose count does not match the stream also turns the sync scan off: that stream is walked as well)
    out.append(Case("bogus_frame_size_tables", streams, n, 1, np.array(exp), "walker", 2, fbs,
                    windows=edge_windows([BS], n, 1)))
    frs = _blocksize_frames(rng, BS, 3 * BS)
    out.append(single("streaminfo_min_ne_max", frs, path="walker", info=1, min_bs=1024, max_bs=BS))
    # streams at every start offset mod 16
    n = 2 * BS + 333
    streams, fbs, exp, gaps = [], [], [], []
    pos = 0
    for s in range(16):
        frs = _blocksize_frames(rng, BS, n)
        d, fb = W.write_stream(frs, 1)
        g = (s - pos) % 16
        gaps.append(bytes([0xFF] * g))
        pos += g + len(d)
        streams.append(d); fbs.append(fb); exp.append(concat(frs).astype(np.int32))
    c = Case("start_offsets_mod_16", streams, n, 1, np.array(exp), "tile", 0, fbs, gaps=gaps,
             windows=edge_windows([BS], n, 5) + edge_windows([BS], n, 15))
    assert sorted(int(x) % 16 for x in c.buffer()[1]) == list(range(16))
    out.append(c)
    out.append(_sync_pairs(rng))
    out.append(_duplicate_header(rng))
    return out


def _verbatim_bytes_frame(payload, number=None):
    """A VERBATIM mono frame whose sample bytes are `payload` (a multiple of 4 bytes, blocksize = len / 4)."""
    x = np.frombuffer(payload, ">i4").astype(np.int64)
    return Frame(x, [Sub("verbatim")], number=number)


def _sync_pairs(rng):
    """FF F8 byte pairs that are not frame headers: across 16-byte chunk edges, 512-byte row edges, and the stream's
    last byte (with F8 the first byte behind the stream)."""
    n0 = 2048
    pre = _blocksize_frames(rng, n0, n0)
    hdr_len = len(W.write_stream(pre, 1, min_bs=n0, max_bs=n0)[0])     # the VERBATIM frame starts here
    for f in pre:
        f.number = None
    raw = bytearray(rng.integers(0, 256, 4 * n0, dtype=np.uint8).tobytes())
    body0 = hdr_len + len(W.frame_header(n0, 1, 0)) + 1               # frame header + subframe header
    for edge in (16, 512):
        for m in range(1, 12):
            p = m * edge * 3 - 1 - body0                              # FF on the last byte of a chunk / row
            if 0 <= p < len(raw) - 1:
                raw[p], raw[p + 1] = 0xFF, 0xF8
    frs = pre + [_verbatim_bytes_frame(bytes(raw))]
    # last frame: a VERBATIM sample tuned until the frame's CRC-16 ends in FF
    tail = rng.integers(-1000, 1000, n0).astype(np.int64)
    for v in range(100000):
        tail[-1] = v
        last = Frame(tail.copy(), [Sub("verbatim")], number=2)
        if W.write_frame(last)[-1] == 0xFF:
            break
    last.number = None
    frs.append(last)
    data, fb = W.write_stream(frs, 1, min_bs=n0, max_bs=n0)
    assert data[body0 - 1] == 0x02 and data[-1] == 0xFF
    n = 3 * n0
    expect = concat(frs).astype(np.int32).reshape(1, -1)
    return Case("sync_pairs_at_chunk_row_and_stream_edges", [data], n, 1, expect, "tile", 0, [fb], tail=b"\xf8" + bytes(40),
                windows=edge_windows([n0], n))


def _duplicate_header(rng):
    """A VERBATIM payload that holds a byte-exact copy of the next frame's header: two sync candidates for one frame
    send the stream to the walker."""
    frs = _blocksize_frames(rng, BS, 3 * BS)
    hdr2 = W.frame_header(BS, 2, 0)
    raw = bytearray(rng.integers(0, 256, 4 * BS, dtype=np.uint8).tobytes())
    raw[1000:1000 + len(hdr2)] = hdr2
    raw[1000 + len(hdr2):1000 + len(hdr2) + 8] = bytes(8)
    frs[1] = _verbatim_bytes_frame(bytes(raw))
    return single("duplicate_sync_candidate", frs, path="walker", info=1)


def _mixed_cases():
    rng = np.random.default_rng(1007)
    out = []
    n = 3 * BS + 100

    def call(name, specs, path, info):
        streams, fbs, exp = [], [], []
        for bs, variable, mn in specs:
            frs = _blocksize_frames(rng, bs, n)
            for f in frs:
                f.variable = variable
            d, fb = W.write_stream(frs, 1, min_bs=mn)
            streams.append(d); fbs.append(fb); exp.append(concat(frs).astype(np.int32))
        return Case(name, streams, n, 1, np.array(exp), path, info, fbs,
                    windows=edge_windows([specs[0][0]], n, 0) + edge_windows([specs[-1][0]], n, len(specs) - 1))

    out.append(call("mixed_first_blocksize_smaller", [(1152, False, None), (BS, False, None), (BS, False, None)], "tile", 0))
    out.append(call("mixed_first_blocksize_larger", [(BS, False, None), (1152, False, None), (576, False, None)], "walker", 2))
    out.append(call("mixed_first_variable", [(BS, True, 1024), (BS, False, None), (1152, False, None)], "walker", 1))
    return out


# ---- invalid syntax ------------------------------------------------------------------------------------------------

def _invalid_cases():
    """Syntax both subframe parsers must reject: the warp-tile one (mono, order <= 12) and the general one (order > 12,
    side channels)."""
    rng = np.random.default_rng(1008)
    out = []

    def case(name, bad_frame, bs=BS):
        frs = _blocksize_frames(rng, bs, 2 * bs)
        frs.insert(1, bad_frame)
        for f in frs:
            f.number = None
        d, fb = W.write_stream(frs, 1)
        return Case(name, [d], 3 * bs, 1, None, "error", frames=[fb])

    def st_case(name, subs, ca=8):
        L = walk(rng, BS, 300)
        lr = np.stack([L, L + 7], 1)
        frs = []
        for j in range(3):
            sigs, _ = W.channel_signals(lr, 1)
            frs.append(Frame(lr, [sub_fixed(sigs[0], 1), sub_fixed(sigs[1], 1)], ca=1))
        frs[1] = Frame(lr, subs(lr, ca), ca=ca)
        d, fb = W.write_stream(frs, 2)
        return Case(name, [d], 3 * BS, 2, None, "error", frames=[fb])

    x = walk(rng, BS, 300)
    co4, co20 = [1, 1, -1, 0], list(rng.integers(-30, 30, 20))
    for tag, coefs in (("tile", co4), ("general", co20)):
        for bad in (("shift", -3), ("shift", -16), ("precision_code", 15), ("method", 2), ("method", 3)):
            s = sub_lpc(x, coefs, 8, 2, porder=1)
            s.bad = bad
            out.append(case(f"invalid_{tag}_{bad[0]}_{bad[1]}", Frame(x, [s])))
        s = sub_lpc(x, coefs, 8, 2)
        s.bad = ("porder", 11 if tag == "tile" else 8)                   # partitions of 2 / 16 samples < order
        out.append(case(f"invalid_{tag}_partition_shorter_than_order", Frame(x, [s])))
    y = walk(rng, 4095, 300)
    for tag, s in (("tile", sub_fixed(y, 2)), ("general", sub_lpc(y, co20, 8, 2))):
        s.bad = ("porder", 1)
        out.append(case(f"invalid_{tag}_partition_order_does_not_divide", Frame(y, [s]), bs=4095))
    for code in (2, 5, 7, 13, 20, 31):
        out.append(case(f"invalid_tile_reserved_type_{code}", Frame(x, [Sub("fixed", order=0, bad=("type", code))])))
    for code in (3, 15):
        out.append(st_case(f"invalid_general_reserved_type_{code}",
                           lambda lr, ca: [Sub("constant", bad=("type", code)), Sub("constant")], ca=8))
    for bad in (("shift", -1), ("precision_code", 15), ("method", 2)):
        def subs(lr, ca, bad=bad):
            sigs, _ = W.channel_signals(lr, ca)
            s1 = sub_lpc(sigs[1], [1, 1, -1, 0], 8, 2, porder=1)
            s1.bad = bad
            return [sub_fixed(sigs[0], 1), s1]
        out.append(st_case(f"invalid_side_channel_{bad[0]}_{bad[1]}", subs, ca=9))
    return out


def _damage_cases():
    """About 64 single-bit flips inside the frames of one stream (tile and general frames): CRC-8 and CRC-16 detect every
    single-bit error, so each must fail."""
    rng = np.random.default_rng(1009)
    x = walk(rng, 4 * BS, 400)
    frs = [Frame(x[:BS], [sub_fixed(x[:BS], 2, porder=3)]),
           Frame(x[BS:2 * BS], [sub_lpc(x[BS:2 * BS], list(rng.integers(-40, 40, 16)), 8, 4, porder=2, method=1)]),
           Frame(x[2 * BS:3 * BS], [sub_lpc(x[2 * BS:3 * BS], [2, -1], 4, 0, porder=5, override={7: ("esc", 20)})]),
           Frame(x[3 * BS:], [Sub("verbatim")])]
    data, fb = W.write_stream(frs, 1)
    first = len(data) - sum(len(f) for f in fb)
    out = []
    pos = np.sort(rng.choice(np.arange(first * 8, len(data) * 8), 64, replace=False))
    # and the first bit of every frame header and CRC-16
    off = first
    extra = []
    for f in fb:
        extra += [off * 8, (off + 3) * 8 + 7, (off + len(f) - 1) * 8]
        off += len(f)
    for p in sorted(set(pos.tolist() + extra)):
        b = bytearray(data)
        b[p >> 3] ^= 0x80 >> (p & 7)
        out.append(Case(f"damage_bit_{p}", [bytes(b)], 4 * BS, 1, None, "error"))
    return out


@functools.lru_cache(maxsize=None)
def valid_cases():
    return tuple(_subframe_cases() + _residual_cases() + _guess_cases() + _stereo_cases() + _header_cases() +
                 _stream_cases() + _mixed_cases())


@functools.lru_cache(maxsize=None)
def invalid_cases():
    return tuple(_invalid_cases())


@functools.lru_cache(maxsize=None)
def damage_cases():
    return tuple(_damage_cases())


def by_name(name):
    for c in valid_cases() + invalid_cases() + damage_cases():
        if c.name == name:
            return c
    raise KeyError(name)
