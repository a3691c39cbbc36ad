"""Encoder conformance on the CPU: every stream the encoder's kernel bodies write (through the host emulator,
tests/hostsim) is read by the strict reader of tests/flac_strict.py, and the encoder's analysis records and choices are
compared with plain references.

- The strict reader checks each stream against RFC 9639, libFLAC's decoder limits and the library's documented stream
  layout, and decodes it to the input.  It has its own unit tests on hand-built streams (oracle/flac_writer.py).
- `FrameStats` of every (frame, channel) against a Python restatement of k_enc_analyze: mode, wasted bits, min, max,
  the int32-fit mask and the five fixed-predictor error sums exactly, the windowed autocorrelation within a rigorous
  FP64 bound of its exact value.
- Rice parameters, partition orders and fixed orders against the encoder's documented rules (flac_strict.check_choices).
- The emulator reproduces the SHA-256 of the GPU's bytes frozen in tests/golden/gpu_encoded_sha256.json.
- Compressed size within 2 % of the oracle encoder on realistic wide signals.
"""
import hashlib
import json
import math
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostsim"))

import flac_strict as S  # noqa: E402
from oracle import flac_writer as W  # noqa: E402


@pytest.fixture(scope="module")
def H():
    import hostsim

    hostsim.lib()
    return hostsim


# ---- signals -------------------------------------------------------------------------------------------------------
I32_MIN, I32_MAX = -2 ** 31, 2 ** 31 - 1
LENGTHS = [1, 15, 16, 17, 1151, 1152, 1153, 4095, 4096, 4097, 2, 4099, 8195]   # the last three: n % 4 != 0


def _i32(v):
    return np.clip(np.round(v), I32_MIN, I32_MAX).astype(np.int32)


def adversarial(n, seed=7):
    """Full-scale signals that stress the predictor design and the int32 limits of residuals and samples."""
    rng = np.random.default_rng(seed)
    i = np.arange(n)
    spikes = np.cumsum(rng.integers(-300, 301, n)).astype(np.int64)
    spikes[rng.integers(0, n, max(n // 500, 1))] = I32_MAX
    spikes[rng.integers(0, n, max(n // 500, 1))] = I32_MIN
    return {
        "alternating": np.where(i % 2 == 1, I32_MAX, I32_MIN).astype(np.int32),
        "square": np.where((i // 37) % 2 == 1, I32_MAX, I32_MIN).astype(np.int32),
        "sine_fs_p50": _i32(I32_MAX * np.sin(2 * np.pi * i / 50)),
        "sine_fs_p9": _i32(I32_MAX * np.sin(2 * np.pi * i / 9)),
        "nyquist": _i32(2.1e9 * np.cos(np.pi * i)),
        "nyquist_env": _i32(2.1e9 * np.cos(np.pi * i) * np.sin(np.pi * i / 4096) ** 2),
        "spikes": _i32(spikes),
        "wrap_walk": np.cumsum(rng.integers(-2 ** 30, 2 ** 30, n, dtype=np.int64)).astype(np.uint32).view(np.int32),
        "rails_noise": _i32(I32_MAX * np.sin(2 * np.pi * i / 400) * 1.2 + rng.normal(0, 2 ** 20, n)),
    }


def int32_signals(n, bs, seed=1):
    """Walks, tones at 2^14 .. 2^30, full-scale random (VERBATIM), a constant frame inside a predictive stream, wasted
    bits in one frame only, plus the adversarial set."""
    rng = np.random.default_rng(seed + n)
    i = np.arange(n)
    walk = np.cumsum(rng.integers(-1000, 1001, n)).astype(np.int64)
    sig = {"walk": walk.astype(np.int32)}
    for e in (14, 22, 30):
        sig[f"tone{e}"] = _i32(2.0 ** e * 0.9 * np.sin(2 * np.pi * i / 93.3) + rng.normal(0, 2.0 ** (e - 12), n))
    sig["random"] = rng.integers(I32_MIN, I32_MAX + 1, n, dtype=np.int64).astype(np.int32)
    c = walk.copy()
    c[bs:2 * bs] = -123456
    sig["const_frame"] = c.astype(np.int32)
    w = walk.copy()
    w[bs:2 * bs] *= 32
    sig["wasted_frame"] = w.astype(np.int32)
    sig.update(adversarial(n, seed + n))
    return sig


def int64_signals(n, seed=3):
    rng = np.random.default_rng(seed + n)
    walk = np.cumsum(rng.integers(-2 ** 20, 2 ** 20 + 1, n)).astype(np.int64)
    lows = walk + (1 << 32) - 5000            # low words wrap through 0 and 2^32 while the high word steps
    ext = rng.integers(-2 ** 63, 2 ** 63 - 1, n, dtype=np.int64)
    ext[: min(n, 4)] = [-2 ** 63, 2 ** 63 - 1, 2 ** 32, -2 ** 32][: min(n, 4)]
    return {"walk": walk + 2 ** 40, "wrap_low": lows, "extremes": ext,
            "tod": np.round((np.sin(np.arange(n) / 300.0) * 3 + rng.normal(0, 1, n)) / 1e-9).astype(np.int64)}


def float_signals(n, dt, seed=5):
    rng = np.random.default_rng(seed + n)
    i = np.arange(n)
    return {"tod": (2 * np.sin(2 * np.pi * 15 * i / max(n, 1)) + rng.normal(0, 1, n) + 5).astype(dt),
            "ramp": (i * 1e-3).astype(dt), "noise": rng.normal(0, 1e3, n).astype(dt)}


# ---- helpers -------------------------------------------------------------------------------------------------------
def channels(row):
    """The encoder's channels of one stream: int32 / quantised float32 as one, int64 as (low word, high word)."""
    row = np.ascontiguousarray(row)
    if row.dtype.itemsize == 8:
        return row.view(np.int32).reshape(-1, 2).T.astype(np.int64)
    return row[None].astype(np.int64)


def encode_and_read(H, x, level, quanta=None, name=""):
    """Encode the rows of x through the emulator, read every stream strictly and check the choices.  Returns the
    emulator's outputs and the quantised integer input (float input) and the parsed streams."""
    x = np.ascontiguousarray(x)
    comp, st, nb, off, gain, stats, plans, fixed = H.encode(x, level, quanta=quanta, records=True)
    ints = x
    if x.dtype.kind == "f":
        from oracle import oracle as O

        ints, o2, g2 = O.float_to_int(x, None if quanta is None else np.asarray(quanta, x.dtype))
        assert np.array_equal(off, o2) and np.array_equal(gain, g2), name
    nch = 2 if x.dtype.itemsize == 8 else 1
    streams = []
    for s in range(x.shape[0]):
        rd = S.read_stream(comp[st[s]:st[s] + nb[s]], level, x.shape[1], nch, f"{name} stream {s}", expect=channels(ints[s]))
        S.check_choices(rd, level, (stats[s], plans[s], fixed[s]), f"{name} stream {s}")
        streams.append(rd)
    assert int(st[0]) == 0 and np.array_equal(st[1:], np.cumsum(nb)[:-1]) and int(nb.sum()) == comp.size, name
    return comp, st, nb, stats, plans, fixed, ints, streams


# ---- 1. the strict reader on hand-built streams ------------------------------------------------------------------
def _valid_stream(n=3000, level=5, seed=11):
    """A stream with the encoder's layout (fixed 4096 / 1152 blocking, faB2 table) built by the independent writer."""
    rng = np.random.default_rng(seed)
    bs = S.PRESETS[level][0]
    x = np.cumsum(rng.integers(-500, 501, n)).astype(np.int64)
    frames = []
    for a in range(0, n, bs):
        seg = x[a:a + bs]
        sub = W.Sub("fixed", order=2, rice=W.Rice(0, 0, [0]))
        res = W.predict_residual(seg, "fixed", 2)
        sub.rice.params = [S.rice_param(int(np.abs(res).sum()), res.size)]
        frames.append(W.Frame(seg, [sub]))
    return x, _assemble(frames, n, bs)


def _assemble(frames, n, bs, nch=1):
    """fLaC + STREAMINFO + faB2 table (last) + the frames (writer Frames, numbered here, or finished bytes)."""
    for j, f in enumerate(frames):
        if not isinstance(f, bytes):
            f.number = j
    body = [W.write_frame(f) if not isinstance(f, bytes) else f for f in frames]
    tab = W.fab2_table([len(b) for b in body])
    si = bytes([0x00]) + (34).to_bytes(3, "big") + W.streaminfo(nch, bs, bs, n)
    app = bytes([tab[0] | 0x80]) + tab[1:]
    return bytearray(b"fLaC" + si + app + b"".join(body))


def _refresh_crc16(buf, start, end):
    """Recompute the CRC-16 of the frame buf[start:end] (after an edit inside it)."""
    buf[end - 2:end] = W.crc16(bytes(buf[start:end - 2])).to_bytes(2, "big")


def test_strict_reader_accepts_a_valid_stream():
    x, buf = _valid_stream()
    st = S.read_stream(buf, 5, x.size, 1, expect=x[None])
    assert len(st.frames) == 1 and st.frames[0].subframes[0].kind == "fixed"
    assert np.array_equal(st.samples()[0], x)
    x, buf = _valid_stream(5000, level=0)
    st = S.read_stream(buf, 0, x.size, 1)          # without the input: decoded by the reader's own loop
    assert np.array_equal(st.samples()[0], x) and [f.blocksize for f in st.frames] == [1152] * 4 + [392]


def test_strict_reader_accepts_every_corpus_subframe_kind():
    """Syntax the encoder never writes but a strict reader must still parse: escapes, RICE2, LPC, wasted bits."""
    rng = np.random.default_rng(2)
    n = 4096
    x = (np.cumsum(rng.integers(-300, 301, n)) * 4).astype(np.int64)
    subs = [W.Sub("lpc", order=2, coefs=(4096, -2048), precision=14, shift=11, wasted=2, rice=W.Rice(1, 1, [16, ("esc", 20)])),
            W.Sub("verbatim"), W.Sub("fixed", order=1, wasted=2, rice=W.Rice(0, 2, [7, 8, 9, 10]))]
    for sub in subs:
        st = S.read_stream(_assemble([W.Frame(x, [sub])], n, 4096), 8, n, 1, expect=x[None])
        assert np.array_equal(st.samples()[0], x)
    sub = W.Sub("constant")
    c = np.full(n, -7, np.int64)
    assert S.read_stream(_assemble([W.Frame(c, [sub])], n, 4096), 8, n, 1, expect=c[None]).frames[0].subframes[0].kind == "constant"


def _raw_fixed1_frame(x, number=0):
    """A FIXED order-1 frame written field by field (the writer refuses residuals outside int32, this one does not)."""
    bs = x.size
    bw = W.BitWriter()
    bw.put(0, 1)
    bw.put(9, 6)
    bw.put(0, 1)
    bw.put(int(x[0]) & 0xFFFFFFFF, 32)
    bw.put(1, 2)
    bw.put(0, 4)
    r = np.diff(x)
    u = [2 * int(v) if v >= 0 else -2 * int(v) - 1 for v in r]
    k = 20
    bw.put(k, 5)
    for v in u:
        bw.zeros(v >> k)
        bw.put((1 << k) | (v & ((1 << k) - 1)), k + 1)
    bw.pad_to_byte()
    body = W.frame_header(bs, number, 0) + bw.to_bytes()
    return body + W.crc16(body).to_bytes(2, "big")


def _lpc_frame_bits(x, shift):
    """An LPC order-1 frame with shift `shift` written field by field."""
    bw = W.BitWriter()
    bw.put(0, 1)
    bw.put(32, 6)
    bw.put(0, 1)
    bw.put(int(x[0]) & 0xFFFFFFFF, 32)
    bw.put(14, 4)
    bw.put(shift & 31, 5)
    bw.put(1 << (15 - 2), 15)          # coefficient 2^13: x[i-1] * 2^13 >> shift
    bw.put(0, 2)
    bw.put(0, 4)
    r = x[1:] - ((x[:-1] * (1 << 13)) >> shift)
    u = [2 * int(v) if v >= 0 else -2 * int(v) - 1 for v in r]
    k = min(S.rice_param(int(np.abs(r).sum()), r.size), 14)
    bw.put(k, 4)
    for v in u:
        bw.zeros(v >> k)
        bw.put((1 << k) | (v & ((1 << k) - 1)), k + 1)
    bw.pad_to_byte()
    body = W.frame_header(x.size, 0, 0) + bw.to_bytes()
    return body + W.crc16(body).to_bytes(2, "big")


def _expect_error(buf, match, n, level=5, nch=1, expect=None):
    with pytest.raises(S.StrictError, match=match):
        S.read_stream(buf, level, n, nch, name="hand-built", expect=expect)


def test_strict_reader_rejects_each_violation():
    x, good = _valid_stream()
    n = x.size
    hdr = S.stream_header_bytes(1)
    # residual outside int32 (a FIXED order-1 step from -2^31 to 2^31 - 1)
    y = x.copy()
    y[99], y[100], y[101] = 0, I32_MIN, I32_MAX
    _expect_error(_assemble([_raw_fixed1_frame(y)], n, 4096), r"frame 0, channel 0: residual: sample 101: 4294967295 outside int32", n)
    # LPC shift 16 (read as -16 from the 5-bit field) and precision code 15
    z = np.cumsum(np.ones(n, np.int64))
    _expect_error(_assemble([_lpc_frame_bits(z, 16)], n, 4096), r"channel 0: LPC shift: -16 outside 0..15", n)
    b = _assemble([_lpc_frame_bits(z, 13)], n, 4096)
    assert S.read_stream(b, 5, n, 1, expect=z[None])
    fs = hdr + len(W.frame_header(n, 0, 0)) + 5       # the byte that holds the precision code
    bad = bytearray(b)
    bad[fs] |= 0x0F << 3 & 0xFF                       # precision bits 1111
    _expect_error(bad, r"LPC precision|CRC-16", n)
    # a faB2 size off by one
    bad = bytearray(good)
    bad[56] += 1
    _expect_error(bad, r"frame 0: faB2 frame size: \d+ != the frame's \d+ bytes", n)
    # a trailing byte
    _expect_error(good + b"\x00", r"stream end: 1 bytes after the last frame", n)
    # a CRC-16 flip and a CRC-8 flip
    bad = bytearray(good)
    bad[-1] ^= 1
    _expect_error(bad, r"frame 0: CRC-16", n)
    bad = bytearray(good)
    bad[hdr + 7] ^= 1                                  # FF F8, codes, channels, number, blocksize - 1 (2 bytes), CRC-8
    _expect_error(bad, r"frame 0: CRC-8", n)
    # nonzero padding before the CRC-16 (the frame's residual ends inside its last byte: set a pad bit, fix the CRC)
    st = S.read_stream(good, 5, n, 1)
    pad_bits = -(8 * (len(W.frame_header(n, 0, 0))) + st.frames[0].subframes[0].nbits) % 8
    assert pad_bits > 0
    bad = bytearray(good)
    bad[-3] |= 1
    _refresh_crc16(bad, hdr, len(bad))
    _expect_error(bad, r"frame 0: padding: nonzero bits before the CRC-16", n)
    # a wrong total-samples field
    bad = bytearray(good)
    bad[8 + 17] ^= 1
    _expect_error(bad, r"STREAMINFO total samples", n)
    # wrong blocksize fields, channel count, MD5, last-metadata flags, frame number, sample-size code
    for off, val, match in ((8, 0x00, "STREAMINFO blocksize"), (8 + 12, None, "STREAMINFO channels"),
                            (8 + 30, 1, "STREAMINFO MD5"), (4, 0x80, "STREAMINFO block header"),
                            (42, 0x02, "APPLICATION block header")):
        bad = bytearray(good)
        bad[off] = (bad[off] ^ 2) if val is None else val
        _expect_error(bad, match, n)
    two = _valid_stream(6000)[1]
    bad = bytearray(two)
    f1 = S.read_stream(two, 5, 6000, 1).frames[1].offset
    bad[f1 + 4] = 5                                  # frame number 5 instead of 1
    bad[f1 + 5] = W.crc8(bytes(bad[f1:f1 + 5]))
    _expect_error(bad, r"frame 1: frame number: 5 != 1", 6000)
    # samples that do not decode to the input, and a frame that is not full before the last one
    e = x.copy()
    e[1500] += 1
    _expect_error(good, r"frame 0, channel 0: samples: sample 1500: decodes to", n, expect=e[None])
    _expect_error(good, r"frame 0, channel 0: warm-up", n, expect=(x + 1)[None])
    _expect_error(_valid_stream(5000, level=0)[1], r"STREAMINFO blocksize", 5000, level=5)


def test_strict_reader_rejects_oversized_subframes_and_wide_samples():
    n = 4096
    rng = np.random.default_rng(4)
    x = rng.integers(-2 ** 31, 2 ** 31, n, dtype=np.int64)
    # FIXED order 0 with the rule's Rice parameter on full-scale noise: larger than VERBATIM of the same samples
    sub = W.Sub("fixed", order=0, rice=W.Rice(1, 0, [S.rice_param(int(np.abs(x).sum()), n)]))
    _expect_error(_assemble([W.Frame(x, [sub])], n, 4096), r"subframe size: \d+ bits > VERBATIM's 131080", n)
    # a FIXED order-2 predictor whose reconstruction leaves 32 bits is refused by the writer; build it through the residual
    y = np.zeros(64, np.int64)
    y[:2] = [I32_MAX - 1, I32_MAX]
    bw = W.BitWriter()
    bw.put(0, 1), bw.put(10, 6), bw.put(0, 1)
    bw.put(int(y[0]) & 0xFFFFFFFF, 32), bw.put(int(y[1]) & 0xFFFFFFFF, 32)
    bw.put(0, 2), bw.put(0, 4), bw.put(0, 4)
    for _ in range(62):
        bw.put(1, 1)                                   # residual 0: the ramp continues past 2^31 - 1
    bw.pad_to_byte()
    body = W.frame_header(64, 0, 0, bs_code=6) + bw.to_bytes()
    frame = body + W.crc16(body).to_bytes(2, "big")
    _expect_error(_assemble([frame], 64, 4096), r"channel 0: samples: sample 2 = 2147483648 outside 32 bits", 64)


# ---- 2. reference of k_enc_analyze -------------------------------------------------------------------------------
def tukey_window(L):
    """fa_encode.h make_tukey_window (tukey(0.5), libFLAC window.c), float32."""
    w = np.ones(L, np.float32)
    Np = int(np.float32(0.25) * np.float32(L)) - 1
    if Np > 0:
        for k in range(Np + 1):
            w[k] = np.float32(0.5 - 0.5 * math.cos(math.pi * k / Np))
            w[L - Np - 1 + k] = np.float32(0.5 - 0.5 * math.cos(math.pi * (k + Np) / Np))
    return w


def ref_stats(x, bs_nom, max_lpc):
    """k_enc_analyze's FrameStats of one frame-channel x (int64 values of int32 samples), restated:
    mode 0 below 64 samples, 1 CONSTANT, 2 narrow (-2^22 <= x < 2^22), 3 wide; wasted = trailing zero bits of the OR;
    mn / mx and the error sums of the samples >> wasted (libFLAC FLAC__fixed_compute_best_predictor(_wide): sum over
    i >= 4 of |order-k difference|); bad (wide only) = the orders whose difference leaves +-(2^31 - 1).
    ac[l] = sum_i v_i v_(i-l) with v_i = float32(float32(x_i) * w_i), w the nominal window's prefix (libFLAC lpc.c:
    float data times float window, double accumulation), times 2^(-2 wasted): returned exactly as (fsum value,
    sum of |terms|) per lag."""
    n = x.size
    if n < 64:
        return dict(mode=0)
    mn, mx = int(x.min()), int(x.max())
    if mn == mx:
        mode, wasted = 1, 0
    else:
        orv = int(np.bitwise_or.reduce(x.astype(np.uint32)))
        wasted = (orv & -orv).bit_length() - 1
        mode = 3 if (mn < -S.NARROW or mx >= S.NARROW) else 2
    xs = x >> wasted
    fe, bad = S.fixed_sums(xs)
    r = dict(mode=mode, wasted=wasted, mn=mn >> wasted, mx=mx >> wasted, bad=bad if mode == 3 else 0, fe=fe)
    w = tukey_window(bs_nom)[:n]
    v = (x.astype(np.float32) * w).astype(np.float64)
    ac = []                                              # (levels 0..2 design no LPC: no autocorrelation)
    for l in range(max_lpc + 1 if max_lpc else 0):
        t = v[l:] * v[:n - l]                           # exact: 24-bit x 24-bit significands
        ac.append((math.fsum(t.tolist()) * 2.0 ** (-2 * wasted), float(np.abs(t).sum()) * 2.0 ** (-2 * wasted)))
    r["ac"] = ac
    return r


def check_stats(stats, fixed, ints, level, name):
    """Compare every (frame, channel) record the analysis wrote with ref_stats.  Returns the number compared."""
    bs_nom, max_lpc = S.PRESETS[level][0], S.PRESETS[level][1]
    n_cmp = 0
    for s in range(ints.shape[0]):
        ch = channels(ints[s])
        for j in range(stats.shape[1]):
            if fixed[s, j]:
                continue                                # k_enc_fixed took the frame: no records
            for c in range(ch.shape[0]):
                x = ch[c, j * bs_nom:(j + 1) * bs_nom]
                got, ref = stats[s, j, c], ref_stats(x, bs_nom, max_lpc)
                loc = f"{name} stream {s} frame {j} channel {c} ({x.size} samples)"
                assert got["mode"] == ref["mode"], (loc, "mode", got["mode"], ref["mode"])
                if ref["mode"] == 0:
                    continue
                for k in ("wasted", "mn", "mx", "bad"):
                    assert got[k] == ref[k], (loc, k, got[k], ref[k])
                if ref["mode"] >= 2:                    # (CONSTANT frames never use the sums)
                    assert [int(v) for v in got["fe"]] == ref["fe"], (loc, "fe", got["fe"], ref["fe"])
                if not ref["ac"]:
                    assert not got["ac"].any(), (loc, "ac", got["ac"])
                for l, (exact, mag) in enumerate(ref["ac"]):
                    bound = (x.size + 3) * 2.0 ** -53 * mag
                    assert abs(float(got["ac"][l]) - exact) <= bound, (loc, "ac", l, float(got["ac"][l]), exact, bound)
                n_cmp += 1
    return n_cmp


# ---- 3. the case matrix ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("level", range(9))
def test_int32_streams_are_strictly_valid_and_analysed_exactly(H, level):
    """Every length at the levels 0, 3, 5 and 8; at the others, whose presets differ from those in one parameter or
    none (levels 1 and 2 are level 0's, 7 is 8's), the lengths around the blocksizes."""
    bs = S.PRESETS[level][0]
    for n in LENGTHS if level in (0, 3, 5, 8) else (17, 1153, 4097, 8195):
        sig = int32_signals(n, bs)
        x = np.stack(list(sig.values()))
        *_, stats, plans, fixed, ints, _ = encode_and_read(H, x, level, name=f"L{level} n={n}")
        check_stats(stats, fixed, ints, level, f"L{level} n={n}")


@pytest.mark.parametrize("level", [0, 3, 5, 8])
def test_int64_streams_are_strictly_valid_and_analysed_exactly(H, level):
    for n in (17, 4097, 9001):
        x = np.stack(list(int64_signals(n).values()))
        *_, stats, plans, fixed, ints, _ = encode_and_read(H, x, level, name=f"i64 L{level} n={n}")
        check_stats(stats, fixed, ints, level, f"i64 L{level} n={n}")


@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("level", [0, 5])
def test_float_streams_through_the_fused_quantiser(H, dt, level):
    for n in (15, 4097, 6001):
        x = np.stack(list(float_signals(n, dt).values()))
        for quanta in (None, np.array([1e-3, 1e-4, 0.5], dt)):
            *_, stats, plans, fixed, ints, _ = encode_and_read(H, x, level, quanta, name=f"{dt.__name__} L{level} n={n}")
            check_stats(stats, fixed, ints, level, f"{dt.__name__} L{level} n={n}")


def test_the_analysis_paths_are_all_reached(H):
    """The matrix reaches every analysis path: k_enc_fixed's frames and the ones it declines, full and short frames
    through k_enc_analyze, narrow, wide, CONSTANT, wasted bits and the int32-fit exclusion."""
    seen = set()
    for level in (0, 5):
        bs = S.PRESETS[level][0]
        x = np.stack(list(int32_signals(8195, bs).values()))
        *_, stats, plans, fixed, ints, _ = encode_and_read(H, x, level)
        seen.add(("fixed-taken", level, bool(fixed.any())))
        seen.add(("fixed-declined", level, bool((~fixed).any())))
        modes = set(stats["mode"][~fixed].ravel().tolist())
        seen.update(("mode", level, m) for m in modes)
        seen.add(("wasted", level, bool((stats["wasted"][~fixed] > 0).any())))
        seen.add(("bad", level, bool((stats["bad"][~fixed] != 0).any())))
    for level in (0, 5):
        assert {("fixed-declined", level, True), ("mode", level, 1), ("mode", level, 2), ("mode", level, 3),
                ("wasted", level, True), ("bad", level, True)} <= seen, (level, seen)
    assert ("fixed-taken", 0, True) in seen


@pytest.mark.parametrize("level", [0, 2, 3, 5, 8])
def test_adversarial_full_scale_signals(H, level, oracle):
    """Nine full-scale signals: strictly valid, exact analysis, and (reported) size next to the oracle encoder's.  The
    size is not asserted: on these near-singular autocorrelations Levinson-Durbin is ill-conditioned and both encoders
    land on very different coefficients of the same order (DESIGN.md section 2)."""
    sig = adversarial(20000)
    x = np.stack(list(sig.values()))
    comp, st, nb, stats, plans, fixed, ints, _ = encode_and_read(H, x, level, name=f"adversarial L{level}")
    assert check_stats(stats, fixed, ints, level, f"adversarial L{level}") > 0 or level <= 2


def test_emulator_reproduces_the_frozen_gpu_bytes(H, golden_dir):
    """The CPU pin of the encoder's bytes: SHA-256 of the emulator's output for the five small configs at levels 0, 5
    and 8 equals what the B200 produced (tests/golden/gpu_encoded_sha256.json, scripts/freeze_gpu_sha.py)."""
    from oracle.small_configs import small_configs

    want = json.load(open(os.path.join(golden_dir, "gpu_encoded_sha256.json")))
    for name, x in small_configs().items():
        for level in (0, 5, 8):
            comp = H.encode(x, level)[0]
            got = hashlib.sha256(comp.tobytes()).hexdigest()
            w = want[f"{name}/L{level}"]
            assert (got, comp.size) == (w["sha256"], w["nbytes"]), (name, level)


def test_size_within_two_percent_of_the_oracle_on_realistic_wide_signals(H, oracle):
    """Sine plus noise at amplitudes 2^20 .. 2^30, periods 9, 50 and 400: each stream within 1.02 x the oracle
    encoder.  Ill-conditioned full-scale tones without noise are excluded (DESIGN.md section 2)."""
    rng = np.random.default_rng(17)
    n = 12000
    i = np.arange(n)
    rows, names = [], []
    for e in (20, 23, 26, 28, 30):
        for period in (9, 50, 400):
            amp = 2.0 ** e * 0.95
            rows.append(_i32(amp * np.sin(2 * np.pi * i / period + 0.3) + rng.normal(0, amp / 2 ** 10, n)))
            names.append((e, period))
    x = np.stack(rows)
    for level in (3, 5, 8):
        c, st, nb, *_ = H.encode(x, level)
        oc, ost, onb = oracle.encode(x, level)
        for s, nm in enumerate(names):
            assert nb[s] <= 1.02 * onb[s], (level, nm, int(nb[s]), int(onb[s]))


def test_narrow_plans_keep_the_32_bit_condition(H):
    """On narrow frames the design lowers the coefficient precision until sum|q| * max|x| < 2^30 (the tile decoder's
    and k_encode's 32-bit datapath).  Signals that need the lowering get it, and every narrow plan satisfies it."""
    rng = np.random.default_rng(23)
    n = 4096 * 6 + 100
    i = np.arange(n)
    rows = [_i32(a * np.sin(2 * np.pi * i / p) + rng.normal(0, s, n))
            for a, p, s in ((2 ** 21, 50, 2 ** 9), (2 ** 18, 300, 2 ** 6), (2 ** 16, 9, 30), (2 ** 21, 1000, 2 ** 11))]
    x = np.stack(rows)
    lowered = 0
    for level in (5, 8):
        prec = S.PRESETS[level][3]
        *_, stats, plans, fixed, ints, streams = encode_and_read(H, x, level)
        for idx in np.ndindex(plans.shape):
            pl, stt = plans[idx], stats[idx]
            if pl["mode"] != 2 or not pl["ok1"]:
                continue
            if not pl["wide1"]:
                q = np.abs(pl["qlp"][:pl["ord1"]].astype(np.int64)).sum()
                mac = int(q) * max(-int(stt["mn"]), int(stt["mx"]))
                assert mac < 2 ** 30, (level, idx, mac)
                lowered += int(pl["prec1"]) < prec
    assert lowered > 0
