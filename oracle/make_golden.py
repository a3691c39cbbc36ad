"""Generate the committed golden fixtures under tests/golden/.  TEST INFRASTRUCTURE ONLY.

Run in the build container (needs /root/reference for the quantiser vectors and the bundled FFmpeg
for the codec vectors):

    python -m oracle.make_golden

Fixtures (all small, .npz):
  quant_f32.npz / quant_f64.npz : inputs + (ints, offsets, gains) produced by the REFERENCE's own
        utils.c (oracle/_ref/libfa_utils.so, compiled from /root/reference) with and without
        quanta, and the restored floats from its int*_to_float*.
  ffmpeg_*.npz : complete 32-bps FLAC streams produced by FFmpeg's independent encoder (mono at
        two levels; stereo with each of the four channel assignments, incl. the 33-bit side
        channel) + the samples they must decode to.
  handmade_verbatim.npz : a frame assembled by hand here (VERBATIM subframe, CRC-8/16 computed in
        numpy) -- a known-answer vector that depends on neither codec.
"""
import os

import numpy as np

from . import ffmpeg_flac as ff
from . import oracle as O
from .flac_writer import crc8, crc16

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
SEED = 123456789  # demo.py:12


def tod(rng, shape, dtype, sigma=1.0):
    """The reference's fake detector data model (demo.py:70-97)."""
    n = shape[-1]
    lead = shape[:-1] + (1,)
    dc = 5 * sigma * (rng.random(size=lead) - 0.5)
    t = np.arange(n)
    minf = 5 / n
    wave = 2 * sigma * np.sin(2 * np.pi * 3 * minf * t) + 6 * sigma * np.sin(2 * np.pi * minf * t)
    scale = rng.random(size=lead)
    return (dc + scale * wave + rng.normal(0.0, sigma, shape)).astype(dtype)


def handmade_verbatim(samples):
    """One mono 32-bps frame with a VERBATIM subframe, wrapped as a full stream."""
    n = len(samples)
    assert 1 <= n <= 256
    hdr = bytearray([0xFF, 0xF8, (6 << 4) | 9, (0 << 4) | (7 << 1), 0x00, n - 1])
    hdr.append(crc8(hdr))
    body = bytearray([0b00000010])  # pad 0, type 000001, no wasted bits
    for s in samples:
        body += int(s & 0xFFFFFFFF).to_bytes(4, "big")
    frame = bytes(hdr) + bytes(body)
    frame += crc16(frame).to_bytes(2, "big")
    return ff.make_stream([frame], 1, max(n, 16), total_samples=n)


def main():
    os.makedirs(OUT, exist_ok=True)
    rng = np.random.default_rng(SEED)
    if O.ref_utils() is None:
        raise SystemExit("oracle/_ref/libfa_utils.so missing: run `make -C oracle` where /root/reference exists")

    for dt, idt, name, qs in ((np.float32, np.int32, "quant_f32", (1e-4, 1e-6)),
                              (np.float64, np.int64, "quant_f64", (1e-7, 1e-15))):
        data = tod(rng, (3, 1000), dt)
        data[1] *= 37.5
        data[2] -= 1000.25
        out = {"data": data}
        for i, q in enumerate(qs):
            qa = np.array([q, 2 * q, 0.5 * q], dt)
            ints, off, gain = O.float_to_int(data, qa, use_ref=True)
            out[f"quanta{i}"] = qa
            out[f"ints{i}"], out[f"off{i}"], out[f"gain{i}"] = ints, off, gain
            out[f"restored{i}"] = O.int_to_float(ints, off, gain, use_ref=True)
        ints, off, gain = O.float_to_int(data, None, use_ref=True)
        out["ints_auto"], out["off_auto"], out["gain_auto"] = ints, off, gain
        out["restored_auto"] = O.int_to_float(ints, off, gain, use_ref=True)
        const = np.full((2, 100), 3.7, dt)
        const[1] = 0.0
        ints, off, gain = O.float_to_int(const, None, use_ref=True)
        out["const"], out["ints_const"], out["off_const"], out["gain_const"] = const, ints, off, gain
        np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)

    if not ff.available():
        raise SystemExit("bundled FFmpeg FLAC codec unavailable")
    n = 12000
    walk = (np.cumsum(rng.integers(-1000, 1001, n)) + rng.integers(-50, 51, n)).astype(np.int32)
    noise = rng.integers(-2 ** 31, 2 ** 31, n, dtype=np.int64).astype(np.int32)
    noise[0], noise[1] = -2 ** 31, 2 ** 31 - 1
    small = np.round(tod(rng, (n,), np.float64) * 1e4).astype(np.int32)
    mono = {"walk": walk, "noise": noise, "tod": small}
    for nm, x in mono.items():
        for lvl in (0, 5, 8):
            fr, fs = ff.encode_frames(x.reshape(-1, 1), lvl)
            st = np.frombuffer(ff.make_stream(fr, 1, fs), np.uint8)
            np.savez_compressed(os.path.join(OUT, f"ffmpeg_mono_{nm}_l{lvl}.npz"), stream=st, samples=x.reshape(-1, 1),
                                blocksize=fs)
    left = walk.astype(np.int64)
    right = left + rng.integers(-30, 31, n)
    st2 = np.stack([left, right], 1).astype(np.int32)
    a64 = (np.cumsum(rng.integers(-2 ** 20, 2 ** 20, n)) + (2 ** 40) * 3).astype(np.int64)
    a64[:4] = [-2 ** 63, 2 ** 63 - 1, 2 ** 32, -2 ** 32]
    lohi = a64.view(np.int32).reshape(-1, 2)
    wide = np.stack([noise, noise[::-1]], 1)
    for nm, x in (("corr", st2), ("lohi", lohi), ("wide", wide)):
        for cm in ("indep", "left_side", "right_side", "mid_side"):
            fr, fs = ff.encode_frames(x, 5, ch_mode=cm)
            st = np.frombuffer(ff.make_stream(fr, 2, fs), np.uint8)
            np.savez_compressed(os.path.join(OUT, f"ffmpeg_stereo_{nm}_{cm}.npz"), stream=st, samples=x, blocksize=fs)
    hv = np.array([0, 1, -1, 2 ** 31 - 1, -2 ** 31, 123456789, -987654321] + list(range(-20, 21)), np.int64)
    st = np.frombuffer(handmade_verbatim(hv), np.uint8)
    np.savez_compressed(os.path.join(OUT, "handmade_verbatim.npz"), stream=st,
                        samples=hv.astype(np.int32).reshape(-1, 1), blocksize=max(len(hv), 16))
    print("golden fixtures written to", OUT)
    tot = sum(os.path.getsize(os.path.join(OUT, f)) for f in os.listdir(OUT))
    print("total bytes", tot)


if __name__ == "__main__":
    main()
