"""Per-stream sample windows (array_decompress_windows / fab_decode_windows) without a GPU: the host-side argument
checks of the Python layer, and the window index space of the kernel bodies through the host emulator (tests/hostsim)
against oracle-decoded slices."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostsim"))

from test_hostsim import _cases  # noqa: E402


@pytest.fixture(scope="module")
def H():
    import hostsim

    hostsim.lib()
    return hostsim


def _tiny():
    """Three fake streams of a 30-byte buffer: enough for the checks that run before any decoding."""
    comp = np.zeros(30, np.uint8)
    return comp, np.array([0, 10, 20], np.int64), np.array([10, 10, 10], np.int64)


@pytest.mark.parametrize("streams, first, last, msg", [
    ([0, 3], 0, 5, "stream index 3 is out of range for 3 streams"),
    ([-1], 0, 5, "stream index -1 is out of range"),
    ([0, 1], [0, -2], [5, 5], r"window 1 \[-2, 5\) lies outside the stream of 100 samples"),
    ([2], 0, 101, r"window 0 \[0, 101\) lies outside the stream"),
    ([0, 1, 2], [0, 7, 3], [5, 6, 3], "window 1: first sample 7 is larger than last sample 6"),
    ([0, 1], [0, 1, 2], 5, "streams, first and last must have the same length"),
    ([0, 1], 0, [5], "streams, first and last must have the same length"),
    ([0.5], 0, 5, "window streams must be integers"),
])
def test_window_arguments_are_checked_on_the_host(streams, first, last, msg):
    import flacarray_b200 as fa

    comp, st, nb = _tiny()
    with pytest.raises(RuntimeError, match=msg):
        fa.array_decompress_windows(comp, 100, st, nb, np.asarray(streams), np.asarray(first), np.asarray(last))


def test_window_offsets_and_gains_go_together():
    import flacarray_b200 as fa

    comp, st, nb = _tiny()
    with pytest.raises(RuntimeError, match="you must also provide the gains"):
        fa.array_decompress_windows(comp, 100, st, nb, [0], 0, 5, stream_offsets=np.zeros(3, np.float32))


def test_byte_windows_are_checked():
    import flacarray_b200 as fa

    comp, st, nb = _tiny()
    with pytest.raises(RuntimeError, match="outside the compressed buffer"):
        fa.array_decompress_windows(comp, 100, st, nb + 5, [0], 0, 5)


@pytest.mark.parametrize("restored, is_int64, dt", [(False, False, np.int32), (False, True, np.int64),
                                                     (True, False, np.float32), (True, True, np.float64)])
def test_zero_windows(restored, is_int64, dt):
    import flacarray_b200 as fa

    comp, st, nb = _tiny()
    fdt = np.float64 if is_int64 else np.float32
    kw = dict(stream_offsets=np.zeros(3, fdt), stream_gains=np.ones(3, fdt)) if restored else {}
    data, offsets = fa.array_decompress_windows(comp, 100, st, nb, np.zeros(0, np.int64), 0, 0, is_int64=is_int64, **kw)
    assert data.shape == (0,) and data.dtype == dt
    assert offsets.dtype == np.int64 and np.array_equal(offsets, [0])


def _draw_windows(rng, n_stream, n, bs):
    """Random windows plus the edge cases: stream start and end, across frame boundaries, whole streams, empty ones,
    repeats; overlapping and unsorted by construction."""
    w = []
    for _ in range(12):
        s = int(rng.integers(0, n_stream))
        a = int(rng.integers(0, n + 1))
        b = int(rng.integers(a, n + 1))
        w.append((s, a, b))
    for s in range(n_stream):
        w += [(s, 0, n), (s, 0, min(1, n)), (s, n - 1, n), (s, n, n), (s, 0, 0), (s, n // 2, n // 2)]
        for j in range(1, 4):
            c = j * bs
            if c < n:
                w += [(s, max(0, c - 3), min(n, c + 3)), (s, c, min(n, c + 1)), (s, max(0, c - 1), c)]
        w += [(s, 0, n)]                      # a repeat
    w += w[:5]                                # more repeats
    idx = rng.permutation(len(w))
    w = [w[i] for i in idx]
    return (np.array([x[0] for x in w], np.int64), np.array([x[1] for x in w], np.int64),
            np.array([x[2] for x in w], np.int64))


def _check(H, comp, st, nb, x, streams, first, last, bsh=4096, is_int64=False):
    y, offs, info = H.decode_windows(comp, st, nb, x.shape[1], streams, first, last, is_int64=is_int64, bsh=bsh)
    assert offs[-1] == (last - first).sum()
    for i in range(streams.size):
        got = y[offs[i]:offs[i + 1]]
        assert np.array_equal(got, x[streams[i], first[i]:last[i]]), (i, streams[i], first[i], last[i])
    return info


def test_window_bodies_on_own_and_foreign_streams(H, oracle):
    rng = np.random.default_rng(41)
    for name, x in _cases(rng).items():
        c, s, n, _, _ = H.encode(x, 5)          # frame-size table
        oc, os_, on = oracle.encode(x, 5)       # foreign: sync scan
        for comp, st, nb in ((c, s, n), (oc, os_, on)):
            ref = oracle.decode(comp, st, nb, x.shape[1])
            assert np.array_equal(ref, x), name
            streams, first, last = _draw_windows(rng, x.shape[0], x.shape[1], 4096)
            info = _check(H, comp, st, nb, ref, streams, first, last)
            assert info % 1000 == 0, name       # no stream needed the walker


def test_window_bodies_other_levels_and_hint_mismatch(H, oracle):
    """Levels 0 (1152-sample frames) and 8; a blocksize hint that is too small (more items than frames) or too large
    (the stream's frames outnumber the window's items: the stream goes to the walker, window by window)."""
    rng = np.random.default_rng(42)
    x = (np.cumsum(rng.integers(-3000, 3001, (3, 10000)), axis=1)).astype(np.int32)
    for level, bs in ((0, 1152), (8, 4096)):
        for comp, st, nb in (H.encode(x, level)[:3], oracle.encode(x, level)):
            streams, first, last = _draw_windows(rng, 3, x.shape[1], bs)
            assert _check(H, comp, st, nb, x, streams, first, last, bsh=bs) % 1000 == 0
            _check(H, comp, st, nb, x, streams, first, last, bsh=512)
            info = _check(H, comp, st, nb, x, streams, first, last, bsh=8192)
            if level == 0:
                assert info % 1000 > 0            # 1152-sample frames under an 8192 hint: walked


def test_window_bodies_int64_and_stereo(H, oracle):
    rng = np.random.default_rng(43)
    a = (np.cumsum(rng.integers(-2 ** 20, 2 ** 20, (2, 9000)), axis=1) + 2 ** 40 * 3).astype(np.int64)
    for comp, st, nb in (H.encode(a, 5)[:3], oracle.encode(a, 5)):
        streams, first, last = _draw_windows(rng, 2, a.shape[1], 4096)
        _check(H, comp, st, nb, a, streams, first, last, is_int64=True)


def test_window_bodies_on_golden_third_party_streams(H, golden_dir):
    import glob

    rng = np.random.default_rng(44)
    for p in sorted(glob.glob(os.path.join(golden_dir, "ffmpeg_*.npz"))):
        with np.load(p) as z:
            stream, samples = z["stream"], z["samples"]
        n, nch = samples.shape
        want = samples.reshape(1, -1).view(np.int64) if nch == 2 else samples.reshape(1, -1)
        streams, first, last = _draw_windows(rng, 1, n, 4096)
        _check(H, stream, np.zeros(1, np.int64), np.array([stream.size], np.int64), want, streams, first, last,
               is_int64=(nch == 2))


def test_window_bodies_guess_and_miss(H, oracle):
    """Frames whose 32-bit prediction guess misses go to the general decoder: window by window as well."""
    rng = np.random.default_rng(45)
    n = 2 * 4096 + 700
    i = np.arange(n)
    env = np.sin(np.pi * (i % 4096) / 4096.0) ** 2
    amp = float(2 ** 30 - 2 ** 26)
    x = np.array([np.clip(np.rint(amp * env * np.sin(2 * np.pi * i / per + 0.3) + rng.normal(0, 3.0, n)), -2 ** 31, 2 ** 31 - 1)
                  for per in (41.0, 113.0, 390.0)]).astype(np.int32)
    comp, st, nb = oracle.encode(x, 5)
    streams, first, last = _draw_windows(rng, 3, n, 4096)
    info = _check(H, comp, st, nb, x, streams, first, last)
    assert info >= 1000 and info % 1000 == 0


def test_bad_window_records_are_skipped_on_the_device(H):
    """The kernels' own record check: out-of-range slots and ranges set ERROR_DECODE_SAMPLE_RANGE (1 << 17)."""
    import ctypes as C

    rng = np.random.default_rng(46)
    x = np.cumsum(rng.integers(-900, 901, (2, 9000)), axis=1).astype(np.int32)
    c, s, n, _, _ = H.encode(x, 5)
    L = H.lib()
    cc = np.concatenate([c, np.zeros(64, np.uint8)])
    for ws, wf, wl in (([2], [0], [10]), ([-1], [0], [10]), ([0], [-1], [10]), ([1], [0], [9001]), ([0], [20], [10])):
        ws, wf, wl = (np.array(v, np.int64) for v in (ws, wf, wl))
        wo = np.zeros(1, np.int64)
        out = np.zeros(16, np.int32)
        info = C.c_int(0)
        err = L.hs_decode_windows(cc.ctypes.data, s.ctypes.data, n.ctypes.data, 2, 9000, 1, ws.ctypes.data, wf.ctypes.data,
                                  wl.ctypes.data, wo.ctypes.data, 1, 4096, out.ctypes.data, C.byref(info))
        assert err == 1 << 17 and not out.any()
