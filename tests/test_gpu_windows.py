"""Per-stream sample windows on the GPU (FlacArray.to_windows, array_decompress_windows, fab_decode_windows): every
window must equal the full decode's [s, a:b] bit for bit, on every decoder path."""
import glob
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def fa():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import __graft_entry__ as g

    g.build()
    import flacarray_b200

    return flacarray_b200


def _host(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)


def _windows(rng, n_stream, n, bs, count=40):
    """Random, overlapping, repeated, unsorted and empty windows, plus stream edges and frame boundaries."""
    w = [(int(rng.integers(0, n_stream)), *sorted(int(v) for v in rng.integers(0, n + 1, 2))) for _ in range(count)]
    for s in range(n_stream):
        w += [(s, 0, n), (s, 0, 1), (s, n - 1, n), (s, n, n), (s, 0, 0), (s, bs - 2, min(n, bs + 2)), (s, bs, min(n, bs + 1))]
    w += w[:7]
    w = [w[i] for i in rng.permutation(len(w))]
    return tuple(np.array([x[i] for x in w], np.int64) for i in range(3))


def _assert_windows(data, offs, full, streams, first, last):
    data = _host(data)
    assert offs.shape == (streams.size + 1,) and offs[0] == 0
    for i in range(streams.size):
        got, want = data[offs[i]:offs[i + 1]], full[streams[i], first[i]:last[i]]
        assert got.dtype == want.dtype and np.array_equal(got.view(np.uint8), np.ascontiguousarray(want).view(np.uint8)), i


def _signal(rng, dt, shape):
    n = shape[-1]
    walk = np.cumsum(rng.normal(0, 1, shape), axis=-1)
    if dt == np.int32:
        return (walk * 300).astype(np.int32)
    if dt == np.int64:
        return (walk * 3e4).astype(np.int64) + 2 ** 40
    x = (walk + rng.normal(0, 0.1, shape) + 5.0).astype(dt)
    return x[..., :n]


@pytest.mark.parametrize("level", [0, 5, 8])
@pytest.mark.parametrize("dt", [np.int32, np.int64, np.float32, np.float64])
def test_to_windows_matches_to_array(fa, dt, level):
    import torch

    rng = np.random.default_rng(7000 + level * 10 + np.dtype(dt).itemsize + (2 if np.dtype(dt).kind == "f" else 0))
    bs = 1152 if level == 0 else 4096
    x = _signal(rng, dt, (2, 3, 12000))
    kw = dict(quanta=1e-3) if np.dtype(dt).kind == "f" else {}
    for dev in (False, True):
        src = torch.from_numpy(x).cuda() if dev else x
        far = fa.FlacArray.from_array(src, level=level, **kw)
        full = _host(far.to_array()).reshape(6, -1)
        streams, first, last = _windows(rng, 6, x.shape[-1], bs)
        data, offs = far.to_windows(streams, first, last)
        assert hasattr(data, "is_cuda") == dev
        _assert_windows(data, offs, full, streams, first, last)
        # tuple-of-index-arrays form (as np.nonzero returns)
        data, offs = far.to_windows(np.unravel_index(streams, (2, 3)), first, last)
        _assert_windows(data, offs, full, streams, first, last)
    # 1-D array: the single stream 0, scalar bounds broadcast
    far = fa.FlacArray.from_array(x[0, 0], level=level, **kw)
    full = _host(far.to_array()).reshape(1, -1)
    data, offs = far.to_windows(np.zeros(3, np.int64), 100, 5000)
    _assert_windows(data, offs, full, np.zeros(3, np.int64), np.full(3, 100), np.full(3, 5000))


def test_windows_on_oracle_encoded_streams(fa, oracle):
    """Foreign streams (no frame-size table): the sync scan, once per referenced stream."""
    import torch

    rng = np.random.default_rng(71)
    x = np.cumsum(rng.integers(-2000, 2001, (5, 20000)), axis=1).astype(np.int32)
    c, s, nb = oracle.encode(x, 5)
    streams, first, last = _windows(rng, 5, x.shape[1], 4096)
    for comp in (c, torch.from_numpy(c).cuda()):
        data, offs = fa.array_decompress_windows(comp, x.shape[1], s, nb, streams, first, last)
        _assert_windows(data, offs, x, streams, first, last)
    # a subset of the streams: the others are never scanned
    keep = streams[streams % 2 == 0]
    data, offs = fa.array_decompress_windows(c, x.shape[1], s, nb, keep, 0, 20000)
    _assert_windows(data, offs, x, keep, np.zeros_like(keep), np.full_like(keep, 20000))


def test_windows_on_golden_third_party_streams(fa, golden_dir):
    """FFmpeg's streams: every stereo assignment, which the general decoder takes."""
    rng = np.random.default_rng(72)
    for p in sorted(glob.glob(os.path.join(golden_dir, "ffmpeg_*.npz"))):
        with np.load(p) as z:
            stream, samples = z["stream"], z["samples"]
        n, nch = samples.shape
        want = samples.reshape(1, -1).view(np.int64) if nch == 2 else samples.reshape(1, -1)
        streams, first, last = _windows(rng, 1, n, 4096, count=10)
        data, offs = fa.array_decompress_windows(stream, n, np.zeros(1, np.int64), np.array([stream.size], np.int64),
                                                 streams, first, last, is_int64=(nch == 2))
        _assert_windows(data, offs, want, streams, first, last)


@pytest.mark.parametrize("log2_amp", [14, 30])
def test_windows_guess_and_miss(fa, oracle, log2_amp):
    """The signals of test_decode_32bit_prediction_guess_and_miss: missed 32-bit guesses come back through the general
    decoder, per window."""
    rng = np.random.default_rng(1000 + log2_amp)
    n = 3 * 4096 + 1500
    i = np.arange(n)
    env = np.sin(np.pi * (i % 4096) / 4096.0) ** 2
    amp = float(2 ** log2_amp - 2 ** (log2_amp - 4))
    rows = []
    for k in range(40):
        ph = rng.uniform(0, 2 * np.pi)
        xk = amp * env * np.sin(2 * np.pi * i / rng.uniform(37.0, 400.0) + ph) + rng.normal(0, 3.0, n)
        rows.append(np.clip(np.rint(xk), -2 ** 31, 2 ** 31 - 1))
    x = np.array(rows).astype(np.int32)
    for c, s, nb in (oracle.encode(x, 5), fa.array_compress(x, level=5)[:3]):
        streams, first, last = _windows(rng, 40, n, 4096)
        data, offs = fa.array_decompress_windows(c, n, s, nb, streams, first, last)
        _assert_windows(data, offs, x, streams, first, last)


def test_windows_flipped_byte_raises(fa):
    rng = np.random.default_rng(73)
    x = np.cumsum(rng.integers(-900, 901, (2, 9000)), axis=1).astype(np.int32)
    comp, starts, nbytes, _, _ = fa.array_compress(x, level=5)
    data, offs = fa.array_decompress_windows(comp, 9000, starts, nbytes, [1, 0], [0, 0], [9000, 9000])
    _assert_windows(data, offs, x, np.array([1, 0]), np.array([0, 0]), np.array([9000, 9000]))
    bad = comp.copy()
    bad[int(starts[1]) + 3000] ^= 0x10
    with pytest.raises(RuntimeError):
        fa.array_decompress_windows(bad, 9000, starts, nbytes, [1], [0], [9000])
    # a window of the intact stream does not touch the damage
    data, offs = fa.array_decompress_windows(bad, 9000, starts, nbytes, [0], [100], [8000])
    _assert_windows(data, offs, x, np.array([0]), np.array([100]), np.array([8000]))


def test_more_than_65535_windows(fa):
    import torch

    rng = np.random.default_rng(74)
    x = ((np.cumsum(rng.normal(0, 1, (7, 50000)), axis=1)) + 3.0).astype(np.float32)
    far = fa.FlacArray.from_array(torch.from_numpy(x).cuda(), quanta=1e-3)
    full = _host(far.to_array())
    nw = 70001
    streams = rng.integers(0, 7, nw)
    first = rng.integers(0, 49990, nw)
    last = first + rng.integers(0, 11, nw)
    data, offs = far.to_windows(streams, first, last)
    data = _host(data)
    want = np.concatenate([full[s, a:b] for s, a, b in zip(streams, first, last)])
    assert np.array_equal(data.view(np.uint32), want.view(np.uint32))
    assert offs[-1] == (last - first).sum()


def _device_records(fa, x, streams, first, last):
    import torch

    from flacarray_b200 import libflacarray as lf

    comp, starts, nbytes, _, _ = fa.array_compress(torch.from_numpy(x).cuda(), level=5)
    dev = comp.device
    st = lf.to_device(starts.reshape(-1), dev, torch.int64)
    nb = lf.to_device(nbytes.reshape(-1), dev, torch.int64)
    woff = np.concatenate([[0], np.cumsum(last - first)]).astype(np.int64)
    rec = [lf.to_device(np.asarray(v, np.int64), dev, torch.int64) for v in (streams, first, last, woff[:-1])]
    return comp, st, nb, rec, int(woff[-1]), int(nb.max())


def test_windows_workspace_too_small(fa):
    """With a caller workspace below fab_decode_windows_workspace_bytes the call fails with ERROR_ALLOC, launches
    nothing; with enough it decodes."""
    import torch

    from flacarray_b200 import _lib

    L = _lib.lib()
    rng = np.random.default_rng(75)
    x = np.cumsum(rng.integers(-500, 501, (16, 40000)), axis=1).astype(np.int32)
    streams = rng.integers(0, 16, 300)
    first = rng.integers(0, 39000, 300)
    last = first + 1000
    comp, st, nb, rec, total, max_nb = _device_records(fa, x, streams, first, last)
    dev = comp.device
    ctx = _lib.context(dev)
    need = L.fab_decode_windows_workspace_bytes(16, 40000, 300, 0, 4096)
    assert need > 0 and L.fab_decode_windows_workspace_bytes(0, 40000, 300, 0, 4096) == 0
    assert need < L.fab_decode_windows_workspace_bytes(16, 40000, 300000, 0, 4096)
    out = torch.empty(total, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    try:
        small = torch.empty(need - 256, dtype=torch.uint8, device=dev)
        ctx.set_workspace(small)
        n0 = ctx.launches()
        rc = L.fab_decode_windows(ctx.handle, comp.data_ptr(), st.data_ptr(), nb.data_ptr(), 16, 40000, 0,
                                  *[r.data_ptr() for r in rec], 300, out.data_ptr(), None, None, max_nb, 4096, stream)
        assert rc == 1 and "workspace too small" in ctx.last_error()
        assert ctx.launches() == n0
        ws = torch.empty(need, dtype=torch.uint8, device=dev)
        ctx.set_workspace(ws)
        rc = L.fab_decode_windows(ctx.handle, comp.data_ptr(), st.data_ptr(), nb.data_ptr(), 16, 40000, 0,
                                  *[r.data_ptr() for r in rec], 300, out.data_ptr(), None, None, max_nb, 4096, stream)
        assert rc == 0 and L.fab_finish(ctx.handle, stream) == 0
    finally:
        ctx.set_workspace(None)
    data = out.cpu().numpy()
    want = np.concatenate([x[s, a:b] for s, a, b in zip(streams, first, last)])
    assert np.array_equal(data, want)


def test_windows_bad_records_rejected_on_device(fa):
    import torch

    from flacarray_b200 import _lib

    L = _lib.lib()
    rng = np.random.default_rng(76)
    x = np.cumsum(rng.integers(-500, 501, (4, 20000)), axis=1).astype(np.int32)
    streams, first, last = np.array([0, 4, 1, 2, 3]), np.array([0, 0, -1, 30, 10]), np.array([50, 50, 10, 20, 20001])
    comp, st, nb, rec, _, max_nb = _device_records(fa, x, streams, first, last)
    dev = comp.device
    ctx = _lib.context(dev)
    out = torch.zeros(256, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    woff = torch.tensor([0, 60, 70, 80, 90], dtype=torch.int64, device=dev)
    rc = L.fab_decode_windows(ctx.handle, comp.data_ptr(), st.data_ptr(), nb.data_ptr(), 4, 20000, 0, rec[0].data_ptr(),
                              rec[1].data_ptr(), rec[2].data_ptr(), woff.data_ptr(), 5, out.data_ptr(), None, None, max_nb,
                              4096, stream)
    assert rc == 0
    assert L.fab_finish(ctx.handle, stream) == 1 << 17
    o = out.cpu().numpy()
    assert np.array_equal(o[:50], x[0, :50]) and not o[50:].any()


def test_windows_launch_count_does_not_grow_with_windows(fa):
    import torch

    from flacarray_b200 import _lib

    rng = np.random.default_rng(77)
    x = np.cumsum(rng.integers(-500, 501, (10, 60000)), axis=1).astype(np.int32)
    comp, starts, nbytes, _, _ = fa.array_compress(torch.from_numpy(x).cuda(), level=5)
    ctx = _lib.context(comp.device)
    counts = []
    for nw in (10, 10000):
        streams = np.arange(nw) % 10                       # the same ten streams
        first = rng.integers(0, 59000, nw)
        last = first + rng.integers(1, 1000, nw)
        n0 = ctx.launches()
        data, offs = fa.array_decompress_windows(comp, 60000, starts, nbytes, streams, first, last)
        counts.append(ctx.launches() - n0)
        _assert_windows(data, offs, x, streams, first, last)
    assert counts[0] == counts[1] > 0
