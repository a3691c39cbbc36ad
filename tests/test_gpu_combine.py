"""Weighted sums across streams on the GPU (fab_combine_rows, array_combine, FlacArray.combine).

* all four dtypes at levels 0, 5 and 8, from device and host bytes, with groups None, labels with -1, i % 7, pairs with
  weights +1 / -1 and n_groups above the largest label, each over the full range and a stream slice: bit-identical to
  the numpy fold over to_array();
* grouping invariance: with the group caps shrunk so that groups straddle decode calls (and host staging gathers),
  the bits do not change;
* more than 65 535 segments, with values planted in both grid.y slabs;
* on_error="fill" around a corrupted stream (the fold over the good streams), "raise" with the decode's message, and a
  corrupted stream that is left out;
* a 1-D FlacArray and every stream left out;
* the C entry point: argument checks, device-side segment checks and recovery, one launch per slab.
"""
import ctypes as C
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "hostsim"))

import hostsim_combine as HC  # noqa: E402

pytestmark = pytest.mark.gpu

DTYPES = [np.int32, np.int64, np.float32, np.float64]
PROCESS = 1 << 14
BAD_SEGMENT = 1 << 17


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


def _same(got, want):
    got, want = np.ascontiguousarray(_host(got)), np.ascontiguousarray(want)
    return got.dtype == want.dtype and got.shape == want.shape and np.array_equal(got.view(np.uint8), want.view(np.uint8))


def _data(dt, shape, seed):
    rng = np.random.default_rng(seed)
    walk = np.cumsum(rng.integers(-300, 301, shape), axis=-1)
    if np.dtype(dt).kind == "f":
        return (walk * 1e-3 + rng.normal(0, 1e-3, shape) + 3.0).astype(dt)
    x = walk * ((1 << 44) + 12345 if dt == np.int64 else 1)        # int64 above 2^53: float64() rounds
    x.reshape(-1, shape[-1])[0, ::97] = np.iinfo(dt).max
    x.reshape(-1, shape[-1])[-1, 5::89] = np.iinfo(dt).min
    return x.astype(dt)


def _far(fa, dt, data, level, where):
    import torch

    src = torch.from_numpy(data).cuda() if where == "device" else data
    if np.dtype(dt).kind == "f":
        return fa.FlacArray.from_array(src, quanta=1e-4, level=level)
    return fa.FlacArray.from_array(src, level=level)


def _groupings(n_stream, seed):
    """(name, weights, groups, n_groups) of the covered groupings over n_stream streams."""
    rng = np.random.default_rng(seed)
    lab = rng.integers(-1, 4, n_stream)
    pairs = np.arange(n_stream) // 2
    pairs[-1] = -1 if n_stream % 2 else pairs[-1]
    return [
        ("common", None, None, None),
        ("labels", rng.uniform(-1, 1, n_stream), lab, None),
        ("mod7", np.full(n_stream, 1.0 / 3.0), np.arange(n_stream) % 7, None),
        ("pairs", np.where(np.arange(n_stream) % 2 == 0, 1.0, -1.0), pairs, None),
        ("wide", rng.uniform(-1, 1, n_stream), np.arange(n_stream) % 3, 9),
    ]


def _want(x, weights, groups, n_groups, ok=None):
    """The numpy fold over to_array() rows x [n_stream, n], shaped like combine returns it."""
    n_stream = x.shape[0]
    w = np.ones(n_stream) if weights is None else np.asarray(weights, np.float64).reshape(-1)
    if groups is None:
        return HC.fold(x, w, np.zeros(n_stream, np.int64), 1, ok)[0]
    g = np.asarray(groups).reshape(-1)
    n_out = int(g.max()) + 1 if n_groups is None else n_groups
    return HC.fold(x, w, g, n_out, ok)


@pytest.mark.parametrize("dt", DTYPES, ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("level", [0, 5, 8])
@pytest.mark.parametrize("where", ["device", "host"])
def test_combine_matches_fold(fa, dt, level, where):
    import torch

    n = 10000
    data = _data(dt, (3, 7, n), 60 + level + np.dtype(dt).itemsize)
    far = _far(fa, dt, data, level, where)
    x = _host(far.to_array()).reshape(21, n)
    for name, w, g, ng in _groupings(21, level):
        for sl in (None, slice(1234, -2000)):
            got = far.combine(weights=w, groups=None if g is None else g.reshape(3, 7), n_groups=ng, stream_slice=sl)
            assert isinstance(got, torch.Tensor) == (where == "device") and (not hasattr(got, "is_cuda") or got.is_cuda)
            xs = x if sl is None else x[:, sl]
            assert _same(got, _want(xs, w, g, ng)), (name, sl)
        # flat groups give the same result
        if g is not None:
            assert _same(far.combine(weights=w, groups=g, n_groups=ng), _want(x, w, g, ng)), name


@pytest.mark.parametrize("dt", [np.int64, np.float32], ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("where", ["device", "host"])
def test_grouping_invariance(fa, dt, where, monkeypatch):
    from flacarray_b200 import libflacarray as lf

    n = 5000
    data = _data(dt, (37, n), 7)
    far = _far(fa, dt, data, 5, where)
    x = _host(far.to_array())
    cases = [(None, None, None), (np.random.default_rng(1).uniform(-1, 1, 37), np.arange(37) % 7, None),
             (None, np.where(np.arange(37) < 30, 0, -1), 2)]
    want = [far.combine(weights=w, groups=g, n_groups=ng) for w, g, ng in cases]
    for (w, g, ng), v in zip(cases, want):
        assert _same(v, _want(x, w, g, ng))
    row = n * np.dtype(dt).itemsize
    monkeypatch.setattr(lf, "_STATS_GROUP_BYTES", 4 * row + 5)         # device: groups of 4 streams
    monkeypatch.setattr(lf, "_PIPE_MIN_BYTES", 0)
    monkeypatch.setattr(lf, "_PIPE_CHUNK_BYTES", 3 * row)               # host: groups of 3 (and the ramp)
    gathered = []
    real = lf._group_bytes

    def spy(comp, starts, nbytes):
        part, rel = real(comp, starts, nbytes)
        gathered.append(part.size == int(nbytes.sum()) and int((starts + nbytes).max() - starts.min()) > part.size)
        return part, rel

    monkeypatch.setattr(lf, "_group_bytes", spy)
    got = [far.combine(weights=w, groups=g, n_groups=ng) for w, g, ng in cases]
    for g, v in zip(got, want):
        assert _same(g, _host(v))
    if where == "host":
        assert any(gathered)                    # the interleaved groups staged gathered bytes


def test_more_than_65535_segments(fa):
    import torch

    ns, n = 70000, 64
    rng = np.random.default_rng(65536)
    x = rng.integers(-1000, 1001, (ns, n)).astype(np.int32)
    x[7, 3] = np.iinfo(np.int32).max
    x[65535 + 9, 60] = np.iinfo(np.int32).min
    w = rng.uniform(-1, 1, ns)
    far = fa.FlacArray.from_array(torch.from_numpy(x).cuda(), level=5)
    got = far.combine(weights=w, groups=np.arange(ns))
    want = w[:, None] * x.astype(np.float64) + 0.0
    assert _same(got, want)
    assert _host(got)[65535 + 9, 60] == w[65535 + 9] * np.iinfo(np.int32).min
    got = fa.FlacArray.from_array(x, level=5).combine(weights=w, groups=np.arange(ns)[::-1].copy())
    assert _same(got, want[::-1])


@pytest.mark.parametrize("dt", DTYPES, ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("where", ["device", "host"])
def test_fill_and_raise(fa, dt, where):
    n_stream = 40
    data = _data(dt, (n_stream, 5000), 1700)
    far = _far(fa, dt, data, 5, where)
    x = _host(far.to_array())
    st = np.asarray(far.stream_starts).reshape(-1)
    nb = np.asarray(far.stream_nbytes).reshape(-1)
    pos = int(st[17] + nb[17] * 2 // 3)
    far._compressed[pos] ^= 0x5A
    ok = np.ones(n_stream, bool)
    ok[17] = False
    w = np.random.default_rng(3).uniform(-1, 1, n_stream)
    for g in (None, np.arange(n_stream) % 3):
        got, status = far.combine(weights=w, groups=g, on_error="fill")
        want_status = np.zeros(n_stream, np.int32)
        want_status[17] = PROCESS
        assert np.array_equal(status, want_status)
        assert _same(got, _want(x, w, g, None, ok))
    with pytest.raises(RuntimeError, match="Decoding failed, return code = "):
        far.combine()
    with pytest.raises(RuntimeError, match="Decoding failed, return code = "):
        far.to_array()
    # a stream that is left out is not examined: no error, status 0
    g = np.zeros(n_stream, np.int64)
    g[17] = -1
    assert _same(far.combine(weights=w, groups=g), _want(x, w, g, None, ok))
    got, status = far.combine(weights=w, groups=g, on_error="fill")
    assert not status.any() and _same(got, _want(x, w, g, None, ok))


def test_one_dimensional_and_everything_left_out(fa):
    import torch

    x = np.cumsum(np.random.default_rng(2).integers(-9, 10, 9000)).astype(np.float32)
    far = fa.FlacArray.from_array(x, quanta=1e-3)
    back = far.to_array()
    assert _same(far.combine(), back.astype(np.float64) + 0.0)
    assert _same(far.combine(weights=[0.5], groups=[0], n_groups=2),
                 np.stack([0.5 * back.astype(np.float64) + 0.0, np.zeros(9000)]))
    got, status = far.combine(stream_slice=slice(100, 200), on_error="fill")
    assert got.shape == (100,) and status.shape == (1,) and status[0] == 0
    far2 = fa.FlacArray.from_array(torch.zeros((3, 100), dtype=torch.int64, device="cuda") + 5)
    got, status = far2.combine(groups=np.full(3, -1), n_groups=3, on_error="fill")
    assert got.is_cuda and got.shape == (3, 100) and not got.any() and status.tolist() == [0, 0, 0]
    got = far2.combine(groups=np.full(3, -1))
    assert got.shape == (0, 100)


def test_c_entry_point(fa):
    import torch

    from flacarray_b200 import _lib

    L = _lib.lib()
    ctx = _lib.context(0)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    n_rows, n = 6, 1000
    rows = torch.arange(n_rows * n, dtype=torch.int32, device="cuda").view(n_rows, n) - 2500
    w = torch.tensor([1.0, -2.0, 0.25, 1.0 / 3.0, 3.0, -1.0], dtype=torch.float64, device="cuda")
    seg = torch.tensor([0, 2, 5, 6], dtype=torch.int64, device="cuda")
    seg_out = torch.tensor([0, 2, 3], dtype=torch.int64, device="cuda")
    out = torch.zeros((4, n), dtype=torch.float64, device="cuda")

    def p(t):
        return C.c_void_p(t.data_ptr()) if t is not None else None

    def call(rows_=rows, n_rows_=n_rows, n_=n, offsets=None, gains=None, w_=w, seg_=seg, seg_out_=seg_out, n_seg=3,
             out_=out, n_out=4, is_int64=0):
        return L.fab_combine_rows(ctx.handle, p(rows_), is_int64, n_rows_, n_, p(offsets), p(gains), None, p(w_),
                                  p(seg_), p(seg_out_), n_seg, p(out_), n_out, st)

    launches = ctx.launches()
    assert call(n_rows_=0) == 1 << 2 and call(n_seg=0) == 1 << 2 and call(n_out=0) == 1 << 2 and call(n_=0) == 1 << 3
    assert call(rows_=None) == 1 << 0 and call(w_=None) == 1 << 0 and call(seg_=None) == 1 << 0
    assert call(seg_out_=None) == 1 << 0 and call(out_=None) == 1 << 0
    assert call(offsets=w) == 1 << 19 and call(gains=w) == 1 << 19
    unaligned = torch.zeros(n_rows * n + 1, dtype=torch.int32, device="cuda")[1:]
    assert call(rows_=unaligned, is_int64=1) == 1 << 19
    assert call(out_=out.view(-1)[1:].view(torch.uint8)[4:]) == 1 << 19
    assert ctx.launches() == launches
    assert L.fab_finish(ctx.handle, st) == 0
    # a good call: one launch, the fold
    assert call() == 0 and ctx.launches() == launches + 1
    assert L.fab_finish(ctx.handle, st) == 0
    xr, wr = rows.cpu().numpy(), w.cpu().numpy()
    want = HC.fold(xr, wr, np.array([0, 0, 2, 2, 2, 3]), 4)
    assert _same(out, want)
    # bad records: flagged in the error mask, their rows untouched, the others computed; the context recovers
    out.zero_()
    assert call(seg_out_=torch.tensor([0, 2, 7], dtype=torch.int64, device="cuda")) == 0      # row 7 of 4
    assert L.fab_finish(ctx.handle, st) == BAD_SEGMENT
    o = out.cpu().numpy()
    assert _same(o[0], want[0]) and _same(o[2], want[2]) and not o[1].any() and not o[3].any()
    out.zero_()
    assert call(seg_=torch.tensor([0, 4, 2, 6], dtype=torch.int64, device="cuda")) == 0          # [4, 2) is refused
    assert L.fab_finish(ctx.handle, st) == BAD_SEGMENT
    o = out.cpu().numpy()
    assert _same(o[0], HC.fold(xr[:4], wr[:4], np.zeros(4, np.int64), 1)[0]) and not o[1].any() and not o[2].any()
    assert _same(o[3], HC.fold(xr[2:], wr[2:], np.zeros(4, np.int64), 1)[0])
    out.zero_()
    assert call() == 0 and L.fab_finish(ctx.handle, st) == 0
    assert _same(out, want)
    # one launch per 65 535 segments
    ns = 70000
    rows2 = torch.ones((ns, 8), dtype=torch.int32, device="cuda")
    w2 = torch.ones(ns, dtype=torch.float64, device="cuda")
    seg2 = torch.arange(ns + 1, dtype=torch.int64, device="cuda")
    out2 = torch.zeros((ns, 8), dtype=torch.float64, device="cuda")
    before = ctx.launches()
    assert call(rows2, ns, 8, None, None, w2, seg2, seg2[:ns], ns, out2, ns) == 0
    assert L.fab_finish(ctx.handle, st) == 0
    assert ctx.launches() == before + 2 and bool((out2 == 1.0).all())
