"""Projections onto templates on the GPU (fab_project_rows, array_project, FlacArray.project).

* all four dtypes, from device and host bytes, 1, 3, 16 and 37 templates, over the full range and a negative stream
  slice: bit-identical to the numpy reference applied to to_array(), and device and host residency give the same bits;
* grouping invariance: with the group caps shrunk so that streams go to the device in several decode calls, the bits
  do not change;
* keep with keep_indices, 1-D templates (the template axis dropped), torch templates, and combine()'s common mode as a
  template;
* on_error="fill" around a corrupted stream (NaN row and status) and "raise" with the decode's message;
* more than 65 535 rows at small n;
* the C entry point: argument checks, a caller-supplied workspace that is too small, launches per call.
"""
import ctypes as C
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "hostsim"))

import hostsim_project as HP  # noqa: E402

pytestmark = pytest.mark.gpu

DTYPES = [np.int32, np.int64, np.float32, np.float64]
PROCESS = 1 << 14


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


def _far(fa, dt, data, where, level=5):
    import torch

    src = torch.from_numpy(data).cuda() if where == "device" else data
    if np.dtype(dt).kind == "f":
        return fa.FlacArray.from_array(src, quanta=1e-4, level=level)
    return fa.FlacArray.from_array(src, level=level)


def _templates(n_tmpl, n, seed):
    """Legendre polynomials 0.., then sine / cosine pairs, then random templates."""
    rng = np.random.default_rng(seed)
    s = np.linspace(-1.0, 1.0, n)
    rows = [np.polynomial.legendre.Legendre.basis(k)(s) for k in range(min(n_tmpl, 3))]
    k = 1
    while len(rows) < min(n_tmpl, 19):
        rows += [np.sin(2 * np.pi * k * np.arange(n) / 1000.0), np.cos(2 * np.pi * k * np.arange(n) / 1000.0)]
        k += 1
    while len(rows) < n_tmpl:
        rows.append(rng.normal(0, 1, n))
    return np.stack(rows[:n_tmpl])


def _want(x, t, ok=None):
    """The numpy reference over to_array() rows x [..., n], shaped like project returns it."""
    lead = x.shape[:-1]
    t2 = np.atleast_2d(t)
    out = HP.reference(x.reshape(-1, x.shape[-1]), t2, ok=None if ok is None else np.asarray(ok).reshape(-1))
    return out.reshape(lead + ((t2.shape[0],) if np.ndim(t) == 2 else ()))


@pytest.mark.parametrize("dt", DTYPES, ids=lambda d: np.dtype(d).name)
def test_project_matches_reference(fa, dt):
    import torch

    n = 9000
    data = _data(dt, (3, 7, n), 60 + np.dtype(dt).itemsize)
    far_d = _far(fa, dt, data, "device")
    far_h = _far(fa, dt, data, "host")
    x = _host(far_d.to_array())
    assert _same(_host(far_h.to_array()), x)
    for n_tmpl in (1, 3, 16, 37):
        for sl in (None, slice(1234, -2000)):
            xs = x if sl is None else x[..., sl]
            t = _templates(n_tmpl, xs.shape[-1], n_tmpl)
            want = _want(xs, t)
            got = far_d.project(t, stream_slice=sl)
            assert isinstance(got, torch.Tensor) and got.is_cuda and got.dtype == torch.float64
            assert _same(got, want), (n_tmpl, sl)
            got_h = far_h.project(t, stream_slice=sl)
            assert isinstance(got_h, np.ndarray) and _same(got_h, want), (n_tmpl, sl)


@pytest.mark.parametrize("dt", [np.int64, np.float32], ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("where", ["device", "host"])
def test_grouping_invariance(fa, dt, where, monkeypatch):
    from flacarray_b200 import libflacarray as lf

    n = 5000
    data = _data(dt, (37, n), 7)
    far = _far(fa, dt, data, where)
    x = _host(far.to_array())
    t = _templates(5, n, 3)
    want = far.project(t)
    assert _same(want, _want(x, t))
    row = n * np.dtype(dt).itemsize
    monkeypatch.setattr(lf, "_STATS_GROUP_BYTES", 4 * row + 5)         # device: groups of 4 streams
    monkeypatch.setattr(lf, "_PIPE_MIN_BYTES", 0)
    monkeypatch.setattr(lf, "_PIPE_CHUNK_BYTES", 3 * row)               # host: groups of 3 (and the ramp)
    calls = []
    real = lf.project_device

    def spy(rows, *a):
        calls.append(a[1])
        return real(rows, *a)

    monkeypatch.setattr(lf, "project_device", spy)
    assert _same(far.project(t), _host(want))
    assert len(calls) > 3 and sum(calls) == 37


def test_keep_one_dimensional_torch_and_common_mode(fa):
    import torch

    n = 6000
    data = _data(np.float32, (4, 5, n), 11)
    far = _far(fa, np.float32, data, "device")
    x = _host(far.to_array())
    keep = np.zeros((4, 5), bool)
    keep[[0, 2, 3], [1, 4, 0]] = True
    t = _templates(3, n, 5)
    got, idx = far.project(t, keep=keep, keep_indices=True)
    assert idx == [(0, 1), (2, 4), (3, 0)]
    assert _same(got, _want(x[keep], t))
    assert _same(far.project(t, keep=keep), _want(x[keep], t))
    # 1-D templates drop the template axis; torch templates on the device or the host give the same bits
    t1 = t[1]
    assert _same(far.project(t1), _want(x, t1))
    assert _same(far.project(torch.from_numpy(t1).cuda()), _want(x, t1))
    assert _same(far.project(torch.from_numpy(t).float()), _want(x, t.astype(np.float32)))
    # the common mode of combine() as a template: coupling of every detector to it
    cm = far.combine()
    got = far.project(cm)
    assert got.shape == (4, 5) and _same(got, _want(x, _host(cm)))
    # a 1-D FlacArray gives one value per template (a scalar for 1-D templates)
    far1 = fa.FlacArray.from_array(data[1, 2], quanta=1e-4)
    x1 = far1.to_array()
    assert _same(far1.project(t), _want(x1[None], t)[0])
    assert _same(far1.project(t1[100:], stream_slice=slice(100, None)), _want(x1[None, 100:], t1[100:])[0])
    # every stream left out
    none = far.project(t, keep=np.zeros((4, 5), bool))
    assert none.shape == (0, 3) and none.is_cuda


@pytest.mark.parametrize("dt", DTYPES, ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("where", ["device", "host"])
def test_fill_and_raise(fa, dt, where):
    n_stream = 40
    data = _data(dt, (n_stream, 5000), 1700)
    far = _far(fa, dt, data, where)
    x = _host(far.to_array())
    st = np.asarray(far.stream_starts).reshape(-1)
    nb = np.asarray(far.stream_nbytes).reshape(-1)
    pos = int(st[17] + nb[17] * 2 // 3)
    far._compressed[pos] ^= 0x5A
    ok = np.ones(n_stream, bool)
    ok[17] = False
    t = _templates(3, 5000, 1)
    got, status = far.project(t, on_error="fill")
    want_status = np.zeros(n_stream, np.int32)
    want_status[17] = PROCESS
    assert np.array_equal(status, want_status)
    assert _same(got, _want(x, t, ok))
    assert np.isnan(_host(got)[17]).all()
    with pytest.raises(RuntimeError, match="Decoding failed, return code = "):
        far.project(t)


def test_more_than_65535_rows(fa):
    import torch

    ns, n = 70000, 64
    rng = np.random.default_rng(65536)
    x = rng.integers(-1000, 1001, (ns, n)).astype(np.int32)
    x[7, 3] = np.iinfo(np.int32).max
    x[65535 + 9, 60] = np.iinfo(np.int32).min
    t = _templates(3, n, 2)
    far = fa.FlacArray.from_array(torch.from_numpy(x).cuda(), level=5)
    assert _same(far.project(t), HP.reference(x, t))
    assert _same(fa.FlacArray.from_array(x, level=5).project(t[2]), HP.reference(x, t[2:])[:, 0])


def test_array_project(fa):
    data = _data(np.float64, (6, 7000), 9)
    comp, starts, nbytes, off, gain = fa.array_compress(data, level=5, quanta=1e-4)
    x = fa.array_decompress(comp, 7000, starts, nbytes, stream_offsets=off, stream_gains=gain, is_int64=True)
    t = _templates(4, 2000, 4)
    got = fa.array_project(comp, 7000, starts, nbytes, t, stream_offsets=off, stream_gains=gain,
                           first_stream_sample=3000, last_stream_sample=5000, is_int64=True)
    assert isinstance(got, np.ndarray) and _same(got, _want(x[:, 3000:5000], t))
    keep = np.array([True, False, True, True, False, False])
    got, status = fa.array_project(comp, 7000, starts, nbytes, t[0], stream_offsets=off, stream_gains=gain, keep=keep,
                                   first_stream_sample=3000, last_stream_sample=5000, is_int64=True, on_error="fill")
    assert _same(got, _want(x[keep, 3000:5000], t[0])) and status.tolist() == [0, 0, 0]


def test_c_entry_point(fa):
    import torch

    from flacarray_b200 import _lib

    L = _lib.lib()
    ctx = _lib.context(0)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    n_rows, n, n_tmpl = 6, 9000, 3
    rows = torch.arange(n_rows * n, dtype=torch.int32, device="cuda").view(n_rows, n) - 25000
    tm = torch.from_numpy(_templates(n_tmpl, n, 8)).cuda()
    out = torch.zeros((n_rows, n_tmpl), dtype=torch.float64, device="cuda")

    def p(t):
        return C.c_void_p(t.data_ptr()) if t is not None else None

    def call(rows_=rows, n_rows_=n_rows, n_=n, offsets=None, gains=None, status=None, tm_=tm, n_tmpl_=n_tmpl, out_=out,
             is_int64=0):
        return L.fab_project_rows(ctx.handle, p(rows_), is_int64, n_rows_, n_, p(offsets), p(gains), p(status), p(tm_),
                                  n_tmpl_, p(out_), st)

    ws = L.fab_project_rows_workspace_bytes(n_rows, n, n_tmpl)
    assert ws >= n_rows * n_tmpl * 3 * 8 and ws % 256 == 0
    assert L.fab_project_rows_workspace_bytes(0, n, 1) == -1 and L.fab_project_rows_workspace_bytes(1, 0, 1) == -1
    assert L.fab_project_rows_workspace_bytes(1, n, 0) == -1
    launches = ctx.launches()
    assert call(n_rows_=0) == 1 << 2 and call(n_tmpl_=0) == 1 << 2 and call(n_=0) == 1 << 3
    assert call(rows_=None) == 1 << 0 and call(tm_=None) == 1 << 0 and call(out_=None) == 1 << 0
    assert call(offsets=tm) == 1 << 19 and call(gains=tm) == 1 << 19
    unaligned = torch.zeros(n_rows * n + 1, dtype=torch.int32, device="cuda")[1:]
    assert call(rows_=unaligned) == 0 and L.fab_finish(ctx.handle, st) == 0       # int32 rows: 4-byte aligned is enough
    launches += 2
    assert call(rows_=unaligned, is_int64=1) == 1 << 19
    assert call(out_=out.view(-1)[1:].view(torch.uint8)[4:]) == 1 << 19
    assert call(tm_=tm.view(-1)[1:].view(torch.uint8)[4:]) == 1 << 19
    assert ctx.launches() == launches
    # a good call: one pass-1 launch and the fold, bit-identical to the reference
    assert call() == 0 and ctx.launches() == launches + 2
    assert L.fab_finish(ctx.handle, st) == 0
    want = HP.reference(rows.cpu().numpy(), tm.cpu().numpy())
    assert _same(out, want)
    # status: NaN rows
    status = torch.tensor([0, 1 << 14, 0, 0, 0, 1 << 13], dtype=torch.int32, device="cuda")
    assert call(status=status) == 0 and L.fab_finish(ctx.handle, st) == 0
    o = out.cpu().numpy()
    assert np.isnan(o[[1, 5]]).all() and _same(o[[0, 2, 3, 4]], want[[0, 2, 3, 4]])
    # a caller-supplied workspace: too small fails with ERROR_ALLOC and launches nothing, large enough works
    small = torch.empty(ws - 256, dtype=torch.uint8, device="cuda")
    big = torch.empty(ws, dtype=torch.uint8, device="cuda")
    try:
        ctx.set_workspace(small)
        before = ctx.launches()
        assert call() == 1 << 0 and ctx.launches() == before
        assert "workspace too small" in ctx.last_error()
        ctx.set_workspace(big)
        out.zero_()
        assert call() == 0 and L.fab_finish(ctx.handle, st) == 0
        assert _same(out, want)
    finally:
        ctx.set_workspace(None)
    # more than 65 535 pieces: two pass-1 launches and the fold
    n2 = 65536 * 4096 + 5
    one = torch.ones((1, n2), dtype=torch.int32, device="cuda")
    t2 = torch.ones((1, n2), dtype=torch.float64, device="cuda")
    o2 = torch.zeros((1, 1), dtype=torch.float64, device="cuda")
    before = ctx.launches()
    assert call(one, 1, n2, tm_=t2, n_tmpl_=1, out_=o2) == 0 and L.fab_finish(ctx.handle, st) == 0
    assert ctx.launches() == before + 3 and float(o2[0, 0]) == float(n2)
    del one, t2
