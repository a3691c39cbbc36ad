"""Per-stream, per-bin statistics on the GPU (fab_row_stats, array_stats, FlacArray.stats).

* all four dtypes at levels 0, 5 and 8, from device and host bytes, for the full range, a keep mask with keep_indices
  and a stream slice, with bins None, 1, 7, n - 1 and n: bit-identical to the Python-integer reference computed from
  the integers array_decompress returns; min / max equal to the decoded array's; mean / std close to numpy's float64;
* grouping invariance (many groups give the same bits as one) and bounded device memory with the group cap shrunk;
* more than 65 535 rows, with values planted in both grid.y slabs;
* every valid stream of tests/flac_corpus.py and the FFmpeg golden streams;
* on_error="fill" around a corrupted stream in both residencies, and "raise" with the decode's message;
* a 1-D FlacArray, keep that selects nothing, and the C entry point's argument checks and workspace rules.
"""
import ctypes as C
import glob
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, "hostsim"))

import flac_corpus as FC  # noqa: E402
import hostsim_stats as HS  # noqa: E402

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


def _all_same(a, b):
    return all(_same(x, y) for x, y in zip(a, b))


def _data(dt, shape, seed):
    rng = np.random.default_rng(seed)
    walk = np.cumsum(rng.integers(-300, 301, shape), axis=-1)
    if np.dtype(dt).kind == "f":
        return (walk * 1e-3 + rng.normal(0, 1e-3, shape) + 3.0).astype(dt)
    x = walk * (1 << 20 if dt == np.int64 else 1)
    x.reshape(-1, shape[-1])[0, ::97] = np.iinfo(dt).max        # extremes in one stream
    x.reshape(-1, shape[-1])[-1, 5::89] = np.iinfo(dt).min
    return x.astype(dt)


def _far(fa, dt, data, level, where):
    import torch

    src = torch.from_numpy(data).cuda() if where == "device" else data
    if np.dtype(dt).kind == "f":
        return fa.FlacArray.from_array(src, quanta=1e-4, level=level)
    return fa.FlacArray.from_array(src, level=level)


def _ints(fa, far):
    """The decoded integers of every stream, [..., n] int32 / int64 (array_decompress without offsets / gains)."""
    return _host(fa.array_decompress(far.compressed, far.stream_size, far.stream_starts, far.stream_nbytes,
                                     is_int64=far._is_int64, no_flatten=True))


def _reference(far, ints, bin, keep=None, first=0, last=None):
    """Python-integer reference of the selection, shaped like FlacArray.stats returns it."""
    last = far.stream_size if last is None else last
    lead = ints.shape[:-1]
    rows = ints.reshape(-1, ints.shape[-1])
    off = None if far.stream_offsets is None else np.asarray(far.stream_offsets).reshape(-1)
    gain = None if far.stream_gains is None else np.asarray(far.stream_gains).reshape(-1)
    if keep is not None:
        sel = np.flatnonzero(keep.reshape(-1))
        rows = rows[sel]
        off = None if off is None else off[sel]
        gain = None if gain is None else gain[sel]
        lead = (sel.size,)
    ref = HS.reference(rows[:, first:last], bin, offsets=off, gains=gain)
    tail = () if bin is None else (ref[0].shape[1],)
    return tuple(r.reshape(lead + tail) for r in ref)


def _check_sanity(stats, arr, bin, dt, far=None, ints=None):
    """min / max equal to the decoded array's, mean / std close to numpy float64 on it: within 2^-24 (float32) or 2^-40
    (float64) times the largest magnitude.  For float32 that magnitude is |x| + |coeff * i|: the restore rounds
    coeff * i and then off + coeff * i to float32, and coeff * i can be much larger than the sample x."""
    n = arr.shape[-1]
    scale = None
    if far is not None and far.stream_offsets is not None and np.dtype(dt).itemsize == 4:
        coeff = 1.0 / np.asarray(far.stream_gains, np.float64).reshape(arr.shape[:-1] + (1,))
        scale = np.abs(coeff) * np.abs(ints.astype(np.float64))
    length = n if bin is None else min(bin, n)
    nb = -(-n // length)
    pad = nb * length - n
    x = arr.astype(np.float64)
    for b in range(nb):
        seg = arr[..., b * length:(b + 1) * length]
        idx = (Ellipsis,) if bin is None else (Ellipsis, b)
        assert np.array_equal(stats.min[idx], seg.min(axis=-1)) and np.array_equal(stats.max[idx], seg.max(axis=-1))
        xs = x[..., b * length:(b + 1) * length]
        mag = np.abs(xs) if scale is None else np.abs(xs) + scale[..., b * length:(b + 1) * length]
        tol = mag.max(axis=-1) * (2.0 ** -24 if np.dtype(dt).itemsize == 4 else 2.0 ** -40) + 1e-300
        assert np.all(np.abs(stats.mean[idx] - xs.mean(axis=-1)) <= tol)
        assert np.all(np.abs(stats.std[idx] - xs.std(axis=-1)) <= tol)
    assert pad >= 0


@pytest.mark.parametrize("dt", DTYPES, ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("level", [0, 5, 8])
@pytest.mark.parametrize("where", ["device", "host"])
def test_stats_match_reference(fa, dt, level, where):
    n = 10000          # three 4096-sample frames; bins of n samples span several reducer pieces
    data = _data(dt, (2, 3, n), 40 + level + np.dtype(dt).itemsize)
    far = _far(fa, dt, data, level, where)
    ints = _ints(fa, far)
    full = _host(far.to_array())
    keep = np.zeros((2, 3), bool)
    keep[0, 1] = keep[1, 0] = keep[1, 2] = True
    for bin in (None, 1, 7, n - 1, n):
        s = far.stats(bin=bin)
        assert type(s).__name__ == "StreamStats"
        assert _all_same(s, _reference(far, ints, bin)), bin
        _check_sanity(s, full, bin, dt, far, ints)
        s, idx = far.stats(keep=keep, bin=bin, keep_indices=True)
        assert [tuple(i) for i in idx] == [(0, 1), (1, 0), (1, 2)]
        assert _all_same(s, _reference(far, ints, bin, keep=keep))
        m = n - 2345 - 1000 if bin == n - 1 else bin
        s = far.stats(stream_slice=slice(1000, -2345), bin=m)
        assert _all_same(s, _reference(far, ints, m, first=1000, last=n - 2345))
        _check_sanity(s, full[..., 1000:n - 2345], m, dt, far, ints[..., 1000:n - 2345])


@pytest.mark.parametrize("dt", [np.int32, np.float64], ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("where", ["device", "host"])
def test_grouping_invariance(fa, dt, where, monkeypatch):
    from flacarray_b200 import libflacarray as lf

    data = _data(dt, (37, 5000), 7)
    far = _far(fa, dt, data, 5, where)
    keep = np.ones(37, bool)
    keep[[3, 20]] = False
    want = [far.stats(bin=b) for b in (None, 333)] + [far.stats(keep=keep, stream_slice=slice(17, 4000), bin=100)]
    row = 5000 * np.dtype(dt).itemsize
    monkeypatch.setattr(lf, "_STATS_GROUP_BYTES", 4 * row + 5)         # groups of 4 streams
    monkeypatch.setattr(lf, "_PIPE_MIN_BYTES", 0)
    monkeypatch.setattr(lf, "_PIPE_CHUNK_BYTES", 3 * row)               # host: groups of 3 (and the ramp)
    assert len(lf._stats_ranges(37, row, lf._STATS_GROUP_BYTES)) == 10
    assert len(lf._chunk_ranges(37, row)) > 5
    got = [far.stats(bin=b) for b in (None, 333)] + [far.stats(keep=keep, stream_slice=slice(17, 4000), bin=100)]
    for g, w in zip(got, want):
        assert _all_same(g, w)


def test_bounded_device_memory(fa, monkeypatch):
    import torch

    from flacarray_b200 import libflacarray as lf

    ns, n = 64, 1 << 20
    x = torch.cumsum(torch.randint(-100, 101, (ns, n), device="cuda", dtype=torch.int32), dim=1, dtype=torch.int32)
    far = fa.FlacArray.from_array(x, level=1)
    del x
    want = far.stats(bin=1 << 16)
    cap = 32 << 20                                                 # decoded 256 MB -> 8 groups
    monkeypatch.setattr(lf, "_STATS_GROUP_BYTES", cap)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    got = far.stats(bin=1 << 16)
    rise = torch.cuda.max_memory_allocated() - base
    results = ns * 16 * (8 * 3 + 4 * 2) + 4 * ns + 8
    ws = int(fa.libflacarray._lib.lib().fab_row_stats_workspace_bytes(8, n, 1 << 16, 0))
    assert _all_same(got, want)
    assert rise <= cap + ws + results + (1 << 20), (rise, cap)     # + the groups' starts / nbytes, allocator rounding


def test_more_than_65535_rows(fa):
    import torch

    ns, n = 70000, 64
    rng = np.random.default_rng(65536)
    x = rng.integers(-1000, 1001, (ns, n)).astype(np.int32)
    x[7, 3] = np.iinfo(np.int32).max
    x[65535 + 9, 60] = np.iinfo(np.int32).min
    x[ns - 1] = np.iinfo(np.int32).min
    far = fa.FlacArray.from_array(torch.from_numpy(x).cuda(), level=5)
    for bin in (None, 10):
        s = far.stats(bin=bin)
        assert _all_same(s, _reference(far, x, bin))
    s = fa.FlacArray.from_array(x, level=5).stats(bin=None)
    assert s.max[7] == np.iinfo(np.int32).max and s.min[65535 + 9] == np.iinfo(np.int32).min


def test_foreign_streams(fa, golden_dir):
    import torch

    for case in FC.valid_cases():
        if not case.full:
            continue
        comp, st, nb = case.buffer()
        exp = case.expect.reshape(len(case.streams), case.stream_size)
        for bin in (None, 1000):
            for src in (comp, torch.from_numpy(comp).cuda()):
                s = fa.array_stats(src, case.stream_size, st, nb, bin=bin, is_int64=case.is_int64)
                ref = HS.reference(exp, bin)
                lead = (len(case.streams),) if len(case.streams) > 1 else ()
                ref = tuple(r.reshape(lead + (() if bin is None else (r.shape[1],))) for r in ref)
                assert _all_same(s, ref), case.name
    files = sorted(glob.glob(os.path.join(golden_dir, "ffmpeg_*.npz")))
    assert files
    for f in files:
        z = np.load(f)
        stream, samples = z["stream"], z["samples"]
        is64 = samples.shape[1] == 2
        exp = FC.as_i64(samples) if is64 else samples[:, 0].copy()
        for bin in (None, 4096):
            s = fa.array_stats(stream, exp.size, 0, stream.size, bin=bin, is_int64=is64)
            ref = HS.reference(exp.reshape(1, -1), bin)
            assert _all_same(s, tuple(r.reshape(() if bin is None else (-1,)) for r in ref)), f


@pytest.mark.parametrize("dt", DTYPES, ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("where", ["device", "host"])
def test_fill_and_raise(fa, dt, where):
    data = _data(dt, (4, 5, 5000), 1700)
    far = _far(fa, dt, data, 5, where)
    ints = _ints(fa, far)
    st = np.asarray(_host(far.stream_starts)).reshape(-1)
    nb = np.asarray(_host(far.stream_nbytes)).reshape(-1)
    pos = int(st[11] + nb[11] * 2 // 3)
    far._compressed[pos] ^= 0x5A
    ok = np.ones((4, 5), bool)
    ok[2, 1] = False
    flt = np.dtype(dt).kind == "f"
    for bin in (None, 777):
        s, status = far.stats(bin=bin, on_error="fill")
        want_status = np.zeros((4, 5), np.int32)
        want_status[2, 1] = PROCESS
        assert np.array_equal(status, want_status)
        ref = _reference(far, ints, bin)
        for g, w in zip(s, ref):
            assert _same(g[ok], w[ok])
        assert np.all(s.count[2, 1] == 0) and np.all(np.isnan(s.mean[2, 1])) and np.all(np.isnan(s.std[2, 1]))
        assert np.all(np.isnan(s.min[2, 1])) if flt else np.all(s.min[2, 1] == 0) and np.all(s.max[2, 1] == 0)
        keep = np.zeros((4, 5), bool)
        keep[2, 0:3] = True
        s, idx, status = far.stats(keep=keep, bin=bin, keep_indices=True, on_error="fill")
        assert status.tolist() == [0, PROCESS, 0] and len(idx) == 3
        assert _same(s.count[[0, 2]], ref[0][2, [0, 2]])
    with pytest.raises(RuntimeError, match="Decoding failed, return code = "):
        far.stats()
    with pytest.raises(RuntimeError, match="Decoding failed, return code = "):
        far.to_array()


def test_one_dimensional_and_empty_keep(fa):
    x = np.cumsum(np.random.default_rng(2).integers(-9, 10, 9000)).astype(np.float32)
    far = fa.FlacArray.from_array(x, quanta=1e-3)
    s = far.stats()
    assert all(v.shape == () for v in s)
    assert s.count == 9000 and s.min.dtype == np.float32 and s.min == far.to_array().min()
    s = far.stats(bin=4000)
    assert s.count.tolist() == [4000, 4000, 1000]
    far2 = fa.FlacArray.from_array(np.zeros((3, 100), np.int64))
    s, idx = far2.stats(keep=np.zeros(3, bool), bin=30, keep_indices=True)
    assert idx == [] and s.count.shape == (0, 4) and s.min.dtype == np.int64
    s, status = far2.stats(keep=np.zeros(3, bool), on_error="fill")
    assert s.mean.shape == (0,) and status.shape == (0,)


def test_c_entry_point_arguments(fa):
    import torch

    from flacarray_b200 import _lib

    L = _lib.lib()
    ctx = _lib.context(0)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rows = torch.arange(1000, dtype=torch.int32, device="cuda")
    outs = [torch.full((8,), -5, dtype=torch.int64, device="cuda") for _ in range(5)]

    def call(n_rows=2, n=500, bin=0, rows_=rows, offsets=None, gains=None, out=outs):
        p = [C.c_void_p(t.data_ptr()) if t is not None else None for t in (rows_, offsets, gains)]
        return L.fab_row_stats(ctx.handle, p[0], 0, n_rows, n, bin, p[1], p[2], None,
                               *[C.c_void_p(t.data_ptr()) if t is not None else None for t in out], st)

    launches = ctx.launches()
    assert call(n_rows=0) == 1 << 2 and call(n=0) == 1 << 3 and call(bin=-1) == 1 << 17
    assert call(n=1 << 33, bin=0) == 1 << 17
    assert call(offsets=outs[0]) == 1 << 19
    assert call(rows_=None) == 1 << 0
    assert call(out=outs[:4] + [None]) == 1 << 0
    assert ctx.launches() == launches
    assert L.fab_row_stats_workspace_bytes(2, 500, 0, 0) == 0
    assert L.fab_row_stats_workspace_bytes(2, 100000, 0, 0) > 0
    assert L.fab_row_stats_workspace_bytes(0, 100, 0, 0) == -1
    # a caller-supplied workspace that is too small: ERROR_ALLOC, no allocation
    big = torch.arange(4 * 100000, dtype=torch.int32, device="cuda")
    res = [torch.empty(4, dtype=torch.int64, device="cuda") for _ in range(5)]
    ws = torch.empty(256, dtype=torch.uint8, device="cuda")      # 4 rows x 13 pieces need 2912 bytes
    ctx.set_workspace(ws)
    try:
        assert call(n_rows=4, n=100000, rows_=big, out=res) == 1 << 0
        assert "workspace too small" in ctx.last_error()
    finally:
        ctx.set_workspace(None)
    assert call(n_rows=4, n=100000, rows_=big, out=res) == 0
    assert L.fab_finish(ctx.handle, st) == 0
    x = big.view(4, 100000).cpu().numpy().astype(np.int64)
    assert res[0].cpu().tolist() == [100000] * 4
    assert res[1].view(torch.int32)[:4].cpu().tolist() == x.min(axis=1).tolist()
    assert res[3].view(torch.float64).cpu().tolist() == [float(sum(int(v) for v in r)) / 100000 for r in x]
