"""Ranges of out-of-threshold samples on the GPU (fab_flag_count / fab_flag_write, array_flag_ranges,
FlacArray.flag_ranges).

* all four dtypes at levels 0 and 5, from device and host bytes, with per-stream thresholds at mean +- k * std from
  stats(), scalar and one-sided thresholds, pads 0, 3 and larger than the stream, a keep mask and a stream slice with
  negative bounds: equal to the ranges numpy finds in to_array();
* grouping invariance (many decode groups give the same ranges as one);
* more than 65 535 rows, with flags planted in both grid.y slabs;
* every valid stream of tests/flac_corpus.py and the FFmpeg golden streams;
* composition with to_windows: every window holds a flagged sample and no flagged sample lies outside the windows;
* on_error="fill" around a corrupted stream in both residencies, and "raise" with the decode's message;
* the C entry points' argument checks (nothing launched) and the caller's workspace (too small: ERROR_ALLOC).
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
import hostsim_flags as HF  # noqa: E402

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


def _data(dt, shape, seed):
    """Random walks with planted glitches: single-sample spikes, short bursts and rail values."""
    rng = np.random.default_rng(seed)
    walk = np.cumsum(rng.integers(-30, 31, shape), axis=-1)
    flat = walk.reshape(-1, shape[-1])
    for r in range(flat.shape[0]):
        for j in rng.integers(0, shape[-1], 6):
            flat[r, j:j + int(rng.integers(1, 4))] += int(rng.choice([-1, 1])) * 100000
    flat[0, :3] = 10 ** 6
    flat[-1, -2:] = -(10 ** 6)
    if np.dtype(dt).kind == "f":
        return (walk * 1e-3 + 3.0).astype(dt)
    x = walk * (1 << 20 if dt == np.int64 else 1)
    if dt == np.int64:
        x.reshape(-1, shape[-1])[1, 100:103] = np.iinfo(np.int64).max
    return x.astype(dt)


def _far(fa, dt, data, level, where):
    import torch

    src = torch.from_numpy(data).cuda() if where == "device" else data
    if np.dtype(dt).kind == "f":
        return fa.FlacArray.from_array(src, quanta=1e-4, level=level)
    return fa.FlacArray.from_array(src, level=level)


def _expect(arr, lo, hi, pad, keep=None, first=0, last=None):
    """The ranges numpy finds in arr [..., n] (to_array's values) for thresholds lo / hi (None, a scalar or one value per
    stream) over samples [first, last): (stream, first, last, nflagged) with flat stream indices."""
    n = arr.shape[-1]
    last = n if last is None else last
    lead = arr.shape[:-1]
    rows = arr.reshape(-1, n)[:, first:last]
    ns = rows.shape[0]
    v = rows.astype(np.float64) if rows.dtype.kind == "f" else rows

    def side(t, rnd):
        if t is None:
            return None
        t = np.asarray(t).reshape(-1)
        if v.dtype.kind == "i" and t.dtype.kind == "f":     # integers: x < ceil(lo), x > floor(hi), exactly
            t = rnd(t).astype(np.int64)
        return np.broadcast_to(t, (ns,))[:, None]

    lo_, hi_ = side(lo, np.ceil), side(hi, np.floor)
    flags = np.zeros(rows.shape, bool)
    if lo_ is not None:
        flags |= v < lo_
    if hi_ is not None:
        flags |= v > hi_
    sel = np.arange(ns) if keep is None else np.flatnonzero(np.asarray(keep).reshape(-1))
    s, f, l_, nf = HF.reference(flags[sel], pad, sample0=first)
    nflag = np.full(ns, -1, np.int64)
    nflag[sel] = nf
    return sel[s] if s.size else s, f, l_, nflag.reshape(lead)


def _same(got, want):
    for g, w, name in zip(got, want, ("stream", "first", "last", "nflagged")):
        g = np.asarray(g)
        assert g.dtype == np.int64 and g.shape == np.asarray(w).shape and np.array_equal(g, w), (name, g, w)


def _sigma_thresholds(far, k, stream_slice=None):
    s = far.stats(stream_slice=stream_slice)
    return s.mean - k * s.std, s.mean + k * s.std


@pytest.mark.parametrize("dt", DTYPES, ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("level", [0, 5])
@pytest.mark.parametrize("where", ["device", "host"])
def test_flag_ranges_match_numpy(fa, dt, level, where):
    n = 10000
    data = _data(dt, (2, 3, n), 70 + level + np.dtype(dt).itemsize)
    far = _far(fa, dt, data, level, where)
    arr = _host(far.to_array())
    flt = np.dtype(dt).kind == "f"
    lo, hi = _sigma_thresholds(far, 3.0)
    if not flt:
        lo, hi = np.ceil(lo).astype(np.int64), np.floor(hi).astype(np.int64)
    keep = np.zeros((2, 3), bool)
    keep[0, 1] = keep[1, 0] = keep[1, 2] = True
    for pad in (0, 3, n + 5):
        r = far.flag_ranges(lo=lo, hi=hi, pad=pad)
        assert type(r).__name__ == "FlagRanges" and r.nflagged.shape == (2, 3)
        _same(r, _expect(arr, lo, hi, pad))
        _same(far.flag_ranges(lo=lo, hi=hi, pad=pad, keep=keep), _expect(arr, lo, hi, pad, keep=keep))
        r = far.flag_ranges(lo=lo.reshape(-1), hi=hi, pad=pad, stream_slice=slice(-8000, -2345))
        _same(r, _expect(arr, lo, hi, pad, first=n - 8000, last=n - 2345))
    med = float(np.median(arr))
    _same(far.flag_ranges(hi=med, pad=2), _expect(arr, None, med, 2))
    _same(far.flag_ranges(lo=med), _expect(arr, med, None, 0))
    if not flt:
        # float thresholds on integers: x < ceil(lo), x > floor(hi)
        _same(far.flag_ranges(lo=med - 0.5, hi=med + 40.5, pad=1), _expect(arr, np.ceil(med - 0.5),
                                                                          np.floor(med + 40.5), 1))
    # lo > hi flags every sample: one range per stream
    r = far.flag_ranges(lo=1.0, hi=0.0)
    assert r.stream.tolist() == list(range(6)) and np.all(r.nflagged == n)


@pytest.mark.parametrize("dt", [np.int32, np.float64], ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("where", ["device", "host"])
def test_grouping_invariance(fa, dt, where, monkeypatch):
    from flacarray_b200 import libflacarray as lf

    data = _data(dt, (37, 5000), 7)
    far = _far(fa, dt, data, 5, where)
    keep = np.ones(37, bool)
    keep[[3, 20]] = False
    lo, hi = _sigma_thresholds(far, 2.0)

    def run():
        return [far.flag_ranges(lo=lo, hi=hi, pad=p) for p in (0, 4)] + \
            [far.flag_ranges(lo=lo, hi=hi, pad=1, keep=keep, stream_slice=slice(17, 4000))]

    want = run()
    row = 5000 * np.dtype(dt).itemsize
    monkeypatch.setattr(lf, "_STATS_GROUP_BYTES", 4 * row + 5)         # groups of 4 streams
    monkeypatch.setattr(lf, "_PIPE_MIN_BYTES", 0)
    monkeypatch.setattr(lf, "_PIPE_CHUNK_BYTES", 3 * row)               # host: groups of 3 (and the ramp)
    assert len(lf._stats_ranges(37, row, lf._STATS_GROUP_BYTES)) == 10
    assert len(lf._chunk_ranges(37, row)) > 5
    for g, w in zip(run(), want):
        _same(g, w)
    assert want[0].stream.size > 37


def test_more_than_65535_rows(fa):
    import torch

    ns, n = 70000, 64
    rng = np.random.default_rng(65536)
    x = rng.integers(-1000, 1001, (ns, n)).astype(np.int32)
    x[7, 3] = 5000
    x[65535 + 9, 60:64] = -5000
    x[ns - 1, 0] = 7000
    for far in (fa.FlacArray.from_array(torch.from_numpy(x).cuda(), level=5), fa.FlacArray.from_array(x, level=5)):
        r = far.flag_ranges(lo=-1500, hi=1500, pad=2)
        _same(r, _expect(x, -1500, 1500, 2))
        assert r.stream.tolist() == [7, 65535 + 9, ns - 1]
        assert r.first.tolist() == [1, 58, 0] and r.last.tolist() == [6, 64, 3]


def test_foreign_streams(fa, golden_dir):
    import torch

    for case in FC.valid_cases():
        if not case.full:
            continue
        comp, st, nb = case.buffer()
        exp = case.expect.reshape(len(case.streams), case.stream_size)
        lo, hi = int(np.percentile(exp, 10)), int(np.percentile(exp, 90))
        for src in (comp, torch.from_numpy(comp).cuda()):
            r = fa.array_flag_ranges(src, case.stream_size, st, nb, lo=lo, hi=hi, pad=3, is_int64=case.is_int64)
            want = _expect(exp, lo, hi, 3)
            lead = np.asarray(st).shape if isinstance(st, np.ndarray) else (1,)
            _same(r, want[:3] + (want[3].reshape(lead),))
    files = sorted(glob.glob(os.path.join(golden_dir, "ffmpeg_*.npz")))
    assert files
    for f in files:
        z = np.load(f)
        stream, samples = z["stream"], z["samples"]
        is64 = samples.shape[1] == 2
        exp = (FC.as_i64(samples) if is64 else samples[:, 0].copy()).reshape(1, -1)
        lo, hi = int(np.percentile(exp, 5)), int(np.percentile(exp, 95))
        r = fa.array_flag_ranges(stream, exp.size, 0, stream.size, lo=lo, hi=hi, pad=10, is_int64=is64)
        _same(r, _expect(exp, lo, hi, 10))


@pytest.mark.parametrize("dt", [np.int32, np.float32], ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("where", ["device", "host"])
def test_composition_with_to_windows(fa, dt, where):
    data = _data(dt, (3, 4, 6000), 31)
    far = _far(fa, dt, data, 5, where)
    arr = _host(far.to_array()).reshape(12, -1)
    lo, hi = _sigma_thresholds(far, 2.5)
    for pad in (0, 7):
        r = far.flag_ranges(lo=lo, hi=hi, pad=pad, stream_slice=slice(500, 5500))
        vals, offs = far.to_windows(r.stream, r.first, r.last)
        vals = _host(vals).astype(np.float64)
        lo_f, hi_f = lo.reshape(-1)[r.stream], hi.reshape(-1)[r.stream]
        covered = np.zeros((12, 6000), bool)
        for i in range(r.stream.size):
            w = vals[offs[i]:offs[i + 1]]
            assert w.size == r.last[i] - r.first[i] and np.any((w < lo_f[i]) | (w > hi_f[i]))
            covered[r.stream[i], r.first[i]:r.last[i]] = True
        v = arr.astype(np.float64)[:, 500:5500]
        flagged = (v < lo.reshape(-1, 1)) | (v > hi.reshape(-1, 1))
        assert not np.any(flagged & ~covered[:, 500:5500])
        assert np.array_equal(flagged.sum(axis=1), r.nflagged.reshape(-1))


@pytest.mark.parametrize("dt", DTYPES, ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("where", ["device", "host"])
def test_fill_and_raise(fa, dt, where):
    data = _data(dt, (4, 5, 5000), 1700)
    far = _far(fa, dt, data, 5, where)
    arr = _host(far.to_array())
    lo, hi = _sigma_thresholds(far, 2.0)
    want = _expect(arr, lo, hi, 1)
    st = np.asarray(_host(far.stream_starts)).reshape(-1)
    nb = np.asarray(_host(far.stream_nbytes)).reshape(-1)
    far._compressed[int(st[11] + nb[11] * 2 // 3)] ^= 0x5A
    r, status = far.flag_ranges(lo=lo, hi=hi, pad=1, on_error="fill")
    want_status = np.zeros((4, 5), np.int32)
    want_status[2, 1] = PROCESS
    assert np.array_equal(status, want_status)
    ok = want[0] != 11
    nfl = want[3].copy()
    nfl[2, 1] = -1
    _same(r, (want[0][ok], want[1][ok], want[2][ok], nfl))
    keep = np.zeros((4, 5), bool)
    keep[2, 0:3] = True
    r, status = far.flag_ranges(lo=lo, hi=hi, pad=1, keep=keep, on_error="fill")
    assert status[2].tolist() == [0, PROCESS, 0, 0, 0] and status.sum() == PROCESS
    assert set(r.stream.tolist()) <= {10, 12} and r.nflagged[2, 1] == -1 and r.nflagged[0, 0] == -1
    with pytest.raises(RuntimeError, match="Decoding failed, return code = "):
        far.flag_ranges(lo=lo, hi=hi)


def test_one_dimensional(fa):
    x = np.cumsum(np.random.default_rng(2).integers(-9, 10, 9000)).astype(np.float32)
    x[4000:4003] = 1e4
    far = fa.FlacArray.from_array(x, quanta=1e-3)
    r = far.flag_ranges(hi=5e3, pad=10)
    assert r.stream.tolist() == [0] and r.first.tolist() == [3990] and r.last.tolist() == [4013]
    assert r.nflagged.tolist() == [3]


def test_c_entry_point_arguments(fa):
    import torch

    from flacarray_b200 import _lib

    L = _lib.lib()
    ctx = _lib.context(0)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    n_rows, n = 4, 100000
    rows = torch.arange(n_rows * n, dtype=torch.int32, device="cuda")
    lo = torch.full((n_rows,), 1000, dtype=torch.int64, device="cuda")
    hi = torch.full((n_rows,), 2 * n + 5000, dtype=torch.int64, device="cuda")
    cnt = torch.full((2 * n_rows,), -5, dtype=torch.int64, device="cuda")
    need = int(L.fab_flag_ranges_workspace_bytes(n_rows, n, 0))
    assert need > n_rows * n // 8 and L.fab_flag_ranges_workspace_bytes(0, n, 0) == -1
    assert L.fab_flag_ranges_workspace_bytes(n_rows, 0, 0) == -1
    work = torch.empty(need, dtype=torch.uint8, device="cuda")

    def p(t):
        return C.c_void_p(t.data_ptr()) if t is not None else None

    def count(n_rows_=n_rows, n_=n, rows_=rows, lo_=lo, offsets=None, gains=None, pad=0, work_=work, wb=need,
              out=cnt):
        return L.fab_flag_count(ctx.handle, p(rows_), 0, n_rows_, n_, p(lo_), p(hi), p(offsets), p(gains), None, pad,
                                p(work_), wb, p(out), p(out[n_rows:]) if out is not None else None, st)

    launches = ctx.launches()
    assert count(n_rows_=0) == 1 << 2 and count(n_=0) == 1 << 3 and count(pad=-1) == 1 << 17
    assert count(offsets=lo) == 1 << 19
    assert count(rows_=None) == 1 << 0 and count(lo_=None) == 1 << 0 and count(out=None) == 1 << 0
    assert count(work_=None) == 1 << 0
    assert count(wb=need - 1) == 1 << 0 and "workspace too small" in ctx.last_error()
    assert count(work_=work[8:], wb=need - 8) == 1 << 19        # a workspace off a 16-byte boundary
    assert ctx.launches() == launches
    assert count(pad=2) == 0
    assert L.fab_finish(ctx.handle, st) == 0
    x = rows.view(n_rows, n).cpu().numpy().astype(np.int64)
    flags = (x < 1000) | (x > 2 * n + 5000)
    want = HF.reference(flags, 2, sample0=100)
    nr = np.bincount(want[0], minlength=n_rows)
    assert cnt[:n_rows].cpu().tolist() == flags.sum(axis=1).tolist() and cnt[n_rows:].cpu().tolist() == nr.tolist()
    assert nr.tolist() == [1, 0, 1, 1]
    first = torch.full((4,), -9, dtype=torch.int64, device="cuda")
    last = torch.full((4,), -9, dtype=torch.int64, device="cuda")
    base = torch.tensor(np.concatenate([[0], np.cumsum(nr)[:-1]]), dtype=torch.int64, device="cuda")

    def write(wb=need, base_=base, pad=2):
        return L.fab_flag_write(ctx.handle, p(rows), 0, n_rows, n, None, pad, p(work), wb, p(base_), 100, p(first),
                                p(last), st)

    launches = ctx.launches()
    assert write(wb=need - 256) == 1 << 0 and write(base_=None) == 1 << 0 and write(pad=-3) == 1 << 17
    assert ctx.launches() == launches
    assert write() == 0 and L.fab_finish(ctx.handle, st) == 0
    assert first.cpu().tolist() == want[1].tolist() + [-9]
    assert last.cpu().tolist() == want[2].tolist() + [-9]
