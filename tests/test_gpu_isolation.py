"""Per-stream fault isolation (fab_decode_isolated, on_error="fill") and verify (fab_verify, array_verify,
FlacArray.verify) on the GPU.

* calls that mix good and bad streams report the bad ones and decode the rest bit for bit, in all four dtypes, from
  device and host bytes, with and without keep masks and sample windows; failed rows are 0 / NaN;
* verify rejects a stream exactly when a lone fab_decode of it raises, stream by stream and in one call per shape;
* the C entry points leave guard bands alone, overwrite every status entry, and leave the context usable;
* more than 65 535 streams: bad streams in both grid.y slabs;
* on_error="raise" is unchanged, call-level errors still raise, and the launch counts are those of fab_decode plus one
  fill launch per slab (verify: no restore).
"""
import ctypes as C
import functools
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

import flac_corpus as FC  # noqa: E402

pytestmark = pytest.mark.gpu

INIT, PROCESS = 1 << 13, 1 << 14
BAD = FC.invalid_cases() + FC.damage_cases()
DTYPES = [np.int32, np.int64, np.float32, np.float64]


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


@functools.lru_cache(maxsize=None)
def _good(stream_size, nch):
    """Two good streams of this shape from the library's encoder, and their integers."""
    import flacarray_b200 as fa

    rng = np.random.default_rng(stream_size * 7 + nch)
    x = np.cumsum(rng.integers(-500, 501, (2, stream_size)), axis=1)
    x = (x * 977 + (x << 33)).astype(np.int64) if nch == 2 else x.astype(np.int32)
    comp, st, nb = (_host(v) for v in fa.array_compress(x, level=5)[:3])
    return [bytes(comp[s:s + n]) for s, n in zip(st, nb)], x


def _call(streams):
    starts = np.cumsum([0] + [len(p) for p in streams[:-1]]).astype(np.int64)
    return np.frombuffer(b"".join(streams), np.uint8).copy(), starts, np.array([len(p) for p in streams], np.int64)


def _sandwich(case):
    """[good, bad, good, bad] back to back, and the good integers."""
    (g0, g1), x = _good(case.stream_size, case.nch)
    comp, st, nb = _call([g0, case.streams[0], g1, case.streams[0]])
    return comp, st, nb, x


def _restore(nch, k=4):
    rng = np.random.default_rng(99 + nch)
    fdt = np.float64 if nch == 2 else np.float32
    return rng.normal(0, 100, k).astype(fdt), (10.0 ** rng.uniform(-1, 5, k)).astype(fdt)


def _cases_for(dt):
    nch = 2 if np.dtype(dt).itemsize == 8 else 1
    return [c for c in BAD if c.nch == nch]


# ---- mixed calls ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("dt", DTYPES, ids=lambda d: np.dtype(d).name)
def test_mixed_calls_fill(fa, oracle, dt):
    import torch

    flt = np.dtype(dt).kind == "f"
    is64 = np.dtype(dt).itemsize == 8
    cases = _cases_for(dt)
    assert cases
    for case in cases:
        comp, st, nb, x = _sandwich(case)
        n = case.stream_size
        kw = dict(is_int64=is64)
        off = gain = None
        want = np.stack([x[0], x[0], x[1], x[1]])
        if flt:
            off, gain = _restore(case.nch)
            kw.update(stream_offsets=off, stream_gains=gain)
            want = oracle.int_to_float(want, off, gain)
        for src in (comp, torch.from_numpy(comp).cuda()):
            for a, b in ((None, None), (n // 3, n // 3 + 1000), (n - 17, n)):
                # a window may miss the bad frames: the same call with on_error="raise" says whether it fails
                try:
                    plain = _host(fa.array_decompress(src, n, st, nb, first_stream_sample=a, last_stream_sample=b, **kw))
                except RuntimeError as e:
                    assert "Decoding failed" in str(e)
                    plain = None
                assert plain is None or a is not None, case.name
                arr, status = fa.array_decompress(src, n, st, nb, first_stream_sample=a, last_stream_sample=b,
                                                  on_error="fill", **kw)
                arr = _host(arr)
                assert status.dtype == np.int32 and status.shape == (4,), (case.name, status)
                assert status[0] == 0 and status[2] == 0 and status[3] == status[1], (case.name, status)
                assert (status[1] != 0) == (plain is None), (case.name, a, b, status)
                sl = slice(a, b)
                assert _same(arr[[0, 2]], want[[0, 2], sl]), (case.name, a, b)
                if plain is not None:
                    assert _same(arr, plain), (case.name, a, b)
                elif flt:
                    assert np.isnan(arr[[1, 3]]).all(), case.name
                else:
                    assert not arr[[1, 3]].any(), case.name
            # keep mask: rows in storage order, status in the same order
            keep = np.array([False, True, True, False])
            arr, idx, status = fa.array_decompress_slice(src, n, st, nb, keep=keep, on_error="fill", **kw)
            assert [tuple(i) for i in idx] == [(1,), (2,)]
            assert status.shape == (2,) and status[0] != 0 and status[1] == 0, (case.name, status)
            assert _same(_host(arr)[1], want[2]), case.name


def test_single_stream_status_shape(fa):
    case = FC.damage_cases()[0]
    comp, st, nb = case.buffer()
    arr, status = fa.array_decompress(comp, case.stream_size, int(st[0]), int(nb[0]), on_error="fill")
    assert arr.shape == (case.stream_size,) and status.shape == (1,) and status[0] == PROCESS
    assert fa.array_verify(comp, case.stream_size, int(st[0]), int(nb[0])).tolist() == [PROCESS]


# ---- verify against decode -----------------------------------------------------------------------------------------

def test_verify_matches_decode(fa):
    import torch

    from flacarray_b200 import libflacarray as lf

    groups = {}
    for case in FC.valid_cases() + BAD:
        comp, st, nb = case.buffer()
        try:
            lf.decode_flac(comp, st, nb, case.stream_size, is_int64=case.is_int64)
            raised = False
        except RuntimeError as e:
            assert "Decoding failed" in str(e)
            raised = True
        for src in (comp, torch.from_numpy(comp).cuda()):
            status = fa.array_verify(src, case.stream_size, st, nb, is_int64=case.is_int64)
            assert status.shape == st.shape and status.dtype == np.int32
            assert bool(status.any()) == raised, (case.name, status)
            assert raised == (not case.valid), case.name
        g = groups.setdefault((case.stream_size, case.nch), [])
        for s in range(len(case.streams)):
            g.append((case.streams[s], case.valid))
    # all cases of one (stream_size, nch) in one call
    for (n, nch), items in groups.items():
        comp, st, nb = _call([s for s, _ in items])
        status = fa.array_verify(comp, n, st, nb, is_int64=nch == 2)
        assert [v == 0 for v in status.tolist()] == [ok for _, ok in items], (n, nch, status)


# ---- the C entry points --------------------------------------------------------------------------------------------

def _c_isolated(fa, comp_d, st_d, nb_d, k, n, is64, out_ptr, status_ptr, first=-1, last=-1, off=None, gain=None):
    import torch

    from flacarray_b200 import _lib

    ctx = _lib.context(comp_d.device)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = _lib.lib().fab_decode_isolated(ctx.handle, C.c_void_p(comp_d.data_ptr()), C.c_void_p(st_d.data_ptr()),
                                        C.c_void_p(nb_d.data_ptr()), k, n, 1 if is64 else 0, first, last,
                                        C.c_void_p(out_ptr), None if off is None else C.c_void_p(off.data_ptr()),
                                        None if gain is None else C.c_void_p(gain.data_ptr()), 0, 0,
                                        C.c_void_p(status_ptr), stream)
    if rc == 0:
        rc = _lib.lib().fab_finish(ctx.handle, stream)
    return rc


def test_c_isolation_guards_status_and_recovery(fa):
    import torch

    case = FC.damage_cases()[0]
    comp, st, nb, x = _sandwich(case)
    n, k = case.stream_size, 4
    dev = torch.device("cuda")
    comp_d, st_d, nb_d = (torch.from_numpy(v).to(dev) for v in (comp, st, nb))
    guard = 4096
    buf = torch.full((guard + k * n + guard,), 0x3C3C3C3C, dtype=torch.int32, device=dev)
    sbuf = torch.full((64 + k + 64,), -7, dtype=torch.int32, device=dev)
    sbuf[64:64 + k] = -1
    rc = _c_isolated(fa, comp_d, st_d, nb_d, k, n, False, buf.data_ptr() + 4 * guard, sbuf.data_ptr() + 4 * 64)
    assert rc == 0
    hb, hs = _host(buf), _host(sbuf)
    assert (hb[:guard] == 0x3C3C3C3C).all() and (hb[guard + k * n:] == 0x3C3C3C3C).all()
    assert (hs[:64] == -7).all() and (hs[64 + k:] == -7).all()
    assert hs[64:64 + k].tolist() == [0, PROCESS, 0, PROCESS]
    rows = hb[guard:guard + k * n].reshape(k, n)
    assert _same(rows[0], x[0]) and _same(rows[2], x[1]) and not rows[[1, 3]].any()
    # a bad sample range is a call-level error
    rc = _c_isolated(fa, comp_d, st_d, nb_d, k, n, False, buf.data_ptr() + 4 * guard, sbuf.data_ptr() + 4 * 64, 5, n + 1)
    assert rc == 1 << 17
    # fab_verify needs its status array
    from flacarray_b200 import _lib

    ctx = _lib.context(dev)
    rc = _lib.lib().fab_verify(ctx.handle, C.c_void_p(comp_d.data_ptr()), C.c_void_p(st_d.data_ptr()),
                               C.c_void_p(nb_d.data_ptr()), k, n, 0, 0, 0, None,
                               C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 1 and "d_status" in ctx.last_error()
    # the next plain fab_decode on the same context succeeds
    (g0, g1), _ = _good(n, 1)
    gc, gst, gnb = _call([g0, g1])
    assert _same(fa.array_decompress(torch.from_numpy(gc).cuda(), n, gst, gnb), x)
    assert _same(fa.array_decompress(gc, n, gst, gnb), x)


def test_call_level_errors_raise_in_fill_mode(fa):
    import torch

    from flacarray_b200 import _lib

    case = FC.damage_cases()[1]
    comp, st, nb, x = _sandwich(case)
    n = case.stream_size
    with pytest.raises(RuntimeError, match="last_sample is beyond end of stream"):
        fa.array_decompress(comp, n, st, nb, first_stream_sample=0, last_stream_sample=n + 1, on_error="fill")
    with pytest.raises(ValueError, match="on_error"):
        fa.array_decompress(comp, n, st, nb, on_error="ignore")
    with pytest.raises(ValueError, match="on_error"):
        fa.array_decompress_slice(comp, n, st, nb, on_error=None)
    # on_error="raise" is today's behaviour, down to the message
    with pytest.raises(RuntimeError, match=r"^Decoding failed, return code = 16384$"):
        fa.array_decompress(comp, n, st, nb)
    # a caller workspace that is too small: ERROR_ALLOC, nothing launched
    ctx = _lib.context(torch.device("cuda"))
    need = _lib.lib().fab_decode_workspace_bytes(4, n, 4096)
    small = torch.empty(max(256, need // 2), dtype=torch.uint8, device="cuda")
    d = torch.from_numpy(comp).cuda()
    try:
        ctx.set_workspace(small)
        n0 = ctx.launches()
        with pytest.raises(RuntimeError, match=r"Decoding failed, return code = 1\b"):
            fa.array_decompress(d, n, st, nb, on_error="fill")
        with pytest.raises(RuntimeError, match=r"Verifying failed, return code = 1\b"):
            fa.array_verify(d, n, st, nb)
        assert ctx.launches() == n0
    finally:
        ctx.set_workspace(None)
    arr, status = fa.array_decompress(d, n, st, nb, on_error="fill")
    assert status.tolist() == [0, PROCESS, 0, PROCESS]


def test_launch_counts(fa):
    import torch

    from flacarray_b200 import _lib

    case = FC.damage_cases()[2]
    comp, st, nb, x = _sandwich(case)
    n = case.stream_size
    d = torch.from_numpy(comp).cuda()
    ctx = _lib.context(d.device)
    off, gain = _restore(1)

    def launches(fn):
        fn()  # warm (first calls may size the scratch block)
        n0 = ctx.launches()
        fn()
        return ctx.launches() - n0

    plain_i = launches(lambda: fa.array_decompress(d, n, st[[0, 2]], nb[[0, 2]]))
    iso_i = launches(lambda: fa.array_decompress(d, n, st, nb, on_error="fill"))
    plain_f = launches(lambda: fa.array_decompress(d, n, st[[0, 2]], nb[[0, 2]], stream_offsets=off[:2], stream_gains=gain[:2]))
    iso_f = launches(lambda: fa.array_decompress(d, n, st, nb, stream_offsets=off, stream_gains=gain, on_error="fill"))
    ver = launches(lambda: fa.array_verify(d, n, st, nb))
    assert iso_i == plain_i + 1 and iso_f == plain_f + 1, (plain_i, iso_i, plain_f, iso_f)
    assert ver == plain_i and plain_f == plain_i + 1, (ver, plain_i, plain_f)


# ---- an array written by this library ------------------------------------------------------------------------------

@pytest.mark.parametrize("dt", DTYPES, ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("where", ["device", "host"])
def test_flacarray_stream_17_corrupted(fa, dt, where):
    import torch

    rng = np.random.default_rng(1700 + np.dtype(dt).itemsize)
    shape = (4, 10, 5000)
    walk = np.cumsum(rng.integers(-300, 301, shape), axis=-1)
    if np.dtype(dt).kind == "f":
        data = (walk * 1e-3 + rng.normal(0, 1e-3, shape)).astype(dt)
        far = fa.FlacArray.from_array(torch.from_numpy(data).cuda() if where == "device" else data, quanta=1e-4)
    else:
        data = (walk * (1 << 20 if dt == np.int64 else 1)).astype(dt)
        far = fa.FlacArray.from_array(torch.from_numpy(data).cuda() if where == "device" else data)
    clean = _host(far.to_array())
    assert far.verify().tolist() == np.zeros((4, 10), np.int32).tolist()
    st = np.asarray(_host(far.stream_starts)).reshape(-1)
    nb = np.asarray(_host(far.stream_nbytes)).reshape(-1)
    pos = int(st[17] + nb[17] * 2 // 3)                 # inside the frames (the metadata is a small head)
    far._compressed[pos] ^= 0x5A                         # (a CUDA tensor or a numpy array)
    status = far.verify()
    want = np.zeros((4, 10), np.int32)
    want[1, 7] = PROCESS
    assert status.shape == (4, 10) and np.array_equal(status, want), status
    arr, st2 = far.to_array(on_error="fill")
    arr = _host(arr)
    assert np.array_equal(st2, want)
    mask = np.ones((4, 10), bool)
    mask[1, 7] = False
    assert _same(arr[mask], clean[mask])
    assert np.isnan(arr[1, 7]).all() if np.dtype(dt).kind == "f" else not arr[1, 7].any()
    keep = np.zeros((4, 10), bool)
    keep[1, 5:9] = True
    arr, idx, st3 = far.to_array(keep=keep, stream_slice=slice(1000, 3000), keep_indices=True, on_error="fill")
    assert [tuple(i) for i in idx] == [(1, 5), (1, 6), (1, 7), (1, 8)]
    assert st3.tolist() == [0, 0, PROCESS, 0]
    arr = _host(arr)
    assert _same(arr[[0, 1, 3]], clean[1, [5, 6, 8], 1000:3000])
    with pytest.raises(RuntimeError, match="Decoding failed"):
        far.to_array()


# ---- more than 65 535 streams --------------------------------------------------------------------------------------

N_MANY = 65535 + 5


def test_more_than_65535_streams_with_bad_streams_in_both_slabs(fa):
    import torch

    rng = np.random.default_rng(6553)
    n = 300
    x = np.cumsum(rng.integers(-500, 501, (N_MANY, n)), axis=1).astype(np.int32)
    comp, st, nb = (_host(v) for v in fa.array_compress(x, level=5)[:3])
    bad = [3, 65534, 65536, N_MANY - 1]
    comp = comp.copy()
    for s in bad:
        comp[int(st[s] + nb[s] - 5)] ^= 0x21              # inside the last frame
    want = np.zeros(N_MANY, np.int32)
    want[bad] = PROCESS
    good = np.ones(N_MANY, bool)
    good[bad] = False
    off, gain = _restore(1, N_MANY)
    for src in (comp, torch.from_numpy(comp).cuda()):
        assert np.array_equal(fa.array_verify(src, n, st, nb), want)
        arr, status = fa.array_decompress(src, n, st, nb, on_error="fill")
        arr = _host(arr)
        assert np.array_equal(status, want)
        assert _same(arr[good], x[good]) and not arr[bad].any()
        arr, status = fa.array_decompress(src, n, st, nb, stream_offsets=off, stream_gains=gain, first_stream_sample=10,
                                          last_stream_sample=290, on_error="fill")
        arr = _host(arr)
        assert np.array_equal(status, want)
        assert np.isnan(arr[bad]).all() and not np.isnan(arr[good]).any()
