"""Decoder conformance on the GPU: every stream of tests/flac_corpus.py (written syntax element by syntax element, see
oracle/flac_writer.py) through every decode entry point of the CUDA library, against the integers the writer was
given, bit for bit; float32 / float64 restore against the oracle's int_to_float; every invalid or damaged stream must
fail without spoiling the next decode.  Plus one call with more than 65 535 streams: every per-stream grid is cut into
grid.y slabs of 65 535, and only streams past the first slab show a slab-offset mistake."""
import ctypes as C
import os
import sys
import zlib

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

import flac_corpus as FC  # noqa: E402

pytestmark = pytest.mark.gpu

VALID = FC.valid_cases()
BAD = FC.invalid_cases() + FC.damage_cases()


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


def _restore_params(case):
    rng = np.random.default_rng(zlib.crc32(case.name.encode()))
    k = len(case.streams)
    fdt = np.float64 if case.is_int64 else np.float32
    off = rng.normal(0, 100, k).astype(fdt)
    gain = (10.0 ** rng.uniform(-1, 6, k)).astype(fdt)
    return off, gain


def _windows(case):
    ws = np.array([w[0] for w in case.windows], np.int64)
    return ws, np.array([w[1] for w in case.windows], np.int64), np.array([w[2] for w in case.windows], np.int64)


def _c_decode(fa, case, comp, st, nb, first, last):
    from flacarray_b200 import _lib

    L = _lib.lib()
    fn = L.decode_i64 if case.is_int64 else L.decode_i32
    fn.restype = C.c_int
    k = st.size
    n = case.stream_size if first < 0 else last - first
    out = np.zeros((k, n), np.int64 if case.is_int64 else np.int32)
    rc = fn(C.c_void_p(comp.ctypes.data), C.c_void_p(st.ctypes.data), C.c_void_p(nb.ctypes.data), C.c_int64(k),
            C.c_int64(case.stream_size), C.c_int64(first), C.c_int64(last), C.c_void_p(out.ctypes.data), C.c_bool(True))
    return rc, out


@pytest.mark.parametrize("case", VALID, ids=[c.name for c in VALID])
def test_valid_case_every_entry_point(fa, case, oracle, monkeypatch):
    import torch

    from flacarray_b200 import libflacarray as lf

    comp, st, nb = case.buffer()
    k, n = len(case.streams), case.stream_size
    dcomp = torch.from_numpy(comp).cuda()
    kw = dict(is_int64=case.is_int64, no_flatten=True)
    ws, wf, wl = _windows(case)
    if case.full:
        for src in (comp, dcomp):
            assert _same(fa.array_decompress(src, n, st, nb, **kw), case.expect), case.name
        rc, out = _c_decode(fa, case, comp, st, nb, -1, -1)
        assert rc == 0 and _same(out, case.expect), case.name
        if k > 1:
            # the chunked host pipeline, one stream per chunk
            monkeypatch.setattr(lf, "_PIPE_MIN_BYTES", 1)
            monkeypatch.setattr(lf, "_PIPE_CHUNK_BYTES", 1)
            assert _same(fa.array_decompress(comp, n, st, nb, **kw), case.expect), case.name
            monkeypatch.undo()
    for i, (s, a, b) in enumerate(case.windows):
        want = case.window_expect(i)
        for src in (comp, dcomp):
            got = fa.array_decompress(src, n, st, nb, first_stream_sample=int(a), last_stream_sample=int(b), **kw)
            assert _same(_host(got)[s], want), (case.name, (s, a, b))
        rc, out = _c_decode(fa, case, comp, st, nb, int(a), int(b))
        assert rc == 0 and _same(out[s], want), (case.name, (s, a, b))
    for src in (comp, dcomp):
        data, offs = fa.array_decompress_windows(src, n, st, nb, ws, wf, wl, is_int64=case.is_int64)
        data = _host(data)
        for i in range(ws.size):
            assert _same(data[offs[i]:offs[i + 1]], case.window_expect(i)), (case.name, case.windows[i])

    # int -> float restore: the fused tile restore, k_restore_fixup (general-decoder frames, walked streams), k_restore_win
    off, gain = _restore_params(case)
    if case.full:
        want = oracle.int_to_float(case.expect, off, gain)
        for src in (comp, dcomp):
            got = fa.array_decompress(src, n, st, nb, stream_offsets=off, stream_gains=gain, **kw)
            assert _same(got, want), case.name
    for src in (comp, dcomp):
        data, offs = fa.array_decompress_windows(src, n, st, nb, ws, wf, wl, stream_offsets=off, stream_gains=gain,
                                                 is_int64=case.is_int64)
        data = _host(data)
        for i, s in enumerate(ws.tolist()):
            want = oracle.int_to_float(np.ascontiguousarray(case.window_expect(i)).reshape(1, -1), off[s:s + 1],
                                       gain[s:s + 1]).reshape(-1)
            assert _same(data[offs[i]:offs[i + 1]], want), (case.name, case.windows[i])


@pytest.mark.parametrize("name", ["stereo_assignments", "escaped_partitions", "stereo_side_channel_extremes",
                                  "variable_blocksizes", "start_offsets_mod_16", "mixed_first_blocksize_larger"])
def test_c_entry_host_pipeline(fa, name):
    """decode_i32 / decode_i64 on host buffers above the size where the library stages them through its chunked
    pipeline (64 MB out, 128 MB chunks): a case's buffer repeated until the output spans three chunks."""
    case = FC.by_name(name)
    comp, st, nb = case.buffer()
    k = st.size
    row = case.stream_size * (8 if case.is_int64 else 4)
    reps = -(-(2 * (128 << 20)) // (row * k)) + 1
    big = np.tile(comp, reps)
    bst = (st[None, :] + comp.size * np.arange(reps, dtype=np.int64)[:, None]).reshape(-1)
    rc, out = _c_decode(fa, case, big, bst, np.tile(nb, reps), -1, -1)
    assert rc == 0
    assert np.array_equal(out.reshape(reps, k, -1), np.broadcast_to(case.expect, (reps,) + case.expect.shape)), name


def test_bad_cases_raise_and_the_context_recovers(fa):
    import torch

    good = FC.valid_cases()[0]
    gcomp, gst, gnb = good.buffer()
    for case in BAD:
        comp, st, nb = case.buffer()
        kw = dict(is_int64=case.is_int64)
        for src in (comp, torch.from_numpy(comp).cuda()):
            with pytest.raises(RuntimeError, match="Decoding failed"):
                fa.array_decompress(src, case.stream_size, st, nb, **kw)
            with pytest.raises(RuntimeError, match="Decoding failed"):
                fa.array_decompress_windows(src, case.stream_size, st, nb, [0], [0], [case.stream_size], **kw)
        rc, _ = _c_decode(fa, case, comp, st, nb, -1, -1)
        assert rc != 0, case.name
        assert _same(fa.array_decompress(gcomp, good.stream_size, gst, gnb, no_flatten=True), good.expect), case.name


N_MANY = 65535 + 5


def _many_pick():
    return np.array([0, 1, 65534, 65535, 65536, N_MANY - 1])


@pytest.mark.parametrize("path", ["general", "walker"])
@pytest.mark.parametrize("nch", [1, 2])
def test_more_than_65535_streams_restore_off_the_tile_path(fa, oracle, path, nch):
    """One written stream (an LPC order-20 frame, or variable blocking) repeated 65 540 times, restored with a different
    offset and gain per stream: the samples the tile decoder does not restore itself (k_restore_fixup, per slab of
    65 535 streams; k_restore for float64; k_restore_win) must use the gains of their own stream."""
    import torch

    from oracle import flac_writer as W

    rng = np.random.default_rng(4300 + nch * 10 + (path == "walker"))
    n = 300
    L = FC.walk(rng, n, 400)
    if nch == 1:
        fr = W.Frame(L, [FC.sub_lpc(L, [16] + [1, -1] * 9 + [0], 9, 4, porder=2)], variable=path == "walker")
        want1 = L.astype(np.int32)
    else:
        lr = np.stack([L, L + rng.integers(-9, 10, n)], 1)
        subs = [FC.sub_fixed(lr[:, 0], 2), FC.sub_lpc(lr[:, 1], [16] + [1, -1] * 9 + [0], 9, 4)] if path == "walker" else \
            [FC.sub_fixed(lr[:, 0], 2), FC.sub_fixed(lr[:, 0] - lr[:, 1], 1)]
        fr = W.Frame(lr, subs, ca=1 if path == "walker" else 8, variable=path == "walker")
        want1 = FC.as_i64(lr)
    one = W.write_stream([fr], nch)[0]
    comp = np.frombuffer(one * N_MANY, np.uint8).copy()
    st = np.arange(N_MANY, dtype=np.int64) * len(one)
    nb = np.full(N_MANY, len(one), np.int64)
    is64 = nch == 2
    fdt = np.float64 if is64 else np.float32
    off = rng.normal(0, 10, N_MANY).astype(fdt)
    gain = (10.0 ** rng.uniform(0, 5, N_MANY)).astype(fdt)
    want = oracle.int_to_float(np.tile(want1, (N_MANY, 1)), off, gain)
    for src in (comp, torch.from_numpy(comp).cuda()):
        got = fa.array_decompress(src, n, st, nb, stream_offsets=off, stream_gains=gain, is_int64=is64)
        assert _same(got, want)
        got = fa.array_decompress(src, n, st, nb, stream_offsets=off, stream_gains=gain, first_stream_sample=50,
                                  last_stream_sample=299, is_int64=is64)
        assert _same(got, want[:, 50:299])
    pick = _many_pick()
    data, offs = fa.array_decompress_windows(comp, n, st, nb, pick, 11, 222, stream_offsets=off, stream_gains=gain,
                                             is_int64=is64)
    assert _same(_host(data), want[pick, 11:222].reshape(-1))


@pytest.mark.parametrize("dt", [np.int32, np.int64, np.float32, np.float64])
def test_more_than_65535_streams(fa, oracle, dt):
    """65 540 streams of 300 samples: encode, full and windowed decode (with restore for floats), checked on both sides
    of every slab edge; for integers also the sync scan of foreign streams (oracle-encoded, no frame-size table)."""
    import torch

    from flacarray_b200 import libflacarray as lf

    rng = np.random.default_rng(4242 + np.dtype(dt).itemsize + (1 if np.dtype(dt).kind == "f" else 0))
    n = 300
    walk = np.cumsum(rng.integers(-500, 501, (N_MANY, n)), axis=1)
    pick = _many_pick()
    if np.dtype(dt).kind == "i":
        x = (walk + (2 ** 40 if dt == np.int64 else 0) * rng.integers(-3, 4, (N_MANY, 1))).astype(dt)
        is64 = dt == np.int64
        for src in (x, torch.from_numpy(x).cuda()):
            comp, st, nb = fa.array_compress(src, level=5)[:3]
            comp, st, nb = _host(comp), _host(st), _host(nb)
            y = _host(fa.array_decompress(comp, n, st, nb, is_int64=is64))
            assert _same(y, x)
            y = _host(fa.array_decompress(torch.from_numpy(comp).cuda(), n, st, nb, first_stream_sample=97,
                                          last_stream_sample=211, is_int64=is64))
            assert _same(y, x[:, 97:211])
            data, offs = fa.array_decompress_windows(comp, n, st, nb, pick, pick % 50, 250 + pick % 50, is_int64=is64)
            for i, s in enumerate(pick.tolist()):
                assert _same(_host(data)[offs[i]:offs[i + 1]], x[s, s % 50:250 + s % 50]), s
        # foreign streams: k_dec_sync in both slabs
        oc, ost, onb = oracle.encode(x, 5)
        y = _host(fa.array_decompress(oc, n, ost, onb, is_int64=is64))
        assert _same(y, x)
        for s in pick.tolist():
            assert _same(oracle.decode(oc, ost[s:s + 1], onb[s:s + 1], n, is_int64=is64)[0], x[s])
        return
    x = (walk * 1e-3 + rng.normal(0, 1e-4, (N_MANY, n)) + np.linspace(-5, 5, N_MANY)[:, None]).astype(dt)
    is64 = dt == np.float64
    std = lf.stream_std(x)
    np.testing.assert_allclose(std[pick], np.std(x[pick].astype(np.float64), axis=-1), rtol=1e-5)
    q = np.full(N_MANY, 1e-4, dt)
    ints, off, gain = fa.float_to_int(x, quanta=q)
    oi, oo, og = oracle.float_to_int(x[pick], q[pick])
    assert _same(_host(ints)[pick], oi) and _same(_host(off)[pick], oo) and _same(_host(gain)[pick], og)
    for src in (x, torch.from_numpy(x).cuda()):
        comp, st, nb, off, gain = fa.array_compress(src, level=5, quanta=q)
        comp, st, nb, off, gain = (_host(v) for v in (comp, st, nb, off, gain))
        assert _same(off[pick], oo) and _same(gain[pick], og)
        full = _host(fa.array_decompress(comp, n, st, nb, stream_offsets=off, stream_gains=gain, is_int64=is64))
        iv = oracle.decode(comp, st[pick], nb[pick], n, is_int64=is64)
        assert _same(iv, oi)
        assert _same(full[pick], oracle.int_to_float(iv, off[pick], gain[pick]))
        win = _host(fa.array_decompress(torch.from_numpy(comp).cuda(), n, st, nb, stream_offsets=off, stream_gains=gain,
                                        first_stream_sample=13, last_stream_sample=290, is_int64=is64))
        assert _same(win, full[:, 13:290])
        data, offs = fa.array_decompress_windows(comp, n, st, nb, pick, 7, 293, stream_offsets=off, stream_gains=gain,
                                                 is_int64=is64)
        assert _same(_host(data), full[pick, 7:293].reshape(-1))
