"""Host-resident compressed bytes go to the device in groups of streams through one staging path (libflacarray._staged
with _bytes_prep).  With several groups forced, every host-resident call returns what the device-resident call returns:
verify statuses, on_error="fill" decodes with keep masks, and windows over back-to-back and scattered streams.  A sparse
keep mask stages only about the kept streams' bytes, and a group's device buffers are released when the caller drops
them."""
import time
import weakref

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

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


def _encoded(fa, dt, shape, seed):
    rng = np.random.default_rng(seed)
    walk = np.cumsum(rng.integers(-300, 301, shape), axis=-1)
    if np.dtype(dt).kind == "f":
        comp, st, nb, off, gain = fa.array_compress((walk * 1e-3).astype(dt), quanta=1e-4, level=5)
    else:
        comp, st, nb, off, gain = fa.array_compress(walk.astype(dt), level=5)
    return comp, st, nb, off, gain


def _damage(comp, st, nb, which):
    comp = comp.copy()
    fst, fnb = st.reshape(-1), nb.reshape(-1)
    for k in which:
        comp[int(fst[k] + fnb[k] * 2 // 3)] ^= 0x5A        # inside the frames: the walker rejects the stream
    return comp


def _groups_of(monkeypatch, lf, nbytes_per_group):
    monkeypatch.setattr(lf, "_PIPE_MIN_BYTES", 1)
    monkeypatch.setattr(lf, "_PIPE_CHUNK_BYTES", int(nbytes_per_group))


def test_verify_host_groups_match_device(fa, monkeypatch):
    import torch

    from flacarray_b200 import libflacarray as lf

    comp, st, nb, _, _ = _encoded(fa, np.int32, (4, 6, 5000), 301)
    bad = [2, 11, 13, 22]
    comp = _damage(comp, st, nb, bad)
    want = np.zeros(24, np.int32)
    want[bad] = PROCESS
    dev = fa.array_verify(torch.from_numpy(comp).cuda(), 5000, st, nb)
    assert np.array_equal(dev.reshape(-1), want), dev
    _groups_of(monkeypatch, lf, 3 * nb.mean())
    assert len(lf._chunk_ranges(24, int(nb.sum()) // 24)) >= 5
    host = fa.array_verify(comp, 5000, st, nb)
    assert host.shape == st.shape and host.dtype == np.int32 and np.array_equal(host, dev)


@pytest.mark.parametrize("dt", [np.int32, np.float32])
def test_fill_with_keep_host_groups_match_device(fa, monkeypatch, dt):
    import torch

    from flacarray_b200 import libflacarray as lf

    n = 5000
    comp, st, nb, off, gain = _encoded(fa, dt, (4, 6, n), 302)
    comp = _damage(comp, st, nb, [1, 10, 15, 20])
    dcomp = torch.from_numpy(comp).cuda()
    idx = np.arange(24).reshape(4, 6)
    for keep in (idx % 3 != 1, idx % 5 == 0):          # dense (covering ranges) and sparse (gathered) selections
        kw = dict(stream_offsets=off, stream_gains=gain, keep=keep, first_stream_sample=700, last_stream_sample=4300,
                  on_error="fill")
        d_arr, d_idx, d_status = fa.array_decompress_slice(dcomp, n, st, nb, **kw)
        assert d_status.any() and not d_status.all()
        _groups_of(monkeypatch, lf, 3 * 3600 * 4)
        assert len(lf._chunk_ranges(int(keep.sum()), 3600 * 4)) >= 2
        h_arr, h_idx, h_status = fa.array_decompress_slice(comp, n, st, nb, **kw)
        monkeypatch.undo()
        assert h_idx == d_idx
        assert h_status.dtype == np.int32 and np.array_equal(h_status, d_status)
        assert _same(h_arr, _host(d_arr))


def test_windows_host_groups_match_device(fa, monkeypatch):
    import torch

    from flacarray_b200 import libflacarray as lf

    n = 6000
    comp, st, nb, _, _ = _encoded(fa, np.int32, (30, n), 303)
    dcomp = torch.from_numpy(comp).cuda()
    rng = np.random.default_rng(304)
    # every stream (back to back), every 2nd (gaps below the streams' bytes), every 5th (gathered)
    for step in (1, 2, 5):
        refs = np.arange(0, 30, step)
        streams = rng.permutation(np.repeat(refs, 3))
        first = rng.integers(0, n - 500, streams.size)
        last = first + rng.integers(0, 500, streams.size)
        d_data, d_off = fa.array_decompress_windows(dcomp, n, st, nb, streams, first, last)
        _groups_of(monkeypatch, lf, 1.5 * nb.mean())
        assert len(lf._chunk_ranges(refs.size, int(nb[refs].sum()) // refs.size)) >= 3
        h_data, h_off = fa.array_decompress_windows(comp, n, st, nb, streams, first, last)
        monkeypatch.undo()
        assert np.array_equal(h_off, d_off)
        assert _same(h_data, _host(d_data))


def test_sparse_keep_stages_only_the_kept_streams(fa, monkeypatch):
    from flacarray_b200 import libflacarray as lf

    n = 4000
    comp, st, nb, _, _ = _encoded(fa, np.int32, (128, n), 305)
    full = fa.array_decompress(comp, n, st, nb)
    keep = np.zeros(128, bool)
    keep[[0, -1]] = True
    staged = []
    copy = lf._Feeder.copy

    def counted(self, dst, src):
        staged.append(src.numel() * src.element_size())
        return copy(self, dst, src)

    monkeypatch.setattr(lf._Feeder, "copy", counted)
    arr, idx = fa.array_decompress_slice(comp, n, st, nb, keep=keep)
    assert idx == [(0,), (127,)]
    assert np.array_equal(arr, full[[0, -1]])
    assert 0 < sum(staged) <= 2 * int(nb[0] + nb[-1]), (sum(staged), int(nb.sum()))


def test_staged_releases_a_group_when_the_caller_drops_it(fa):
    import torch

    from flacarray_b200 import libflacarray as lf

    dev = torch.device("cuda", torch.cuda.current_device())
    src = torch.arange(40 * 1000, dtype=torch.int32).view(40, 1000)
    ranges = [(0, 5), (5, 12), (12, 20), (20, 33), (33, 40)]
    for a, b, dc in lf._staged(dev, ranges, lf._rows_prep(src, dev)):
        assert torch.equal(dc.cpu(), src[a:b])
        time.sleep(0.02)      # the helper thread's executor drops its own reference to a finished group right after it
        ref = weakref.ref(dc)
        del dc
        assert ref() is None
