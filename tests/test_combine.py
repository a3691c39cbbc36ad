"""Weighted sums across streams on the CPU: the host emulation of fab_combine_rows (tests/hostsim/hostsim_combine.cpp)
against the numpy fold acc = acc + w_k * float64(x_k), bit for bit.

* int32 and int64 rows of random data and of INT32 / INT64 extremes, int64 values above 2^53 (round to nearest even),
  float32 and float64 rows restored with the library's offsets and gains, weights 1, 1/3 and random in [-1, 1];
* segments of one row and of many rows (several row tiles), an output row continued from a previous call, rows with
  n % 4 != 0 that start off a 16-byte boundary, n = 1, failed rows skipped, bad segment records flagged and skipped;
* the argument checks of array_combine / FlacArray.combine raise ValueError without a device.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, "hostsim"))

BAD_SEGMENT = 1 << 17


@pytest.fixture(scope="module")
def HC():
    import hostsim_combine

    hostsim_combine.lib()
    return hostsim_combine


def _same(got, want):
    got, want = np.ascontiguousarray(got), np.ascontiguousarray(want)
    return got.dtype == want.dtype and got.shape == want.shape and np.array_equal(got.view(np.uint8), want.view(np.uint8))


def _rows(dtype, n_rows, n, seed):
    rng = np.random.default_rng(seed)
    info = np.iinfo(dtype)
    x = rng.integers(info.min, info.max, (n_rows, n), dtype=dtype, endpoint=True)
    x[::3] = np.cumsum(rng.integers(-1000, 1001, (x[::3].shape)), axis=1).astype(dtype)     # typical time streams
    return x


def _unaligned(x):
    """The same rows starting one element past a 16-byte boundary."""
    flat = np.empty(x.size + 1, x.dtype)
    y = flat[1:].reshape(x.shape)
    y[...] = x
    return y


def _segments(groups):
    """Segments of rows already sorted by group (no -1): row bounds and output rows."""
    cut = np.flatnonzero(groups[1:] != groups[:-1]) + 1
    bounds = np.concatenate([[0], cut, [groups.size]]).astype(np.int64)
    return bounds, groups[bounds[:-1]].astype(np.int64)


def _run(HC, x, w, groups, n_groups, **kw):
    """Emulated combine of rows sorted by group into a zero-filled [n_groups, n]."""
    seg, seg_out = _segments(groups)
    out = np.zeros((n_groups, x.shape[1]))
    assert HC.combine_rows(x, w, seg, seg_out, out, **kw) == 0
    return out


def _weights(kind, n_rows, seed):
    rng = np.random.default_rng(seed)
    if kind == "one":
        return np.ones(n_rows)
    if kind == "third":
        return np.full(n_rows, 1.0 / 3.0)
    return rng.uniform(-1.0, 1.0, n_rows)


N = 203           # not a multiple of 4 and more than one 64-column chunk of the emulated blocks


@pytest.mark.parametrize("dtype", [np.int32, np.int64])
@pytest.mark.parametrize("wkind", ["one", "third", "random"])
@pytest.mark.parametrize("layout", ["one_group", "groups", "singles"])
def test_integer_rows(HC, dtype, wkind, layout):
    n_rows = 75                          # more than two 32-row tiles in one segment
    x = _rows(dtype, n_rows, N, 3 + (dtype == np.int64))
    w = _weights(wkind, n_rows, 9)
    groups = {"one_group": np.zeros(n_rows, np.int64), "groups": np.repeat(np.arange(5), [1, 40, 2, 30, 2]),
              "singles": np.arange(n_rows)}[layout]
    n_groups = int(groups.max()) + 1
    want = HC.fold(x, w, groups, n_groups)
    assert _same(_run(HC, x, w, groups, n_groups), want)
    assert _same(_run(HC, _unaligned(x), w, groups, n_groups), want)


@pytest.mark.parametrize("dtype", [np.int32, np.int64])
def test_extremes_and_rounding(HC, dtype):
    info = np.iinfo(dtype)
    x = np.empty((6, N), dtype)
    x[0] = info.min
    x[1] = info.max
    x[2, 0::2], x[2, 1::2] = info.min, info.max
    x[3] = info.max - np.arange(N, dtype=dtype)
    x[4] = info.min + np.arange(N, dtype=dtype)
    x[5] = -np.arange(N, dtype=dtype)
    if dtype == np.int64:
        # above 2^53 float64(x) rounds to nearest even: ties and non-ties both ways
        base = (1 << 53) + np.arange(N, dtype=np.int64)
        x[3] = base
        x[4] = -(base * 3 + 1)
        assert not np.array_equal(x[3].astype(np.float64).astype(np.int64), x[3])
    for w in (np.ones(6), np.array([1.0, 1.0, -1.0, 1.0 / 3.0, 0.5, -2.0])):
        for groups in (np.zeros(6, np.int64), np.array([0, 0, 1, 1, 2, 2])):
            n_groups = int(groups.max()) + 1
            assert _same(_run(HC, x, w, groups, n_groups), HC.fold(x, w, groups, n_groups))


@pytest.mark.parametrize("is_int64", [False, True])
def test_float_restore(HC, oracle, is_int64):
    """Rows restored with offsets and gains from the library's quantisation: the fold of the restored values in the
    array's type, widened, not a restore in double."""
    fdt = np.float64 if is_int64 else np.float32
    rng = np.random.default_rng(21)
    n_rows = 40
    scale = rng.choice([1.0, 1e3, 1e-6], (n_rows, 1))
    f = (rng.normal(0, 1, (n_rows, N)) * scale + rng.normal(0, 5, (n_rows, 1))).astype(fdt)
    for q in (np.full(n_rows, 1e-4, fdt), None):
        ints, off, gain = oracle.float_to_int(f, q)
        back = oracle.int_to_float(ints, off, gain)
        assert back.dtype == fdt
        for wkind in ("one", "third", "random"):
            w = _weights(wkind, n_rows, 5)
            for groups in (np.zeros(n_rows, np.int64), np.repeat(np.arange(4), 10)):
                n_groups = int(groups.max()) + 1
                got = _run(HC, ints, w, groups, n_groups, offsets=off, gains=gain)
                assert _same(got, HC.fold(back, w, groups, n_groups))
                assert _same(_run(HC, _unaligned(ints), w, groups, n_groups, offsets=off, gains=gain), got)


def test_continues_from_stored_value(HC):
    """A group split over two calls: the second call starts from what the first stored, and the bits equal one call."""
    x = _rows(np.int32, 50, N, 31)
    w = _weights("random", 50, 32)
    want = HC.fold(x, w, np.zeros(50, np.int64), 1)
    out = np.zeros((3, N))
    assert HC.combine_rows(x[:17], w[:17], [0, 17], [1], out) == 0
    assert HC.combine_rows(x[17:], w[17:], [0, 33], [1], out) == 0
    assert _same(out[1], want[0]) and not out[0].any() and not out[2].any()
    # starting from zero again would be a different number
    fresh = np.zeros((1, N))
    HC.combine_rows(x[17:], w[17:], [0, 33], [0], fresh)
    assert not _same(fresh[0], want[0])


def test_one_sample_rows(HC):
    x = np.array([[5], [-3], [np.iinfo(np.int32).max], [7]], np.int32)
    w = np.array([0.25, 1.0 / 3.0, -1.0, 2.0])
    groups = np.array([0, 0, 1, 2])
    assert _same(_run(HC, x, w, groups, 3), HC.fold(x, w, groups, 3))
    x64 = np.array([[(1 << 62) + 1], [-(1 << 60) - 3]], np.int64)
    assert _same(_run(HC, x64, np.ones(2), np.zeros(2, np.int64), 1), HC.fold(x64, np.ones(2), np.zeros(2, np.int64), 1))


@pytest.mark.parametrize("restored", [False, True])
def test_failed_rows_skipped(HC, oracle, restored):
    n_rows = 45
    x = _rows(np.int32, n_rows, N, 41)
    w = _weights("random", n_rows, 42)
    status = np.zeros(n_rows, np.int32)
    status[[0, 7, 33, 44]] = [1 << 14, 1 << 13, 1 << 14, 1 << 14]
    groups = np.repeat([0, 1], [33, 12])
    kw = {}
    vals = x
    if restored:
        f = (np.random.default_rng(43).normal(0, 1, (n_rows, N))).astype(np.float32)
        x, off, gain = oracle.float_to_int(f, np.full(n_rows, 1e-4, np.float32))
        vals = oracle.int_to_float(x, off, gain).copy()
        vals[status != 0] = np.nan                 # what the isolated decode leaves in a failed float row
        kw = dict(offsets=off, gains=gain)
    got = _run(HC, x, w, groups, 2, status=status, **kw)
    assert _same(got, HC.fold(vals, w, groups, 2, ok=status == 0))
    assert np.isfinite(got).all()


def test_bad_segment_records(HC):
    """A record that breaks a rule sets the error bit and writes nothing; the other segments are computed."""
    x = _rows(np.int64, 12, N, 51)
    w = _weights("random", 12, 52)
    good = HC.fold(x, w, np.repeat(np.arange(4), 3), 4)
    # (row bounds, output rows, the records the rules refuse): a record is refused when its rows leave [0, 12], its
    # output row leaves [0, 4) or is not above the previous record's
    cases = [
        ([0, 3, 6, 9, 12], [0, 1, 9, 3], [2, 3]),        # output row out of range (and the next is not above it)
        ([0, 3, 6, 9, 12], [0, 1, -1, 3], [2]),          # negative output row
        ([0, 3, 6, 9, 12], [0, 2, 1, 3], [2]),           # output rows not increasing: the later record is refused
        ([0, 3, 7, 6, 12], [0, 1, 2, 3], [2]),           # row bounds decreasing
        ([0, 3, 6, 9, 13], [0, 1, 2, 3], [3]),           # past the last row
        ([-1, 3, 6, 9, 12], [0, 1, 2, 3], [0]),          # before the first row
    ]
    for seg, seg_out, bad in cases:
        out = np.zeros((4, N))
        assert HC.combine_rows(x, w, seg, seg_out, out) == BAD_SEGMENT, (seg, seg_out)
        written = set()
        for s in range(4):
            if s in bad:
                continue
            lo, hi, o = seg[s], seg[s + 1], seg_out[s]
            written.add(o)
            want = HC.fold(x[lo:hi], w[lo:hi], np.zeros(hi - lo, np.int64), 1)[0]
            assert _same(out[o], want), (seg, seg_out, s)
        for o in set(range(4)) - written:
            assert not out[o].any() and not np.signbit(out[o]).any(), (seg, seg_out, o)
    out = np.zeros((4, N))
    assert HC.combine_rows(x, w, [0, 3, 6, 9, 12], [0, 1, 2, 3], out) == 0
    assert _same(out, good)


# ---- argument checks of array_combine / FlacArray.combine: no device needed ----------------------------------------

def _starts():
    return np.array([0, 10, 20], np.int64), np.array([10, 10, 10], np.int64)


def _combine(**kw):
    import flacarray_b200 as fa

    st, nb = _starts()
    return fa.array_combine(np.zeros(30, np.uint8), 100, st, nb, **kw)


@pytest.mark.parametrize("kw,match", [
    (dict(weights=np.ones(2)), "weights"),
    (dict(weights=np.ones(4)), "weights"),
    (dict(weights=np.ones(3, bool)), "weights"),
    (dict(groups=np.zeros(2, np.int64)), "groups"),
    (dict(groups=np.zeros((2, 2), np.int64)), "groups"),
    (dict(groups=np.zeros(3)), "integers"),
    (dict(groups=np.zeros(3, bool)), "integers"),
    (dict(groups=[0.0, 1.0, 2.0]), "integers"),
    (dict(groups=np.array([0, -2, 1])), "groups"),
    (dict(groups=np.array([0, 1, 3]), n_groups=3), "groups"),
    (dict(groups=np.array([0, 1, 2]), n_groups=2), "groups"),
    (dict(groups=np.array([-1, -1, -1]), n_groups=-1), "n_groups"),
    (dict(groups=np.array([0, 0, 0]), n_groups=1.0), "n_groups"),
    (dict(groups=np.array([0, 0, 0]), n_groups=True), "n_groups"),
    (dict(on_error="ignore"), "on_error"),
    (dict(first_stream_sample=5, last_stream_sample=5), "empty"),
    (dict(first_stream_sample=7, last_stream_sample=3), "empty"),
    (dict(last_stream_sample=101), "outside"),
])
def test_bad_arguments_raise(kw, match):
    with pytest.raises(ValueError, match=match):
        _combine(**kw)


def test_flacarray_combine_arguments_raise():
    import flacarray_b200 as fa

    st, nb = _starts()
    far = fa.FlacArray(None, shape=(3, 100), global_shape=(3, 100), compressed=np.zeros(30, np.uint8), dtype=np.float32,
                       stream_starts=st, stream_nbytes=nb, stream_offsets=np.zeros(3, np.float32),
                       stream_gains=np.ones(3, np.float32))
    with pytest.raises(ValueError, match="empty"):
        far.combine(stream_slice=slice(50, 50))
    with pytest.raises(ValueError, match="empty"):
        far.combine(stream_slice=slice(-10, 20))
    with pytest.raises(ValueError, match="step"):
        far.combine(stream_slice=slice(0, 50, 2))
    with pytest.raises(ValueError, match="groups"):
        far.combine(groups=np.array([[0, 1, 2]]).reshape(1, 3)[:, :2])
    with pytest.raises(ValueError, match="weights"):
        far.combine(weights=np.ones(5))
    with pytest.raises(ValueError, match="on_error"):
        far.combine(on_error="skip")


def test_accepted_group_forms():
    """Leading-shape or flat groups, any integer dtype, and n_groups above the largest label all pass the checks."""
    from flacarray_b200 import libflacarray as lf

    w, g, n = lf.check_combine_args(6, None, np.array([[0, -1, 2], [2, 0, -1]], np.int8), None)
    assert w.dtype == np.float64 and np.all(w == 1) and g.tolist() == [0, -1, 2, 2, 0, -1] and n == 3
    w, g, n = lf.check_combine_args(6, np.arange(6, dtype=np.float32), [0, 0, 0, 0, 0, 0], 5)
    assert w.tolist() == [0, 1, 2, 3, 4, 5] and n == 5
    assert lf.check_combine_args(3, None, None, None)[2] == 1
    assert lf.check_combine_args(3, None, np.full(3, -1), None)[2] == 0


def test_no_device_raises():
    """With no CUDA device visible array_combine raises; there is no CPU path."""
    code = ("import numpy as np, flacarray_b200 as fa\n"
            "try:\n"
            "    fa.array_combine(np.zeros(20, np.uint8), 100, np.array([0, 10]), np.array([10, 10]))\n"
            "except RuntimeError as e:\n"
            "    assert 'CUDA' in str(e), e\n"
            "    print('raised')\n")
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=300)
    assert res.returncode == 0 and "raised" in res.stdout, res.stdout + res.stderr
