"""Per-stream, per-bin statistics on the CPU: the host emulation of fab_row_stats (tests/hostsim/hostsim_stats.cpp)
against a pure-Python reference built from Python integers and float(int), bit for bit.

* int32 and int64 rows of random data and rows made of INT32_MIN / INT32_MAX / INT64_MIN / INT64_MAX (Q reaches 2^126
  per sample), with bins 1, 7, n - 1, n and None, n not a multiple of the piece, pieces both of the library's length and
  short enough that a bin spans many of them, and rows that do not start on a 16-byte boundary;
* a single-sample row; float mapping with offsets and gains from the library's quantisation, gain 1 and tiny quanta;
  filled rows;
* the finisher's round-to-nearest-even conversion against float(int), ties included;
* argument checks (bin, empty sample range, on_error) raise without a device, and array_stats raises rather than falling
  back when no CUDA device is visible.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, "hostsim"))

I32 = np.iinfo(np.int32)
I64 = np.iinfo(np.int64)


@pytest.fixture(scope="module")
def HS():
    import hostsim_stats

    hostsim_stats.lib()
    return hostsim_stats


def _same(got, want):
    return all(g.dtype == w.dtype and g.shape == w.shape and np.array_equal(g.view(np.uint8), w.view(np.uint8))
               for g, w in zip(got, want))


def _rows(dtype, n_rows, n, seed):
    rng = np.random.default_rng(seed)
    info = np.iinfo(dtype)
    x = rng.integers(info.min, info.max, (n_rows, n), dtype=dtype, endpoint=True)
    x[1] = np.cumsum(rng.integers(-1000, 1001, n)).astype(dtype)        # a typical time stream
    return x


def _unaligned(x):
    """The same rows starting one element past a 16-byte boundary."""
    flat = np.empty(x.size + 1, x.dtype)
    y = flat[1:].reshape(x.shape)
    y[...] = x
    return y


N = 203           # not a multiple of any piece


@pytest.mark.parametrize("dtype", [np.int32, np.int64])
@pytest.mark.parametrize("bin", [None, 1, 7, N - 1, N])
@pytest.mark.parametrize("piece", [0, 24, 100])
def test_random_rows(HS, dtype, bin, piece):
    x = _rows(dtype, 3, N, 5 + (dtype == np.int64))
    got, ppb = HS.row_stats(x, bin, piece=piece)
    assert _same(got, HS.reference(x, bin))
    if piece and bin in (None, N - 1, N):
        assert ppb > 1                   # the bin spans several pieces: the merge ran
    if bin in (1, 7):
        got, _ = HS.row_stats(_unaligned(x), bin, piece=piece)
        assert _same(got, HS.reference(x, bin))


@pytest.mark.parametrize("dtype", [np.int32, np.int64])
@pytest.mark.parametrize("bin", [None, 1, 7, N - 1])
def test_extreme_rows(HS, dtype, bin):
    info = np.iinfo(dtype)
    x = np.empty((4, N), dtype)
    x[0] = info.min
    x[1] = info.max
    x[2, 0::2], x[2, 1::2] = info.min, info.max
    x[3] = info.min
    x[3, ::5] = info.max - 1
    for piece in (0, 32):
        got, _ = HS.row_stats(x, bin, piece=piece)
        assert _same(got, HS.reference(x, bin))
    got, _ = HS.row_stats(_unaligned(x), bin, piece=16)
    assert _same(got, HS.reference(x, bin))


@pytest.mark.parametrize("dtype", [np.int32, np.int64])
def test_single_sample_rows(HS, dtype):
    x = np.array([[np.iinfo(dtype).min], [5], [-3]], dtype)
    for bin in (None, 1, 7):
        got, _ = HS.row_stats(x, bin)
        assert _same(got, HS.reference(x, bin))
        assert list(got[0].reshape(-1)) == [1, 1, 1]
        assert list(got[4].reshape(-1)) == [0.0, 0.0, 0.0]


@pytest.mark.parametrize("is_int64", [False, True])
@pytest.mark.parametrize("bin", [None, 7, 100])
def test_float_mapping(HS, oracle, is_int64, bin):
    """Offsets and gains as the library's quantisation makes them: quanta 1e-4 of a noisy signal, gain exactly 1 (quanta
    1), and quanta so small that the integers use the full range."""
    fdt = np.float64 if is_int64 else np.float32
    rng = np.random.default_rng(11)
    f = (rng.normal(0, 1, (3, N)) * np.array([[1.0], [1e3], [1e-6]]) + np.array([[5.0], [-2e4], [1e-3]])).astype(fdt)
    for q in (np.full(3, 1e-4, fdt), np.ones(3, fdt), None):
        ints, off, gain = oracle.float_to_int(f, q)
        if q is not None and float(q[0]) == 1.0:
            assert np.all(gain == 1)
        got, _ = HS.row_stats(ints, bin, offsets=off, gains=gain, piece=64)
        want = HS.reference(ints, bin, offsets=off, gains=gain)
        assert _same(got, want)
        # min / max are those of the restored samples
        back = oracle.int_to_float(ints, off, gain)
        if bin is None:
            assert np.array_equal(got[1][:, 0], back.min(axis=1)) and np.array_equal(got[2][:, 0], back.max(axis=1))


@pytest.mark.parametrize("dtype", [np.int32, np.int64])
@pytest.mark.parametrize("restored", [False, True])
def test_filled_rows(HS, dtype, restored):
    x = _rows(dtype, 4, N, 17)
    status = np.array([0, 1 << 14, 0, 1 << 13], np.int32)
    fdt = np.float64 if dtype == np.int64 else np.float32
    off = np.array([1.5, -2.0, 0.25, 3.0], fdt) if restored else None
    gain = np.array([1e3, 10.0, 1.0, 7.0], fdt) if restored else None
    for bin in (None, 7):
        got, _ = HS.row_stats(x, bin, offsets=off, gains=gain, status=status, piece=50)
        want = HS.reference(x, bin, offsets=off, gains=gain, status=status)
        assert _same(got, want)
        assert np.all(got[0][[1, 3]] == 0) and np.all(np.isnan(got[3][[1, 3]])) and np.all(np.isnan(got[4][[1, 3]]))
        if restored:
            assert np.all(np.isnan(got[1][[1, 3]])) and np.all(np.isnan(got[2][[1, 3]]))
        else:
            assert np.all(got[1][[1, 3]] == 0) and np.all(got[2][[1, 3]] == 0)


def test_round_to_nearest_even(HS):
    rng = np.random.default_rng(3)
    vals = [0, 1, (1 << 53) - 1, 1 << 53, (1 << 53) + 1, (1 << 54) + 2, (1 << 54) + 6, (1 << 256) - 1,
            ((1 << 53) - 1) << 200, (((1 << 53) - 1) << 200) + (1 << 199), (((1 << 52) + 1) << 100) + (1 << 99),
            (((1 << 52) + 1) << 100) + (1 << 99) + 1, ((1 << 52) << 100) + (1 << 99)]
    for bits in range(1, 257):
        for _ in range(8):
            vals.append(int(rng.integers(0, 1 << 62)) << max(0, bits - 62) | int(rng.integers(0, 2)))
            vals.append(int.from_bytes(rng.bytes(32), "little") >> (256 - bits))
    for v in vals:
        v %= 1 << 256
        assert HS.dbl_u256(v) == float(v), hex(v)


# ---- argument checks of array_stats / FlacArray.stats: no device needed -------------------------------------------------

def _starts():
    return np.array([0, 10], np.int64), np.array([10, 10], np.int64)


@pytest.mark.parametrize("bin", [0, -3, 1.5, True, "4", np.float64(2.0)])
def test_bad_bin_raises(bin):
    import flacarray_b200 as fa

    st, nb = _starts()
    with pytest.raises(ValueError, match="bin"):
        fa.array_stats(np.zeros(20, np.uint8), 100, st, nb, bin=bin)


def test_too_long_bin_raises():
    from flacarray_b200 import libflacarray as lf

    assert lf.check_bin(None, (1 << 32) - 1) == (1 << 32) - 1
    with pytest.raises(ValueError, match="2\\^32"):
        lf.check_bin(None, 1 << 32)
    with pytest.raises(ValueError, match="2\\^32"):
        lf.check_bin(1 << 40, 1 << 33)
    assert lf.check_bin(1 << 40, 100) == 100


@pytest.mark.parametrize("first,last", [(5, 5), (7, 3), (0, 0)])
def test_empty_range_raises(first, last):
    import flacarray_b200 as fa

    st, nb = _starts()
    with pytest.raises(ValueError, match="empty"):
        fa.array_stats(np.zeros(20, np.uint8), 100, st, nb, first_stream_sample=first, last_stream_sample=last)


def test_flacarray_stats_arguments_raise():
    import flacarray_b200 as fa

    st, nb = _starts()
    far = fa.FlacArray(None, shape=(2, 100), global_shape=(2, 100), compressed=np.zeros(20, np.uint8), dtype=np.int32,
                       stream_starts=st, stream_nbytes=nb)
    with pytest.raises(ValueError, match="empty"):
        far.stats(stream_slice=slice(50, 50))
    with pytest.raises(ValueError, match="empty"):
        far.stats(stream_slice=slice(-10, 20))
    with pytest.raises(ValueError, match="step"):
        far.stats(stream_slice=slice(0, 50, 2))
    with pytest.raises(ValueError, match="bin"):
        far.stats(bin=0)
    with pytest.raises(ValueError, match="on_error"):
        far.stats(on_error="ignore")


def test_unknown_on_error_raises():
    import flacarray_b200 as fa

    st, nb = _starts()
    with pytest.raises(ValueError, match="on_error"):
        fa.array_stats(np.zeros(20, np.uint8), 100, st, nb, on_error="skip")


def test_keep_nothing_needs_no_device():
    import flacarray_b200 as fa

    st, nb = _starts()
    s = fa.array_stats(np.zeros(20, np.uint8), 100, st, nb, keep=np.zeros(2, bool), bin=30)
    assert s.count.shape == (0, 4) and s.count.dtype == np.int64 and s.min.dtype == np.int32
    assert s.mean.dtype == np.float64 and s.std.shape == (0, 4)


def test_no_device_raises():
    """With no CUDA device visible array_stats raises; there is no CPU path."""
    code = ("import numpy as np, flacarray_b200 as fa\n"
            "try:\n"
            "    fa.array_stats(np.zeros(20, np.uint8), 100, np.array([0, 10]), np.array([10, 10]))\n"
            "except RuntimeError as e:\n"
            "    assert 'CUDA' in str(e), e\n"
            "    print('raised')\n")
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=300)
    assert res.returncode == 0 and "raised" in res.stdout, res.stdout + res.stderr
