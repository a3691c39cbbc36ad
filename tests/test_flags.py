"""Ranges of out-of-threshold samples on the CPU: the host emulation of fab_flag_count + fab_flag_write
(tests/hostsim/hostsim_flags.cpp, the bodies of flacarray_b200/csrc/fa_flags.h) against a numpy reference, exactly.

* runs that cross piece boundaries and runs that end on a piece's last sample, with pieces short enough that a row spans
  many of them; gaps of exactly 2 * pad + 1 (merged) and 2 * pad + 2 (not merged); pad 0, 1, 7 and larger than the row;
* no flagged samples, all flagged, alternating flags; the first and last samples of the row flagged; rows that do not
  start on a 16-byte boundary;
* int32 and int64 rows with INT64_MIN / INT64_MAX values and bounds, L > H, rows with a non-zero status;
* flag_bounds against a per-sample restore and compare: exhaustively over a 2^20-wide int32 window, on random int64
  samples, for coeff > 0 and < 0, with thresholds equal to a restored value (not flagged);
* argument checks raise ValueError without a device, and the malformed inputs once more under ASan + UBSan.
"""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, "hostsim"))

I64 = np.iinfo(np.int64)


@pytest.fixture(scope="module")
def HF():
    import hostsim_flags

    hostsim_flags._lib()
    return hostsim_flags


def _check(HF, rows, L, H, pad, piece=32, status=None, sample0=0):
    """Emulated ranges equal the numpy reference; returns the reference."""
    got = HF.flag_ranges(rows, L, H, pad=pad, piece=piece, status=status, sample0=sample0)
    want = HF.reference(HF.flags_of(rows, L, H), pad, status=status, sample0=sample0)
    for g, w, name in zip(got, want, ("stream", "first", "last", "nflag")):
        assert np.array_equal(g, w), (name, g, w)
    nr = np.bincount(want[0], minlength=rows.shape[0])
    assert np.array_equal(got[4], nr)
    return want


def _unaligned(x):
    """The same rows starting one element past a 16-byte boundary."""
    flat = np.empty(x.size + 1, x.dtype)
    y = flat[1:].reshape(x.shape)
    y[...] = x
    return y


def _planted(dtype, n, flagged):
    """Rows of zeros with the samples in `flagged` (one list per row) set to 100."""
    x = np.zeros((len(flagged), n), dtype)
    for r, idx in enumerate(flagged):
        x[r, list(idx)] = 100
    return x


@pytest.mark.parametrize("dtype", [np.int32, np.int64])
@pytest.mark.parametrize("piece", [32, 64, 0])
def test_runs_across_pieces(HF, dtype, piece):
    """Runs crossing piece boundaries, ending on a piece's last sample, starting on a piece's first; rows of 203 samples
    (n % 4 != 0, so every row but the first starts off a 16-byte boundary)."""
    n = 203
    flagged = [range(28, 40), range(60, 64), range(64, 70), [0, 31, 32, 95, 96, 127, 128, 202], range(0, 203), []]
    x = _planted(dtype, n, flagged)
    for pad in (0, 1, 7):
        _check(HF, x, -5, 5, pad, piece)
        _check(HF, _unaligned(x), -5, 5, pad, piece)


@pytest.mark.parametrize("dtype", [np.int32, np.int64])
def test_rows_of_many_pieces(HF, dtype):
    """Rows of 82 pieces: the offsets pass walks them 32 at a time, carrying the last flagged sample forwards and the
    next one backwards from one group of 32 pieces to the next -- runs and gaps across samples 1024 and 2048."""
    n = 2600
    flagged = [[1020, 1027], [1023, 1024], [1000, 1030, 2040, 2049], [5, 1024 + 3 * 32 * 32 // 3, 2047, 2048, 2599],
               [1023], list(range(990, 1060, 9))]
    x = _planted(dtype, n, flagged)
    for pad in (0, 3, 4, 15):
        _check(HF, x, -1, 1, pad, 32)
        _check(HF, _unaligned(x), -1, 1, pad, 32)


@pytest.mark.parametrize("dtype", [np.int32, np.int64])
@pytest.mark.parametrize("pad", [0, 1, 7, 20])
def test_gap_of_exactly_two_pad_plus_one(HF, dtype, pad):
    """Flagged samples 2 * pad + 1 apart share a range; 2 * pad + 2 apart they do not -- also across piece boundaries."""
    n = 300
    g = 2 * pad + 1
    starts = [3, 30, 62, 95]
    merged = [[s, s + g] for s in starts]
    split = [[s, s + g + 1] for s in starts]
    x = _planted(dtype, n, merged + split)
    want = _check(HF, x, -1, 1, pad, 32)
    assert np.array_equal(np.bincount(want[0], minlength=8), [1] * 4 + [2] * 4)


@pytest.mark.parametrize("dtype", [np.int32, np.int64])
def test_large_pad(HF, dtype):
    """A pad larger than the row (up to INT64_MAX) covers the whole row with one range."""
    x = _planted(dtype, 150, [[70], [0, 149], [5, 140], []])
    for pad in (150, 151, 10 ** 12, int(I64.max)):
        s, f, l_, _ = _check(HF, x, -1, 1, pad, 32, sample0=1000)
        assert s.tolist() == [0, 1, 2] and f.tolist() == [1000] * 3 and l_.tolist() == [1150] * 3


@pytest.mark.parametrize("dtype", [np.int32, np.int64])
def test_none_all_alternating(HF, dtype):
    """No flagged samples, all flagged, alternating flags (n / 2 ranges at pad 0, one at pad >= 1)."""
    n = 257
    x = np.zeros((3, n), dtype)
    x[1] = 9
    x[2, ::2] = 9
    for pad in (0, 1, 3):
        s, f, l_, nf = _check(HF, x, -1, 1, pad, 64)
        assert nf.tolist() == [0, n, (n + 1) // 2]
        assert np.sum(s == 2) == ((n + 1) // 2 if pad == 0 else 1)
    _check(HF, x, -1, 1, 0, 0)


@pytest.mark.parametrize("dtype", [np.int32, np.int64])
def test_first_and_last_samples(HF, dtype):
    """The first and last samples of the row flagged, with a sample0 offset: ranges clip to [sample0, sample0 + n)."""
    x = _planted(dtype, 97, [[0], [96], [0, 96], [1, 95]])
    for pad in (0, 1, 2, 5):
        s, f, l_, _ = _check(HF, x, -1, 1, pad, 32, sample0=500)
        assert f.min() >= 500 and l_.max() <= 597


@pytest.mark.parametrize("dtype", [np.int32, np.int64])
def test_random_rows(HF, dtype):
    rng = np.random.default_rng(7 + (dtype == np.int64))
    x = rng.integers(-1000, 1001, (5, 333)).astype(dtype)
    L = np.array([-990, -900, -500, 0, -2000], np.int64)
    H = np.array([990, 900, 500, 0, 2000], np.int64)
    for pad in (0, 2, 9):
        for piece in (32, 96, 0):
            _check(HF, x, L, H, pad, piece)


def test_int64_extremes(HF):
    """INT64_MIN / INT64_MAX samples and bounds, and L > H (every sample flagged)."""
    x = np.zeros((6, 130), np.int64)
    x[:, ::7] = I64.min
    x[:, 3::11] = I64.max
    x[:, 5::13] = I64.min + 1
    x[:, 6::17] = I64.max - 1
    L = np.array([I64.min, I64.min + 1, -1, I64.min, 1, I64.max], np.int64)
    H = np.array([I64.max, I64.max - 1, 1, I64.max - 1, 0, I64.min], np.int64)
    s, f, l_, nf = _check(HF, x, L, H, 0, 32)
    assert nf[0] == 0 and nf[4] == 130 and nf[5] == 130
    _check(HF, _unaligned(x), L, H, 1, 64)


def test_int32_rows_with_int64_bounds(HF):
    """int32 rows with bounds beyond the int32 range: L below INT32_MIN, H above INT32_MAX, L above INT32_MAX (all
    flagged) and H below INT32_MIN (all flagged)."""
    i32 = np.iinfo(np.int32)
    x = np.zeros((5, 101), np.int32)
    x[:, ::5] = i32.min
    x[:, 2::7] = i32.max
    L = np.array([int(i32.min) - 1, int(i32.min), int(i32.max) + 1, I64.min, int(i32.min) + 1], np.int64)
    H = np.array([int(i32.max) + 1, int(i32.max) - 1, I64.max, int(i32.min) - 1, int(i32.max)], np.int64)
    s, f, l_, nf = _check(HF, x, L, H, 0, 32)
    assert nf[0] == 0 and nf[2] == 101 and nf[3] == 101


@pytest.mark.parametrize("dtype", [np.int32, np.int64])
def test_rows_with_status(HF, dtype):
    rng = np.random.default_rng(3)
    x = rng.integers(-50, 51, (4, 200)).astype(dtype)
    status = np.array([0, 1 << 14, 0, 1 << 13], np.int32)
    s, f, l_, nf = _check(HF, x, -40, 40, 1, 32, status=status)
    assert nf[1] == -1 and nf[3] == -1 and not np.isin(s, [1, 3]).any()


def test_float_rows_match_per_sample_compare(HF):
    """Float rows: [L, H] from flag_bounds in the scan gives the flags of the restored values."""
    rng = np.random.default_rng(12)
    for is_int64 in (False, True):
        dt, fdt = (np.int64, np.float64) if is_int64 else (np.int32, np.float32)
        x = rng.integers(-5000, 5001, (4, 150)).astype(dt)
        off = np.array([0.5, -3.0, 1e3, 0.0], fdt)
        gain = np.array([100.0, -7.0, 1e-3, 3.0], fdt)
        coeff = np.array([_coeff(g, is_int64) for g in gain])
        lo = np.array([-20.0, -np.inf, 900.0, 5.0])
        hi = np.array([20.0, 100.0, np.inf, -5.0])             # the last row: lo > hi, every sample flagged
        got = HF.flag_ranges(x, lo, hi, pad=2, offsets=off, gains=gain, piece=32)
        want = HF.reference(HF.flags_of(x, lo, hi, off, coeff), 2)
        for g, w in zip(got, want):
            assert np.array_equal(g, w)
        assert got[3][3] == 150


def _coeff(gain, is_int64):
    return float(np.float64(1.0 / np.float64(gain))) if is_int64 else float(np.float32(1.0 / np.float64(gain)))


# ---- flag_bounds --------------------------------------------------------------------------------------------------------

def _bounds_agree(HF, is_int64, off, coeff, lo, hi, xs):
    L, H = HF.flag_bounds(is_int64, off, coeff, lo, hi)
    v = HF.restore(xs, off, coeff, is_int64)
    direct = (v < lo) | (v > hi)
    by_bounds = (xs < L) | (xs > H)
    assert np.array_equal(direct, by_bounds), (off, coeff, lo, hi, L, H)
    return L, H


@pytest.mark.parametrize("coeff", [1e-4, 3.7, -2.5e-3, -1.0])
def test_bounds_int32_exhaustive_window(HF, coeff):
    """Every int32 of a 2^20-wide window around each threshold, thresholds at a restored value (not flagged) and just
    beside one."""
    off = np.float32(0.375)
    c = np.float32(coeff)
    for x0 in (0, 123457, -2 ** 30, 2 ** 31 - 2 ** 19 - 1):
        xs = np.arange(x0 - 2 ** 19, x0 + 2 ** 19, dtype=np.int64)
        xs = xs[(xs >= -2 ** 31) & (xs < 2 ** 31)].astype(np.int32)
        t = float(HF.restore(np.array([x0], np.int32), off, c, False)[0])
        for lo, hi in ((t, np.inf), (-np.inf, t), (t, t), (np.nextafter(t, -np.inf), np.nextafter(t, np.inf)),
                       (t - abs(float(c)) * 1000, t + abs(float(c)) * 1000)):
            L, H = _bounds_agree(HF, False, float(off), float(c), lo, hi, xs)
            if lo == t or hi == t:
                assert L <= x0 <= H                          # the equal value is not flagged


@pytest.mark.parametrize("coeff", [1e-12, 2.5, -1e-9, -3.0])
def test_bounds_int64_random(HF, coeff):
    rng = np.random.default_rng(99)
    off = -12.5
    xs = np.concatenate([rng.integers(I64.min, I64.max, 20000, dtype=np.int64, endpoint=True),
                         rng.integers(-10 ** 6, 10 ** 6, 20000, dtype=np.int64), np.array([I64.min, I64.max, 0, -1, 1])])
    for x0 in (0, 10 ** 5, -(10 ** 15), int(I64.max) - 5):
        t = float(HF.restore(np.array([x0], np.int64), off, coeff, True)[0])
        near = np.arange(max(x0 - 3000, int(I64.min)), min(x0 + 3000, int(I64.max)), dtype=np.int64)
        for lo, hi in ((t, np.inf), (-np.inf, t), (t, t), (t - abs(coeff) * 1e4, t + abs(coeff) * 1e4)):
            L, H = _bounds_agree(HF, True, off, coeff, lo, hi, np.concatenate([xs, near]))
            if lo == t or hi == t:
                assert L <= x0 <= H


def test_bounds_empty_and_full(HF):
    """lo > hi, thresholds beyond every restored value, and open sides."""
    for is_int64 in (False, True):
        assert HF.flag_bounds(is_int64, 0.0, 1.0, 5.0, 4.0)[0] > HF.flag_bounds(is_int64, 0.0, 1.0, 5.0, 4.0)[1]
        L, H = HF.flag_bounds(is_int64, 0.0, 1.0, -np.inf, np.inf)
        lim = (I64.min, I64.max) if is_int64 else (-2 ** 31, 2 ** 31 - 1)
        assert (L, H) == lim
        L, H = HF.flag_bounds(is_int64, 0.0, 1.0, 1e300, np.inf)
        assert L > H
        L, H = HF.flag_bounds(is_int64, 0.0, -1.0, -np.inf, -1e300)
        assert L > H


# ---- argument checks of array_flag_ranges / FlacArray.flag_ranges: no device needed ------------------------------------

def _starts():
    return np.array([0, 10], np.int64), np.array([10, 10], np.int64)


@pytest.mark.parametrize("kw", [
    dict(), dict(lo=None, hi=None), dict(lo=np.nan), dict(hi=np.array([1.0, np.nan])), dict(lo=True),
    dict(hi=np.array([True, False])), dict(lo="3"), dict(hi=np.array([1, 2, 3])), dict(lo=np.zeros((3, 1))),
    dict(lo=0, pad=-1), dict(lo=0, pad=True), dict(lo=0, pad=1.5), dict(lo=0, pad=np.float64(2.0)),
    dict(lo=0, first_stream_sample=5, last_stream_sample=5), dict(lo=0, first_stream_sample=7, last_stream_sample=3),
    dict(lo=0, on_error="skip"), dict(lo=0, keep=np.array([1, 0])),
])
def test_bad_arguments_raise(kw):
    import flacarray_b200 as fa

    st, nb = _starts()
    with pytest.raises(ValueError):
        fa.array_flag_ranges(np.zeros(20, np.uint8), 100, st, nb, **kw)


def test_threshold_conversion_for_integer_streams():
    """Integer thresholds as they are, a float lo as x < ceil(lo), a float hi as x > floor(hi), exact at +-2^63."""
    from flacarray_b200 import libflacarray as lf

    L, H, pad = lf.check_flag_args(3, 2.5, np.array([7.9, -1.0, 2.0 ** 70]), np.int64(4), False)
    assert L.tolist() == [3, 1, 3] and H.tolist() == [7, 0, I64.max] and pad == 4    # stream 1: every sample flagged
    L, H, _ = lf.check_flag_args(2, -(2 ** 63), 2 ** 63 - 1, 0, False)
    assert L.tolist() == [I64.min] * 2 and H.tolist() == [I64.max] * 2
    L, H, _ = lf.check_flag_args(2, None, np.array([2.0 ** 63, -(2.0 ** 63)]), 0, False)
    assert L.tolist() == [I64.min] * 2 and H.tolist() == [I64.max, I64.min]    # only INT64_MIN is kept by stream 1
    L, H, _ = lf.check_flag_args(1, None, -(2 ** 63) - 1, 0, False)          # below every int64: every sample
    assert L[0] > H[0]
    L, H, _ = lf.check_flag_args(1, 9223372036854775807, None, 0, False)
    assert (L[0], H[0]) == (I64.max, I64.max)
    L, H, _ = lf.check_flag_args(1, 2 ** 63, None, 0, False)                 # above every int64: every sample
    assert L[0] > H[0]
    L, H, _ = lf.check_flag_args(2, -np.inf, np.array([np.inf, -np.inf]), 0, False)
    assert L[0] == I64.min and H[0] == I64.max and L[1] > H[1]
    lo, hi, _ = lf.check_flag_args(2, 3, None, 0, True)
    assert lo.dtype == np.float64 and lo.tolist() == [3.0, 3.0] and np.all(np.isinf(hi))


def test_flacarray_flag_ranges_arguments_raise():
    import flacarray_b200 as fa

    st, nb = _starts()
    far = fa.FlacArray(None, shape=(2, 100), global_shape=(2, 100), compressed=np.zeros(20, np.uint8), dtype=np.int32,
                       stream_starts=st, stream_nbytes=nb)
    with pytest.raises(ValueError, match="empty"):
        far.flag_ranges(lo=0, stream_slice=slice(50, 50))
    with pytest.raises(ValueError, match="step"):
        far.flag_ranges(lo=0, stream_slice=slice(0, 50, 2))
    with pytest.raises(ValueError, match="lo, hi"):
        far.flag_ranges()
    with pytest.raises(ValueError, match="pad"):
        far.flag_ranges(hi=3, pad=-2)
    with pytest.raises(ValueError, match="on_error"):
        far.flag_ranges(hi=3, on_error="ignore")


def test_keep_nothing_needs_no_device():
    import flacarray_b200 as fa

    st, nb = _starts()
    r = fa.array_flag_ranges(np.zeros(20, np.uint8), 100, st, nb, lo=-1, keep=np.zeros(2, bool))
    assert type(r).__name__ == "FlagRanges" and r.stream.size == 0 and r.nflagged.tolist() == [-1, -1]
    r, status = fa.array_flag_ranges(np.zeros(20, np.uint8), 100, st, nb, hi=1, keep=np.zeros(2, bool), on_error="fill")
    assert status.tolist() == [0, 0] and r.first.dtype == np.int64


def test_c_entry_rejects_arguments(HF):
    x = np.zeros((2, 64), np.int32)
    with pytest.raises(ValueError, match="error 131072"):
        HF.flag_ranges(x, 0, 0, pad=-1)
    with pytest.raises(ValueError, match="error 131072"):
        HF.flag_ranges(x, 0, 0, piece=48)


def test_no_device_raises():
    """With no CUDA device visible array_flag_ranges raises; there is no CPU path."""
    code = ("import numpy as np, flacarray_b200 as fa\n"
            "try:\n"
            "    fa.array_flag_ranges(np.zeros(20, np.uint8), 100, np.array([0, 10]), np.array([10, 10]), lo=0)\n"
            "except RuntimeError as e:\n"
            "    assert 'CUDA' in str(e), e\n"
            "    print('raised')\n")
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=300)
    assert res.returncode == 0 and "raised" in res.stdout, res.stdout + res.stderr


def test_malformed_inputs_under_address_and_ub_sanitizers(tmp_path):
    """Unaligned rows, extreme values and bounds, huge pads, all-flagged and failed rows once more, against an ASan +
    UBSan build of the emulator in a child process: every read and write stays inside the buffers and slots."""
    import hostsim
    import hostsim_flags

    env = hostsim.sanitizer_env()
    if env is None:
        pytest.skip("libasan / libubsan not available")
    so = str(tmp_path / "libhostsim_flags_asan.so")
    hostsim_flags.build(so, hostsim.SANITIZE)
    script = textwrap.dedent(f"""
        import sys
        import numpy as np
        sys.path[:0] = [{os.path.join(HERE, "hostsim")!r}]
        import hostsim_flags as HF
        HF._lib({so!r})
        I = np.iinfo(np.int64)
        ok = 0
        for dt in (np.int32, np.int64):
            x = np.zeros((4, 101), dt)
            x[:, ::3] = np.iinfo(dt).min
            x[:, 1::5] = np.iinfo(dt).max
            x[3] = 1
            flat = np.empty(x.size + 1, dt)
            y = flat[1:].reshape(x.shape)
            y[...] = x
            L = np.array([I.min, -5, 1, 0], np.int64)
            H = np.array([I.max, 5, 0, 0], np.int64)
            st = np.array([0, 1 << 14, 0, 0], np.int32)
            for rows in (x, y):
                for pad in (0, 3, 200, int(I.max)):
                    for piece in (32, 0):
                        got = HF.flag_ranges(rows, L, H, pad=pad, piece=piece, status=st, sample0=7)
                        want = HF.reference(HF.flags_of(x, L, H), pad, status=st, sample0=7)
                        ok += all(np.array_equal(g, w) for g, w in zip(got, want))
            for bad in (dict(pad=-1), dict(piece=40)):
                try:
                    HF.flag_ranges(x, L, H, **bad)
                except ValueError:
                    ok += 1
        print("flags", ok)
    """)
    r = subprocess.run([sys.executable, "-c", script], env=env, capture_output=True, text=True, timeout=900)
    out = r.stdout + r.stderr
    assert r.returncode == 0, out[-4000:]
    assert "ERROR: AddressSanitizer" not in out and "runtime error" not in out, out[-4000:]
    assert "flags 36" in r.stdout, out[-4000:]
