"""Projections onto templates on the CPU: the host emulation of fab_project_rows (tests/hostsim/hostsim_project.cpp)
against the numpy reference (per 4096-sample piece p = p + T[t, i] * v[i], then the pieces folded in order), bit for bit.

* int32 and int64 rows of random data and of INT32 / INT64 extremes, int64 values above 2^53 (round to nearest even),
  float32 and float64 rows restored with the library's offsets and gains;
* n = 1, n < 4096, n a multiple of 4096 and n = k * 4096 + 1; rows with n % 4 != 0 that start off a 16-byte boundary;
* 1, 3 and 37 templates (one, and more than one, register chunk) with negative, tiny and huge values;
* failed rows give NaN;
* the argument checks of array_project / FlacArray.project raise ValueError without a device, and the emulation runs
  clean under AddressSanitizer + UBSan.
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

PIECE = 4096


@pytest.fixture(scope="module")
def HP():
    import hostsim_project

    hostsim_project.lib()
    return hostsim_project


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


def _templates(n_tmpl, n, seed):
    """Legendre-like smooth templates, sines, random ones, and rows of negative, tiny (1e-300) and huge (1e250) values."""
    rng = np.random.default_rng(seed)
    s = np.linspace(-1.0, 1.0, n)
    t = np.empty((n_tmpl, n))
    for k in range(n_tmpl):
        kind = k % 6
        if kind == 0:
            t[k] = s ** (k // 6)
        elif kind == 1:
            t[k] = np.sin(2 * np.pi * (k + 1) * np.arange(n) / 97.0)
        elif kind == 2:
            t[k] = rng.normal(0, 1, n)
        elif kind == 3:
            t[k] = -rng.uniform(0.5, 2.0, n)
        elif kind == 4:
            t[k] = rng.normal(0, 1, n) * 1e-300
        else:
            t[k] = rng.normal(0, 1, n) * 1e250
    return t


# n = 1, below one piece with n % 4 != 0, exactly two pieces, and two pieces and one sample
SIZES = [1, 1203, 2 * PIECE, 2 * PIECE + 1]


@pytest.mark.parametrize("dtype", [np.int32, np.int64])
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("n_tmpl", [1, 3, 37])
def test_integer_rows(HP, dtype, n, n_tmpl):
    n_rows = 40 if n_tmpl < 37 or n < PIECE else 33      # more than one 32-row block
    x = _rows(dtype, n_rows, n, 3 + n + n_tmpl)
    t = _templates(n_tmpl, n, 9 + n)
    want = HP.reference(x, t)
    got = HP.project_rows(x, t)
    assert _same(got, want)
    assert _same(HP.project_rows(_unaligned(x), t), want)


@pytest.mark.parametrize("dtype", [np.int32, np.int64])
def test_extremes_and_rounding(HP, dtype):
    n = PIECE + 7
    info = np.iinfo(dtype)
    x = np.empty((6, n), dtype)
    x[0] = info.min
    x[1] = info.max
    x[2, 0::2], x[2, 1::2] = info.min, info.max
    x[3] = info.max - np.arange(n, dtype=dtype)
    x[4] = info.min + np.arange(n, dtype=dtype)
    x[5] = -np.arange(n, dtype=dtype)
    if dtype == np.int64:
        # above 2^53 float64(x) rounds to nearest even: ties and non-ties both ways
        base = (1 << 53) + np.arange(n, dtype=np.int64)
        x[3] = base
        x[4] = -(base * 3 + 1)
        assert not np.array_equal(x[3].astype(np.float64).astype(np.int64), x[3])
    t = _templates(6, n, 4)
    assert _same(HP.project_rows(x, t), HP.reference(x, t))
    assert _same(HP.project_rows(x, np.ones((1, n))), HP.reference(x, np.ones((1, n))))


@pytest.mark.parametrize("is_int64", [False, True])
@pytest.mark.parametrize("n", [1203, PIECE + 1])
def test_float_restore(HP, oracle, is_int64, n):
    """Rows restored with offsets and gains from the library's quantisation: the projection of the restored values in
    the array's type, widened, not of a restore in double."""
    fdt = np.float64 if is_int64 else np.float32
    rng = np.random.default_rng(21 + n)
    n_rows = 35
    scale = rng.choice([1.0, 1e3, 1e-6], (n_rows, 1))
    f = (rng.normal(0, 1, (n_rows, n)) * scale + rng.normal(0, 5, (n_rows, 1))).astype(fdt)
    t = _templates(5, n, 2)
    for q in (np.full(n_rows, 1e-4, fdt), None):
        ints, off, gain = oracle.float_to_int(f, q)
        back = oracle.int_to_float(ints, off, gain)
        assert back.dtype == fdt
        got = HP.project_rows(ints, t, offsets=off, gains=gain)
        assert _same(got, HP.reference(back, t))
        assert _same(HP.project_rows(_unaligned(ints), t, offsets=off, gains=gain), got)


def test_piece_order_is_the_definition(HP):
    """The pieces are folded in order after each is summed on its own: a straight running sum over all samples differs
    for these rows, so the piece length is visible in the bits."""
    n = 3 * PIECE
    x = _rows(np.int64, 4, n, 77)
    t = _templates(3, n, 78)
    got = HP.project_rows(x, t)
    assert _same(got, HP.reference(x, t))
    straight = np.zeros((4, 3))
    v = x.astype(np.float64)
    for i in range(n):
        straight = straight + t[None, :, i] * v[:, None, i]
    assert not _same(got, straight)


@pytest.mark.parametrize("restored", [False, True])
def test_failed_rows_are_nan(HP, oracle, restored):
    n_rows, n = 45, PIECE + 100
    x = _rows(np.int32, n_rows, n, 41)
    status = np.zeros(n_rows, np.int32)
    status[[0, 7, 33, 44]] = [1 << 14, 1 << 13, 1 << 14, 1 << 14]
    kw = {}
    vals = x
    if restored:
        f = (np.random.default_rng(43).normal(0, 1, (n_rows, n))).astype(np.float32)
        x, off, gain = oracle.float_to_int(f, np.full(n_rows, 1e-4, np.float32))
        vals = oracle.int_to_float(x, off, gain)
        kw = dict(offsets=off, gains=gain)
    t = _templates(3, n, 44)
    got = HP.project_rows(x, t, status=status, **kw)
    assert _same(got, HP.reference(vals, t, ok=status == 0))
    assert np.isnan(got[status != 0]).all() and np.isfinite(got[status == 0]).all()


def test_argument_errors(HP):
    x = _rows(np.int32, 3, 10, 1)
    for rows, t, bits in ((x[:0], np.ones((1, 10)), 1 << 2), (x, np.ones((0, 10)), 1 << 2),
                          (np.zeros((3, 0), np.int32), np.ones((1, 0)), 1 << 3)):
        with pytest.raises(ValueError, match=f"\\({bits}\\)"):
            HP.project_rows(rows, t)


# ---- argument checks of array_project / FlacArray.project: no device needed ----------------------------------------

def _starts():
    return np.array([0, 10, 20], np.int64), np.array([10, 10, 10], np.int64)


def _project(templates, **kw):
    import flacarray_b200 as fa

    st, nb = _starts()
    return fa.array_project(np.zeros(30, np.uint8), 100, st, nb, templates, **kw)


@pytest.mark.parametrize("templates,kw,match", [
    (np.ones(100, bool), {}, "real"),
    (np.ones(100, np.complex128), {}, "real"),
    (np.array(["a"] * 100), {}, "real"),
    (np.ones((2, 2, 100)), {}, "1-D"),
    (np.float64(1.0), {}, "1-D"),
    (np.ones(99), {}, "samples"),
    (np.ones((2, 101)), {}, "samples"),
    (np.ones(100), dict(first_stream_sample=10), "samples"),
    (np.ones((0, 100)), {}, "no template"),
    (np.ones(100), dict(on_error="ignore"), "on_error"),
    (np.ones(0), dict(first_stream_sample=5, last_stream_sample=5), "empty"),
    (np.ones(0), dict(first_stream_sample=7, last_stream_sample=3), "empty"),
    (np.ones(101), dict(last_stream_sample=101), "outside"),
])
def test_bad_arguments_raise(templates, kw, match):
    with pytest.raises(ValueError, match=match):
        _project(templates, **kw)


def test_torch_templates_checked_without_device():
    import torch

    for t, match in ((torch.ones(100, dtype=torch.bool), "real"), (torch.ones(100, dtype=torch.complex64), "real"),
                     (torch.ones(3, 99), "samples"), (torch.ones(1, 1, 100), "1-D"), (torch.ones(0, 100), "no template")):
        with pytest.raises(ValueError, match=match):
            _project(t)
    from flacarray_b200 import libflacarray as lf

    assert lf.check_project_args(torch.ones(100, dtype=torch.int16), 100) == (1, True)
    assert lf.check_project_args(np.ones((5, 7), np.float32), 7) == (5, False)
    assert lf.check_project_args([[1, 2], [3, 4], [5, 6]], 2) == (3, False)


def test_flacarray_project_arguments_raise():
    import flacarray_b200 as fa

    st, nb = _starts()
    far = fa.FlacArray(None, shape=(3, 100), global_shape=(3, 100), compressed=np.zeros(30, np.uint8), dtype=np.float32,
                       stream_starts=st, stream_nbytes=nb, stream_offsets=np.zeros(3, np.float32),
                       stream_gains=np.ones(3, np.float32))
    with pytest.raises(ValueError, match="empty"):
        far.project(np.ones(0), stream_slice=slice(50, 50))
    with pytest.raises(ValueError, match="empty"):
        far.project(np.ones(0), stream_slice=slice(-10, 20))
    with pytest.raises(ValueError, match="step"):
        far.project(np.ones(25), stream_slice=slice(0, 50, 2))
    with pytest.raises(ValueError, match="samples"):
        far.project(np.ones(100), stream_slice=slice(-30, None))
    with pytest.raises(ValueError, match="real"):
        far.project(np.ones((2, 100), bool))
    with pytest.raises(ValueError, match="on_error"):
        far.project(np.ones(100), on_error="skip")


def test_no_device_raises():
    """With no CUDA device visible array_project raises; there is no CPU path."""
    code = ("import numpy as np, flacarray_b200 as fa\n"
            "try:\n"
            "    fa.array_project(np.zeros(20, np.uint8), 100, np.array([0, 10]), np.array([10, 10]), np.ones(100))\n"
            "except RuntimeError as e:\n"
            "    assert 'CUDA' in str(e), e\n"
            "    print('raised')\n")
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=300)
    assert res.returncode == 0 and "raised" in res.stdout, res.stdout + res.stderr


def test_emulation_under_address_and_ub_sanitizers(tmp_path):
    """Unaligned rows, extremes, partial row tiles and last pieces, several chunks and failed rows once more, against
    an ASan + UBSan build of the emulator in a child process: every read and write stays inside the buffers."""
    import hostsim

    env = hostsim.sanitizer_env()
    if env is None:
        pytest.skip("libasan / libubsan not available")
    import hostsim_project

    so = str(tmp_path / "libhostsim_project_asan.so")
    hostsim_project.build(so, hostsim.SANITIZE)
    script = textwrap.dedent(f"""
        import sys
        import numpy as np
        sys.path[:0] = [{os.path.join(HERE, "hostsim")!r}]
        import hostsim_project as HP
        HP.lib({so!r})
        ok = 0
        for dt in (np.int32, np.int64):
            for n in (1, 37, 4097):
                x = np.zeros((35, n), dt)
                x[:, ::3] = np.iinfo(dt).min
                x[:, 1::5] = np.iinfo(dt).max
                flat = np.empty(x.size + 1, dt)
                y = flat[1:].reshape(x.shape)
                y[...] = x
                st = np.zeros(35, np.int32)
                st[[1, 34]] = 1 << 14
                ok_rows = st == 0
                for n_tmpl in (1, 3, 17):
                    t = np.random.default_rng(n_tmpl).normal(0, 1, (n_tmpl, n))
                    want = HP.reference(x, t, ok=ok_rows)
                    for rows in (x, y):
                        got = HP.project_rows(rows, t, status=st)
                        ok += np.array_equal(got.view(np.uint64), want.view(np.uint64))
        print("project", ok)
    """)
    r = subprocess.run([sys.executable, "-c", script], env=env, capture_output=True, text=True, timeout=1800)
    out = r.stdout + r.stderr
    assert r.returncode == 0, out[-4000:]
    assert "ERROR: AddressSanitizer" not in out and "runtime error" not in out, out[-4000:]
    assert "project 36" in r.stdout, out[-4000:]
