"""CPU-side checks: the C-ABI library builds for sm_100a, loads, and exports every symbol that
include/flacarray_b200.h declares; the product path fails loudly without a GPU."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def so_path():
    from flacarray_b200 import _lib

    return _lib.build()


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "flacarray_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    names = re.findall(r"\b(?:int|void|int64_t|double|const char\*)\s+\*?\s*([a-z_0-9]+)\s*\(", text)
    return sorted(set(names))


def test_header_symbols_are_exported(so_path):
    from flacarray_b200 import _lib

    L = ctypes.CDLL(so_path)
    declared = _declared_symbols()
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(L, name), f"{name} declared in the header but not exported"
    assert sorted(_lib.EXPORTED) == declared


def test_sass_is_sm100(so_path):
    import shutil
    import subprocess

    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-lelf", so_path], capture_output=True, text=True).stdout
    assert "sm_100a" in out


_NO_CPU_FALLBACK = """
import numpy as np
import pytest
import torch

assert not torch.cuda.is_available()
import flacarray_b200 as fa

with pytest.raises(RuntimeError, match="no CPU fallback"):
    fa.array_compress(np.zeros((2, 64), np.int32))
with pytest.raises(RuntimeError, match="no CPU fallback"):
    fa.float_to_int(np.zeros((2, 64), np.float32), quanta=1e-3)
"""


def test_no_cpu_fallback():
    """Without a CUDA device the product path raises.  Runs in a child process that sees no device, so that it
    checks the same on a machine with a GPU."""
    import subprocess
    import sys

    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = subprocess.run([sys.executable, "-s", "-c", _NO_CPU_FALLBACK], cwd=ROOT, env=env, capture_output=True,
                         text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]


def test_argument_validation_matches_reference():
    """Checks that happen before any device work (pyx:551-559, :751-789; compress.py:47-59)."""
    import flacarray_b200 as fa
    from flacarray_b200.libflacarray import decode_flac, encode_flac

    with pytest.raises(ValueError):
        fa.array_compress(np.zeros((0, 5), np.int32))
    with pytest.raises(RuntimeError, match="requires specifying either quanta or precision"):
        fa.array_compress(np.zeros((2, 5), np.float32))
    with pytest.raises(RuntimeError, match="both quanta and precision"):
        fa.array_compress(np.zeros((2, 5), np.float32), quanta=1.0, precision=3)
    with pytest.raises(ValueError, match="Unsupported data type"):
        fa.array_compress(np.zeros((2, 5), np.int16))
    with pytest.raises(RuntimeError, match="Only 32bit or 64bit integer"):
        encode_flac(np.zeros((2, 5), np.float32), 5)
    with pytest.raises(RuntimeError, match="C-contiguous"):
        encode_flac(np.zeros((5, 4), np.int32).T, 5)
    with pytest.raises(RuntimeError, match="levels 0-8"):
        encode_flac(np.zeros((2, 5), np.int32), 9)
    c = np.zeros(10, np.uint8)
    s = np.zeros(1, np.int64)
    with pytest.raises(RuntimeError, match="type uint8"):
        decode_flac(c.astype(np.int8), s, s, 5)
    with pytest.raises(RuntimeError, match="starts data should be of type int64"):
        decode_flac(c, s.astype(np.int32), s, 5)
    with pytest.raises(RuntimeError, match="non-zero output stream size"):
        decode_flac(c, s, s, 0)
    with pytest.raises(RuntimeError, match="last_sample is beyond end"):
        decode_flac(c, s, s, 5, first_sample=0, last_sample=6)
    with pytest.raises(RuntimeError, match="first_sample is beyond"):
        decode_flac(c, s, s, 5, first_sample=5, last_sample=5)
    with pytest.raises(RuntimeError, match="larger than last_sample"):
        decode_flac(c, s, s, 5, first_sample=3, last_sample=2)


def test_keep_select_matches_reference_loop():
    from flacarray_b200.utils import keep_select, select_keep_indices

    rng = np.random.default_rng(0)
    starts = np.arange(24, dtype=np.int64).reshape(2, 3, 4) * 10
    nbytes = starts + 1
    keep = rng.random((2, 3, 4)) > 0.5
    s, n, idx = keep_select(keep, starts, nbytes)
    # the reference's nditer loop (utils.py:436-444)
    es, en, eidx = [], [], []
    it = np.nditer(keep, order="C", flags=["multi_index"])
    for st in it:
        if st:
            es.append(starts[it.multi_index]); en.append(nbytes[it.multi_index]); eidx.append(it.multi_index)
    assert s.tolist() == es and n.tolist() == en and idx == eidx
    assert s.dtype == np.int64 and isinstance(idx[0], tuple)
    off = rng.random((2, 3, 4)).astype(np.float32)
    assert np.array_equal(select_keep_indices(off, idx), np.array([off[i] for i in idx], np.float32))
    assert keep_select(None, starts, nbytes) == (starts, nbytes, None)
    with pytest.raises(RuntimeError):
        keep_select(keep[0], starts, nbytes)


def test_host_pipeline_chunks_cover_every_stream_once():
    """Host-buffer pipelines cut the array into whole-stream chunks: every stream exactly once, in order, with a short
    first and last chunk (the only copy-in / copy-out nothing overlaps) when the array is long enough."""
    from flacarray_b200 import libflacarray as lf

    for n_stream, bps in [(1, 10), (2, 1 << 30), (7, 50 << 20), (1000, 4_000_000), (4096, 16_000_000), (50, 4_000_000),
                          (100, 1000), (3, 100_000_000), (12345, 40_000)]:
        r = lf._chunk_ranges(n_stream, bps)
        assert r[0][0] == 0 and r[-1][1] == n_stream
        assert all(a < b for a, b in r) and all(r[i][1] == r[i + 1][0] for i in range(len(r) - 1))
        if n_stream * bps < lf._PIPE_MIN_BYTES:
            assert len(r) == 1
    sizes = [b - a for a, b in lf._chunk_ranges(1000, 4_000_000)]
    assert sizes[0] < sizes[1] < sizes[2] and sizes[-1] < sizes[-2] < sizes[-3]
    assert max(sizes) * 4_000_000 <= lf._PIPE_CHUNK_BYTES * 1.05
