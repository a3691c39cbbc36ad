"""Encoder conformance on the GPU (-m gpu): the CUDA encoder writes the same bytes as the host emulator of its kernel
bodies (tests/hostsim) over the CPU matrix of tests/test_encoder_conformance.py, and the paths only a GPU reaches at
real sizes -- several batches of encoder launches with both slot buffers in use, k_enc_fixed's frames mixed with the
frames it declines in one batch, the host-buffer pipelined C entry points above 64 MB -- write strictly valid streams
whose bytes do not depend on their neighbours, their batch or their alignment."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostsim"))

import flac_strict as S  # noqa: E402
import test_encoder_conformance as T  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def fa():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import __graft_entry__ as g

    g.build()
    import flacarray_b200

    return flacarray_b200


@pytest.fixture(scope="module")
def H():
    import hostsim

    hostsim.lib()
    return hostsim


def first_difference(a, b, level, stream_size, nch):
    """'frame j' of the first byte where two encodings a (GPU) and b (emulator) of one stream differ."""
    n = min(a.size, b.size)
    d = np.flatnonzero(a[:n] != b[:n])
    i = int(d[0]) if d.size else n
    rd = S.read_stream(b, level, stream_size, nch)
    j = next((f"frame {f.number}" for f in rd.frames if f.offset <= i < f.offset + f.nbytes), "the stream header")
    return f"{j} (byte {i} of the stream)"


# Signals on which a choice may hinge on near-tied size estimates: the design stage compares them through a
# single-precision log2, which the GPU computes with its approximate MUFU.LG2 and the emulator with the C library's
# log2f.  Their GPU bytes are checked by the strict reader and the choice rules instead of against the emulator.
NEAR_TIES = set(T.adversarial(8))


def gpu_equals_emulator(fa, H, sig, level, quanta=None, name=""):
    """Encode the signals of the dict `sig` on the GPU and in the emulator: the same bytes stream by stream (strictly
    valid GPU streams for the NEAR_TIES signals)."""
    x = np.stack(list(sig.values()))
    comp, st, nb, off, gain = fa.array_compress(x, level=level, quanta=quanta)
    comp, st, nb = np.asarray(comp), np.asarray(st).reshape(-1), np.asarray(nb).reshape(-1)
    e = H.encode(x, level, quanta=None if quanta is None else np.asarray(quanta, x.dtype))
    nch = 2 if x.dtype.itemsize == 8 else 1
    ints = x
    if x.dtype.kind == "f":
        assert np.array_equal(np.asarray(off).reshape(-1), e[3]) and np.array_equal(np.asarray(gain).reshape(-1), e[4]), name
        from oracle import oracle as O

        ints = O.float_to_int(x, np.asarray(quanta, x.dtype))[0]
    for s, key in enumerate(sig):
        g, h = comp[st[s]:st[s] + nb[s]], e[0][e[1][s]:e[1][s] + e[2][s]]
        if np.array_equal(g, h):
            continue
        if key not in NEAR_TIES:
            pytest.fail(f"{name}: GPU bytes of stream {s} ({key}) differ from the emulator's at " +
                        first_difference(g, h, level, x.shape[1], nch))
        rd = S.read_stream(g, level, x.shape[1], nch, f"{name} stream {s} ({key}), GPU", expect=T.channels(ints[s]))
        S.check_choices(rd, level, name=f"{name} stream {s} ({key}), GPU")


@pytest.mark.parametrize("level", range(9))
def test_gpu_bytes_equal_the_emulator_int32(fa, H, level):
    bs = S.PRESETS[level][0]
    for n in T.LENGTHS:
        gpu_equals_emulator(fa, H, T.int32_signals(n, bs), level, name=f"int32 L{level} n={n}")


def test_gpu_bytes_equal_the_emulator_int64_float(fa, H):
    for level in (0, 3, 5, 8):
        for n in (17, 4097, 9001):
            gpu_equals_emulator(fa, H, T.int64_signals(n), level, name=f"int64 L{level} n={n}")
    for dt in (np.float32, np.float64):
        for level in (0, 5):
            for n in (15, 4097, 6001):
                for q in (np.array([1e-3, 1e-4, 0.5], dt), np.array([1e-6, 2.0, 1e-2], dt)):
                    gpu_equals_emulator(fa, H, T.float_signals(n, dt), level, q, name=f"{np.dtype(dt).name} L{level} n={n}")
    for level in (0, 2, 3, 5, 8):
        gpu_equals_emulator(fa, H, T.adversarial(20000), level, name=f"adversarial L{level}")


# ---- real sizes ----------------------------------------------------------------------------------------------------
N_STREAM, STREAM_SIZE = 2000, 135000      # level 0: 118 frames per stream, 236 000 frames: two batches of 231 409


def mixed_level0(seed=91):
    """Rows that k_enc_fixed takes (walks) and rows whose frames it declines: wasted bits, wide samples, constant
    stretches and full-scale noise, interleaved so that every batch holds both kinds."""
    rng = np.random.default_rng(seed)
    x = np.cumsum(rng.integers(-200, 201, (N_STREAM, STREAM_SIZE), dtype=np.int32), axis=1, dtype=np.int32)
    kind = np.arange(N_STREAM) % 5
    x[kind == 1] <<= 3                                              # wasted bits
    x[kind == 2] += 1 << 24                                         # wide samples
    x[kind == 3, 5000:9000] = 77                                    # constant frames inside a predictive stream
    x[kind == 4, ::7] = rng.integers(-2 ** 31, 2 ** 31, x[kind == 4, ::7].shape, dtype=np.int64).astype(np.int32)
    return x


def batch_edges(level, nch, n_stream, stream_size):
    """The streams holding the first and the last frame of every batch of encoder launches (fa_api.cu enc_workspace)."""
    bs = S.PRESETS[level][0]
    nf = -(-stream_size // bs)
    total = n_stream * nf
    batch = min(total, max(1024, (1 << 30) // ((16 + 2 + nch * (4 * bs + 8) + 15) & ~15)))
    out = set()
    for b0 in range(0, total, batch):
        out.update({b0 // nf, (min(b0 + batch, total) - 1) // nf})
    return sorted(out), -(-total // batch)


def check_sampled_streams(fa, H, x, comp, st, nb, level, seed):
    nch = 2 if x.dtype.itemsize == 8 else 1
    edges, nbatch = batch_edges(level, nch, *x.shape)
    assert nbatch >= 2
    rng = np.random.default_rng(seed)
    sample = sorted(set(edges) | set(rng.choice(x.shape[0], 4, replace=False).tolist()) | {0, x.shape[0] - 1})
    for s in sample:
        b = comp[st[s]:st[s] + nb[s]]
        S.read_stream(b, level, x.shape[1], nch, f"stream {s}", expect=T.channels(x[s]))
        one = np.asarray(fa.array_compress(np.ascontiguousarray(x[s:s + 1]), level=level)[0])
        assert np.array_equal(one, b), f"stream {s}: encoded alone on the GPU, different bytes"
        if s in edges[:2] or s == sample[-1]:        # (the emulator takes a few seconds per long stream)
            assert np.array_equal(H.encode(x[s:s + 1], level)[0], b), f"stream {s}: the emulator's bytes differ"
    return sample


def test_many_batches_mixed_fixed_kernel_frames(fa, H):
    """One level-0 call of 236 000 frames (two batches, both slot buffers), each batch mixing frames k_enc_fixed takes
    with frames it declines.  Sampled streams, and the first and last stream of every batch, are strictly valid and
    equal to the same stream encoded alone (GPU and emulator); the whole output round-trips through the GPU decoder."""
    x = mixed_level0()
    comp, st, nb, _, _ = fa.array_compress(x, level=0)
    comp, st, nb = np.asarray(comp), np.asarray(st).reshape(-1), np.asarray(nb).reshape(-1)
    check_sampled_streams(fa, H, x, comp, st, nb, 0, seed=5)
    assert np.array_equal(np.asarray(fa.array_decompress(comp, STREAM_SIZE, st, nb)).reshape(x.shape), x)


def test_host_pipelined_entry_point_above_64mb(fa, H):
    """The same array through the host-buffer C entry point (chunked pinned staging above 64 MB) gives the same bytes
    as the device path, and its streams pass the same checks."""
    from flacarray_b200 import _lib

    L = C.CDLL(_lib.SO_PATH)
    libc = C.CDLL(None)
    x = mixed_level0(seed=92)
    starts = np.zeros(N_STREAM, np.int64)
    nbt = C.c_int64(0)
    buf = C.POINTER(C.c_ubyte)()
    L.encode_i32_threaded.restype = C.c_int
    rc = L.encode_i32_threaded(C.c_void_p(x.ctypes.data), C.c_int64(N_STREAM), C.c_int64(STREAM_SIZE), C.c_uint32(0),
                               C.byref(nbt), C.c_void_p(starts.ctypes.data), C.byref(buf))
    assert rc == 0 and nbt.value > 0
    comp = np.ctypeslib.as_array(buf, shape=(nbt.value,)).copy()
    libc.free(buf)
    nb = np.empty(N_STREAM, np.int64)
    nb[:-1] = np.diff(starts)
    nb[-1] = nbt.value - starts[-1]
    dev = np.asarray(fa.array_compress(x, level=0)[0])
    assert np.array_equal(comp, dev)
    check_sampled_streams(fa, H, x, comp, starts, nb, 0, seed=6)
