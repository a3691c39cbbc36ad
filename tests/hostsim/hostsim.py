"""ctypes loader of the host emulation of the kernel bodies (tests/hostsim/hostsim.cpp).

TEST HARNESS ONLY: exercises the logic of flacarray_b200/csrc kernel bodies on the CPU so that the
GPU-less container can catch bit-level mistakes early.  Never imported by the product package.
"""
import ctypes as C
import glob
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "hostsim.cpp")
_CXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
_LIB = None

# compiler flags of an AddressSanitizer + UBSan build (see sanitizer_env)
SANITIZE = ["-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined", "-fno-omit-frame-pointer"]


def build(path, flags=("-O2",)):
    """Compile the emulator library to `path` with the optimisation / instrumentation `flags`."""
    subprocess.run([_CXX, *flags, "-std=c++20", "-ffp-contract=off", "-fPIC", "-shared", "-pthread", _SRC, "-o", path],
                   check=True, capture_output=True)


def _sanitizer_runtime(name):
    try:
        p = subprocess.run([_CXX, f"-print-file-name={name}"], capture_output=True, text=True, check=True).stdout.strip()
    except (OSError, subprocess.CalledProcessError):
        return None
    return p if os.path.isabs(p) and os.path.exists(p) else None


def sanitizer_env():
    """The environment of a child process that loads a SANITIZE build, or None without the sanitizer runtimes."""
    asan, ubsan = _sanitizer_runtime("libasan.so"), _sanitizer_runtime("libubsan.so")
    if asan is None or ubsan is None:
        return None
    return dict(os.environ, LD_PRELOAD=f"{asan} {ubsan}", ASAN_OPTIONS="detect_leaks=0:abort_on_error=0",
                UBSAN_OPTIONS="halt_on_error=1:print_stacktrace=1", PYTHONDONTWRITEBYTECODE="1")


def lib(prebuilt=None):
    """The emulator library, built next to this file when older than its sources; `prebuilt`: load that build instead
    (e.g. one with sanitizers)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    so = prebuilt or os.path.join(_HERE, "libhostsim.so")
    deps = [_SRC] + glob.glob(os.path.join(_HERE, "..", "..", "flacarray_b200", "csrc", "*.h"))
    if prebuilt is None and (not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in deps)):
        build(so)
    L = C.CDLL(so)
    p, i64 = C.c_void_p, C.c_int64
    L.hs_encode_bound.restype = i64
    L.hs_encode_bound.argtypes = [i64, i64, C.c_int, C.c_int]
    L.hs_encode.restype = C.c_int
    L.hs_encode.argtypes = [p, C.c_int, i64, i64, C.c_int, p, p, i64, p, p, p, p, C.POINTER(C.c_longlong)]
    L.hs_encode_records.restype = C.c_int
    L.hs_encode_records.argtypes = L.hs_encode.argtypes + [p, p, p]
    L.hs_decode.restype = C.c_int
    L.hs_decode.argtypes = [p, p, p, i64, i64, C.c_int, i64, i64, p, C.c_int, C.POINTER(C.c_int)]
    L.hs_decode_isolated.restype = C.c_int
    L.hs_decode_isolated.argtypes = [p, p, p, i64, i64, C.c_int, i64, i64, p, p, C.POINTER(C.c_int)]
    L.hs_decode_windows.restype = C.c_int
    L.hs_decode_windows.argtypes = [p, p, p, i64, i64, C.c_int, p, p, p, p, i64, C.c_int, p, C.POINTER(C.c_int)]
    L.hs_meta.restype = C.c_int
    L.hs_meta.argtypes = [p, p, p, i64, i64, C.c_int, C.c_int, p, p, i64, p, p]
    L.hs_float_to_int.restype = C.c_int
    L.hs_float_to_int.argtypes = [p, C.c_int, i64, i64, p, p, p, p]
    L.hs_int_to_float.argtypes = [p, C.c_int, i64, i64, p, p, p]
    L.hs_row_stats.restype = C.c_int
    L.hs_row_stats.argtypes = [p, C.c_int, i64, i64, i64, i64] + [p] * 8 + [C.POINTER(i64), C.POINTER(i64)]
    L.hs_dbl_u256.restype = C.c_double
    L.hs_dbl_u256.argtypes = [p]
    L.hs_combine_rows.restype = C.c_int
    L.hs_combine_rows.argtypes = [p, C.c_int, i64, i64] + [p] * 6 + [i64, p, i64, C.POINTER(C.c_int)]
    _LIB = L
    return L


_DT = {np.dtype(np.int32): 0, np.dtype(np.int64): 1, np.dtype(np.float32): 2, np.dtype(np.float64): 3}


# csrc/fa_encode.h FrameStats and FramePlan, one record per (frame, channel)
FRAME_STATS = np.dtype([("mode", "<i4"), ("wasted", "<i4"), ("mn", "<i4"), ("mx", "<i4"), ("bad", "<u4"), ("pad", "<u4"),
                        ("fe", "<u8", 5), ("ac", "<f8", 13)])
FRAME_PLAN = np.dtype([(k, "u1") for k in ("mode", "wasted", "ok0", "ok1", "ord0", "ord1", "shift1", "prec1", "wide1",
                                           "maxp0", "maxp1")] + [("pad", "u1", 5), ("qlp", "<i2", 12),
                                                                 ("fixed_bits", "<u4"), ("pad2", "<u4")])


def encode(arr, level=5, quanta=None, records=False):
    """Emulated fab_encode: (bytes, starts, nbytes, offsets, gains).  records=True appends (stats, plans, fixed):
    FRAME_STATS and FRAME_PLAN arrays [n_stream, nframes, nch] as k_enc_analyze and k_enc_design left them, and a bool
    array [n_stream, nframes] of the frames k_enc_fixed took (their records stay zero)."""
    L = lib()
    a = np.ascontiguousarray(arr)
    a2 = a.reshape(1, -1) if a.ndim == 1 else a.reshape(-1, a.shape[-1])
    n_stream, stream_size = a2.shape
    dt = _DT[a2.dtype]
    nch = 2 if dt in (1, 3) else 1
    cap = L.hs_encode_bound(n_stream, stream_size, nch, level)
    out = np.zeros(cap, np.uint8)
    starts = np.zeros(n_stream, np.int64)
    nbytes = np.zeros(n_stream, np.int64)
    fdt = a2.dtype if dt >= 2 else np.float32
    offs = np.zeros(n_stream, fdt)
    gains = np.zeros(n_stream, fdt)
    q = None if quanta is None else np.ascontiguousarray(quanta, fdt)
    tot = C.c_longlong(0)
    args = [a2.ctypes.data, dt, n_stream, stream_size, level, None if q is None else q.ctypes.data, out.ctypes.data, cap,
            starts.ctypes.data, nbytes.ctypes.data, offs.ctypes.data, gains.ctypes.data, C.byref(tot)]
    if records:
        sb, pb = C.c_int(0), C.c_int(0)
        L.hs_record_sizes(C.byref(sb), C.byref(pb))
        assert (sb.value, pb.value) == (FRAME_STATS.itemsize, FRAME_PLAN.itemsize), "FrameStats / FramePlan layout changed"
        nf = -(-stream_size // (1152 if level <= 2 else 4096))
        stats = np.zeros((n_stream, nf, nch), FRAME_STATS)
        plans = np.zeros((n_stream, nf, nch), FRAME_PLAN)
        fixed = np.zeros((n_stream, nf), np.uint8)
        err = L.hs_encode_records(*args, stats.ctypes.data, plans.ctypes.data, fixed.ctypes.data)
    else:
        err = L.hs_encode(*args)
    if err:
        raise RuntimeError(f"Encoding failed, return code = {err}")
    res = (out[:tot.value].copy(), starts, nbytes, offs, gains)
    return res + (stats, plans, fixed.astype(bool)) if records else res


def _inputs(compressed, starts, nbytes):
    # the throughput decoder reads whole 16-byte chunks: give the host buffer the slack every CUDA allocation has
    c = np.concatenate([np.ascontiguousarray(compressed, np.uint8), np.zeros(64, np.uint8)])
    return c, np.ascontiguousarray(starts, np.int64).reshape(-1), np.ascontiguousarray(nbytes, np.int64).reshape(-1)


def decode(compressed, starts, nbytes, stream_size, first=-1, last=-1, is_int64=False, mode=0):
    """mode 0: the serial reference (meta_body, sync_body, frame_body, walker), mode 1: walker only, mode 2: emulated
    fab_decode.  Returns (data, walked); mode 2: walked = streams walked + 1000 * frames left to the general decoder."""
    L = lib()
    c, st, nb = _inputs(compressed, starts, nbytes)
    n = st.size
    nd = stream_size if not (first >= 0 and last >= 0) else max(last - first, 0)
    nch = 2 if is_int64 else 1
    out = np.zeros((n, nd, nch), np.int32)
    walked = C.c_int(0)
    err = L.hs_decode(c.ctypes.data, st.ctypes.data, nb.ctypes.data, n, stream_size, nch, first, last,
                      out.ctypes.data, mode, C.byref(walked))
    if err:
        raise RuntimeError(f"Decoding failed, return code = {err}")
    res = out.reshape(n, nd * nch).view(np.int64) if is_int64 else out.reshape(n, nd)
    return res, walked.value


def decode_isolated(compressed, starts, nbytes, stream_size, first=-1, last=-1, is_int64=False, store=True):
    """Emulated fab_decode_isolated (store=True) or fab_verify (store=False, whole streams).  Returns (data, status,
    info): data [n, n_decode] int32 / int64 (None when not storing), status int32 [n], info = streams walked + 1000 *
    frames left to the general decoder.  Raises on a call-level error."""
    L = lib()
    c, st, nb = _inputs(compressed, starts, nbytes)
    n = st.size
    nd = stream_size if not (first >= 0 and last >= 0) else max(last - first, 0)
    nch = 2 if is_int64 else 1
    out = np.full((n, nd, nch), 0x5A5A5A5A, np.int32) if store else None
    status = np.full(n, -1, np.int32)
    info = C.c_int(0)
    err = L.hs_decode_isolated(c.ctypes.data, st.ctypes.data, nb.ctypes.data, n, stream_size, nch, first, last,
                               None if out is None else out.ctypes.data, status.ctypes.data, C.byref(info))
    if err:
        raise RuntimeError(f"Decoding failed, return code = {err}")
    if out is not None:
        out = out.reshape(n, nd * nch).view(np.int64) if is_int64 else out.reshape(n, nd)
    return out, status, info.value


def verify(compressed, starts, nbytes, stream_size, is_int64=False):
    """Emulated fab_verify: (status, info)."""
    _, status, info = decode_isolated(compressed, starts, nbytes, stream_size, is_int64=is_int64, store=False)
    return status, info


def decode_windows(compressed, starts, nbytes, stream_size, streams, first, last, is_int64=False, bsh=4096):
    """Emulated fab_decode_windows with packed output and blocksize hint `bsh`.  Returns (flat data, window offsets,
    info) where window i is data[offsets[i]:offsets[i + 1]] and info = windows walked + 1000 * items left to the general
    decoder."""
    L = lib()
    c, st, nb = _inputs(compressed, starts, nbytes)
    ws = np.ascontiguousarray(streams, np.int64).reshape(-1)
    wf = np.ascontiguousarray(first, np.int64).reshape(-1)
    wl = np.ascontiguousarray(last, np.int64).reshape(-1)
    lens = np.maximum(wl - wf, 0)
    offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    wo = np.ascontiguousarray(offs[:-1])
    nch = 2 if is_int64 else 1
    out = np.zeros((int(offs[-1]) + 1) * nch, np.int32)
    info = C.c_int(0)
    err = L.hs_decode_windows(c.ctypes.data, st.ctypes.data, nb.ctypes.data, st.size, stream_size, nch, ws.ctypes.data,
                              wf.ctypes.data, wl.ctypes.data, wo.ctypes.data, ws.size, bsh, out.ctypes.data, C.byref(info))
    if err:
        raise RuntimeError(f"Decoding failed, return code = {err}")
    out = out[:int(offs[-1]) * nch]
    return (out.view(np.int64) if is_int64 else out), offs, info.value


def meta(compressed, starts, nbytes, stream_size, nch, warp):
    """Stage 1 alone, the product's warp body (warp=True) or the serial reference meta_body, with the frame tables
    sized as fab_decode sizes them.  Returns (meta [n, 4] int64: the StreamMeta records, frame offsets [n, cap + 1],
    stream flags [n], status [n])."""
    L = lib()
    c, st, nb = _inputs(compressed, starts, nbytes)
    n = st.size
    m = np.full((n, 4), -7, np.int64)
    fo = np.full(n * (int(stream_size) + 1), -1, np.int64)       # room for any cap (blocksize >= 16 > 1)
    flag = np.full(n, -7, np.int32)
    status = np.full(n, -7, np.int32)
    cap = L.hs_meta(c.ctypes.data, st.ctypes.data, nb.ctypes.data, n, stream_size, nch, 1 if warp else 0, m.ctypes.data,
                    fo.ctypes.data, fo.size, flag.ctypes.data, status.ctypes.data)
    assert cap > 0
    return m, fo[:n * (cap + 1)].reshape(n, cap + 1), flag, status
