"""ctypes loader of the host emulation of the kernel bodies (tests/hostsim/hostsim.cpp).

TEST HARNESS ONLY: exercises the logic of flacarray_b200/csrc kernel bodies on the CPU so that the
GPU-less container can catch bit-level mistakes early.  Never imported by the product package.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def lib(prebuilt=None):
    """The emulator library, built next to this file when stale; `prebuilt`: load that build instead (e.g. one with
    sanitizers)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    so = prebuilt or os.path.join(_HERE, "libhostsim.so")
    srcs = [os.path.join(_HERE, "hostsim.cpp")] + [
        os.path.join(_HERE, "..", "..", "flacarray_b200", "csrc", f)
        for f in ("fa_simt.h", "fa_bits.h", "fa_quant.h", "fa_decode.h", "fa_decode_tile.h", "fa_encode.h", "fa_encode_fixed.h")]
    if prebuilt is None and (not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs)):
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.run([cxx, "-O2", "-std=c++20", "-ffp-contract=off", "-fPIC", "-shared", "-pthread",
                        srcs[0], "-o", so], check=True, capture_output=True)
    L = C.CDLL(so)
    L.hs_encode_bound.restype = C.c_int64
    L.hs_encode_bound.argtypes = [C.c_int64, C.c_int64, C.c_int, C.c_int]
    L.hs_encode.restype = C.c_int
    L.hs_encode.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_int64,
                            C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_longlong)]
    L.hs_decode.restype = C.c_int
    L.hs_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_int64, C.c_int64,
                            C.c_void_p, C.c_int, C.POINTER(C.c_int)]
    L.hs_float_to_int.restype = C.c_int
    L.hs_float_to_int.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.hs_int_to_float.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    _LIB = L
    return L


_DT = {np.dtype(np.int32): 0, np.dtype(np.int64): 1, np.dtype(np.float32): 2, np.dtype(np.float64): 3}


def encode(arr, level=5, quanta=None):
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
    err = L.hs_encode(a2.ctypes.data, dt, n_stream, stream_size, level, None if q is None else q.ctypes.data,
                      out.ctypes.data, cap, starts.ctypes.data, nbytes.ctypes.data, offs.ctypes.data,
                      gains.ctypes.data, C.byref(tot))
    if err:
        raise RuntimeError(f"Encoding failed, return code = {err}")
    return out[:tot.value].copy(), starts, nbytes, offs, gains


def decode(compressed, starts, nbytes, stream_size, first=-1, last=-1, is_int64=False, mode=0):
    L = lib()
    # the throughput decoder reads whole 16-byte chunks: give the host buffer the slack every CUDA allocation has
    c = np.concatenate([np.ascontiguousarray(compressed, np.uint8), np.zeros(64, np.uint8)])
    st = np.ascontiguousarray(starts, np.int64).reshape(-1)
    nb = np.ascontiguousarray(nbytes, np.int64).reshape(-1)
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
