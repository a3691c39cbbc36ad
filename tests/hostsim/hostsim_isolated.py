"""ctypes loader of the host emulation of the isolated decode and of verify (tests/hostsim/hostsim_isolated.cpp).

TEST HARNESS ONLY, like hostsim.py: runs the kernel bodies of flacarray_b200/csrc the way fab_decode_isolated and
fab_verify drive them, on the CPU.  Never imported by the product package.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

ERROR_DECODE_INIT = 1 << 13
ERROR_DECODE_PROCESS = 1 << 14


def lib(prebuilt=None):
    """The emulator library, built next to this file when stale; `prebuilt`: load that build instead (e.g. one with
    sanitizers)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    so = prebuilt or os.path.join(_HERE, "libhostsim_isolated.so")
    srcs = [os.path.join(_HERE, "hostsim_isolated.cpp")] + [
        os.path.join(_HERE, "..", "..", "flacarray_b200", "csrc", f)
        for f in ("fa_simt.h", "fa_bits.h", "fa_quant.h", "fa_decode.h", "fa_decode_tile.h")]
    if prebuilt is None and (not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs)):
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.run([cxx, "-O2", "-std=c++20", "-ffp-contract=off", "-fPIC", "-shared", "-pthread",
                        srcs[0], "-o", so], check=True, capture_output=True)
    L = C.CDLL(so)
    L.hs_decode_isolated.restype = C.c_int
    L.hs_decode_isolated.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_int64,
                                     C.c_int64, C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_int)]
    _LIB = L
    return L


def _inputs(compressed, starts, nbytes):
    # the throughput decoder reads whole 16-byte chunks: give the host buffer the slack every CUDA allocation has
    c = np.concatenate([np.ascontiguousarray(compressed, np.uint8), np.zeros(64, np.uint8)])
    return c, np.ascontiguousarray(starts, np.int64).reshape(-1), np.ascontiguousarray(nbytes, np.int64).reshape(-1)


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
                               None if out is None else out.ctypes.data, 1 if store else 0, status.ctypes.data,
                               C.byref(info))
    if err:
        raise RuntimeError(f"Decoding failed, return code = {err}")
    if out is not None:
        out = out.reshape(n, nd * nch).view(np.int64) if is_int64 else out.reshape(n, nd)
    return out, status, info.value


def verify(compressed, starts, nbytes, stream_size, is_int64=False):
    """Emulated fab_verify: (status, info)."""
    _, status, info = decode_isolated(compressed, starts, nbytes, stream_size, is_int64=is_int64, store=False)
    return status, info
