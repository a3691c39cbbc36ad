"""ctypes loader of the host emulation of the per-stream window decode (tests/hostsim/hostsim_windows.cpp).

TEST HARNESS ONLY, like hostsim.py (whose encoder the window tests use to make streams): runs the kernel bodies of
flacarray_b200/csrc the way fab_decode_windows drives them, on the CPU.  Never imported by the product package.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    so = os.path.join(_HERE, "libhostsim_windows.so")
    srcs = [os.path.join(_HERE, "hostsim_windows.cpp")] + [
        os.path.join(_HERE, "..", "..", "flacarray_b200", "csrc", f)
        for f in ("fa_simt.h", "fa_bits.h", "fa_quant.h", "fa_decode.h", "fa_decode_tile.h")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.run([cxx, "-O2", "-std=c++20", "-ffp-contract=off", "-fPIC", "-shared", "-pthread",
                        srcs[0], "-o", so], check=True, capture_output=True)
    L = C.CDLL(so)
    L.hs_decode_windows.restype = C.c_int
    L.hs_decode_windows.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.POINTER(C.c_int)]
    _LIB = L
    return L


def decode_windows(compressed, starts, nbytes, stream_size, streams, first, last, is_int64=False, bsh=4096):
    """Emulated fab_decode_windows with packed output.  Returns (flat data, window offsets, info) where window i is
    data[offsets[i]:offsets[i + 1]] and info = windows walked + 1000 * items left to the general decoder."""
    L = lib()
    # the throughput decoder reads whole 16-byte chunks: give the host buffer the slack every CUDA allocation has
    c = np.concatenate([np.ascontiguousarray(compressed, np.uint8), np.zeros(64, np.uint8)])
    st = np.ascontiguousarray(starts, np.int64).reshape(-1)
    nb = np.ascontiguousarray(nbytes, np.int64).reshape(-1)
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
