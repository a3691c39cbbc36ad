"""ctypes loader of the host emulation of fab_combine_rows (tests/hostsim/hostsim_combine.cpp), and the numpy fold the
combined rows are compared with bit for bit.

TEST HARNESS ONLY, like hostsim.py: runs the kernel body of flacarray_b200/csrc/fa_combine.h the way fab_combine_rows
drives it, on the CPU.  Never imported by the product package.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
THREADS = 32          # threads per emulated block: a block covers THREADS * kCombineCols columns and tiles of THREADS rows
COLS = 2


def lib():
    """The emulator library, built next to this file when stale."""
    global _LIB
    if _LIB is not None:
        return _LIB
    so = os.path.join(_HERE, "libhostsim_combine.so")
    srcs = [os.path.join(_HERE, "hostsim_combine.cpp")] + [
        os.path.join(_HERE, "..", "..", "flacarray_b200", "csrc", f) for f in ("fa_simt.h", "fa_quant.h", "fa_combine.h")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.run([cxx, "-O2", "-std=c++20", "-ffp-contract=off", "-fPIC", "-shared", "-pthread", srcs[0], "-o", so],
                       check=True, capture_output=True)
    L = C.CDLL(so)
    L.hs_combine_rows.restype = C.c_int
    L.hs_combine_rows.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_int64] + [C.c_void_p] * 6 + [
        C.c_int64, C.c_void_p, C.c_int64, C.POINTER(C.c_int)]
    _LIB = L
    return L


def _ptr(a):
    return None if a is None else a.ctypes.data


def combine_rows(rows, weights, seg, seg_out, out, offsets=None, gains=None, status=None):
    """Emulated fab_combine_rows on rows [n_rows, n] int32 / int64, adding into `out` [n_out, n] float64 in place.
    Returns the error bits of the segment checks."""
    rows = np.asarray(rows)
    assert rows.ndim == 2 and rows.strides[1] == rows.itemsize and rows.strides[0] == rows.shape[1] * rows.itemsize
    assert out.dtype == np.float64 and out.flags.c_contiguous and out.shape[1] == rows.shape[1]
    is_int64 = rows.dtype == np.int64
    fdt = np.float64 if is_int64 else np.float32
    weights = np.ascontiguousarray(weights, np.float64)
    seg = np.ascontiguousarray(seg, np.int64)
    seg_out = np.ascontiguousarray(seg_out, np.int64)
    if offsets is not None:
        offsets = np.ascontiguousarray(offsets, fdt)
        gains = np.ascontiguousarray(gains, fdt)
    if status is not None:
        status = np.ascontiguousarray(status, np.int32)
    err = C.c_int(0)
    rc = lib().hs_combine_rows(rows.ctypes.data, 1 if is_int64 else 0, rows.shape[0], rows.shape[1], _ptr(offsets),
                               _ptr(gains), _ptr(status), weights.ctypes.data, seg.ctypes.data, seg_out.ctypes.data,
                               seg_out.size, out.ctypes.data, out.shape[0], C.byref(err))
    if rc:
        raise ValueError("fab_combine_rows rejects these arguments")
    return err.value


def fold(x, weights, groups, n_groups, ok=None):
    """The definition: for every group g, acc = +0.0, then acc = acc + w_k * float64(x_k) over the streams k of g in
    storage order (numpy multiplies and adds with separate rounding).  x: [n_stream, n] as to_array returns it."""
    x = np.asarray(x)
    out = np.zeros((n_groups, x.shape[-1]))
    for k in range(x.shape[0]):
        if groups[k] >= 0 and (ok is None or ok[k]):
            out[groups[k]] = out[groups[k]] + np.float64(weights[k]) * x[k].astype(np.float64)
    return out
