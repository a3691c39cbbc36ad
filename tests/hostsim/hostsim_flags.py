"""The pure-numpy reference the ranges of fab_flag_count / fab_flag_write are compared with exactly, and the wrappers of
their host emulation (hs_flag_ranges, hs_flag_bounds in tests/hostsim/hostsim_flags.cpp).

TEST HARNESS ONLY, like hostsim.py: runs the kernel bodies of flacarray_b200/csrc/fa_flags.h the way fab_flag_count and
fab_flag_write drive them, on the CPU.  Never imported by the product package.  hostsim_flags.cpp is its own library,
built with hostsim.py's compiler and flags (hostsim.build builds hostsim.cpp only).
"""
import ctypes as C
import glob
import os
import subprocess

import numpy as np

import hostsim

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "hostsim_flags.cpp")
_LIB = None


def build(path, flags=("-O2",)):
    """Compile the flag emulator library to `path` with the optimisation / instrumentation `flags` (hostsim.SANITIZE:
    an ASan + UBSan build to load in a process started with hostsim.sanitizer_env())."""
    subprocess.run([hostsim._CXX, *flags, "-std=c++20", "-ffp-contract=off", "-fPIC", "-shared", "-pthread", _SRC, "-o",
                    path], check=True, capture_output=True)


def _lib(prebuilt=None):
    """The flag emulator library, built next to this file when older than its sources; `prebuilt`: load that build
    instead (e.g. one with sanitizers)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    so = prebuilt or os.path.join(_HERE, "libhostsim_flags.so")
    deps = [_SRC] + glob.glob(os.path.join(_HERE, "..", "..", "flacarray_b200", "csrc", "*.h"))
    if prebuilt is None and (not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in deps)):
        tmp = f"{so}.{os.getpid()}.tmp"                 # test processes running side by side never load a partial file
        build(tmp)
        os.replace(tmp, so)
    L = C.CDLL(so)
    p, i64 = C.c_void_p, C.c_int64
    L.hs_flag_ranges.restype = C.c_int
    L.hs_flag_ranges.argtypes = [p, C.c_int, i64, i64, p, p, p, p, p, i64, i64, i64, p, p, p, p, i64, C.POINTER(i64)]
    L.hs_flag_bounds.restype = None
    L.hs_flag_bounds.argtypes = [C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.POINTER(C.c_longlong),
                                 C.POINTER(C.c_longlong)]
    _LIB = L
    return L


def _ptr(a):
    return None if a is None else a.ctypes.data


def flag_ranges(rows, lo, hi, pad=0, offsets=None, gains=None, status=None, piece=0, sample0=0):
    """Emulated fab_flag_count + fab_flag_write on rows [n_rows, n] int32 / int64.  lo / hi: one int64 bound per row
    (integer rows) or one float64 threshold per row (with offsets / gains).  Returns (stream, first, last, nflag,
    nrange) with the per-row counts of the count call; raises ValueError for arguments the C entry points reject."""
    if not rows.flags.c_contiguous:
        rows = np.ascontiguousarray(rows)
    is_int64 = rows.dtype == np.int64
    n_rows, n = rows.shape
    restore = offsets is not None
    if restore:
        fdt = np.float64 if is_int64 else np.float32
        offsets = np.ascontiguousarray(offsets, fdt)
        gains = np.ascontiguousarray(gains, fdt)
        lo = np.ascontiguousarray(np.broadcast_to(np.asarray(lo, np.float64), (n_rows,)))
        hi = np.ascontiguousarray(np.broadcast_to(np.asarray(hi, np.float64), (n_rows,)))
    else:
        lo = np.ascontiguousarray(np.broadcast_to(np.asarray(lo, np.int64), (n_rows,)))
        hi = np.ascontiguousarray(np.broadcast_to(np.asarray(hi, np.int64), (n_rows,)))
    if status is not None:
        status = np.ascontiguousarray(status, np.int32)
    cap = n_rows * (n // 2 + 1)
    nflag = np.full(n_rows, -7, np.int64)
    nrange = np.full(n_rows, -7, np.int64)
    first = np.full(cap + 1, -7, np.int64)
    last = np.full(cap + 1, -7, np.int64)
    total = C.c_int64(0)
    rc = _lib().hs_flag_ranges(rows.ctypes.data, 1 if is_int64 else 0, n_rows, n, lo.ctypes.data, hi.ctypes.data,
                               _ptr(offsets), _ptr(gains), _ptr(status), int(pad), int(piece), int(sample0),
                               nflag.ctypes.data, nrange.ctypes.data, first.ctypes.data, last.ctypes.data, cap,
                               C.byref(total))
    if rc:
        raise ValueError(f"fab_flag_count rejects these arguments (error {rc})")
    t = total.value
    assert np.all(first[t:] == -7) and np.all(last[t:] == -7), "a write outside the ranges' slots"
    stream = np.repeat(np.arange(n_rows, dtype=np.int64), np.maximum(nrange, 0))
    return stream, first[:t], last[:t], nflag, nrange


def flag_bounds(is_int64, off, coeff, lo, hi):
    """The emulated flag_bounds: (L, H) with L > H meaning every sample is flagged."""
    L, H = C.c_longlong(0), C.c_longlong(0)
    _lib().hs_flag_bounds(1 if is_int64 else 0, float(off), float(coeff), float(lo), float(hi), C.byref(L), C.byref(H))
    return L.value, H.value


def restore(x, off, coeff, is_int64):
    """fa_quant.h restore_f32 / restore_f64 of integers x (array), widened to float64: off + coeff * x in the storage
    type, no FMA."""
    x = np.asarray(x)
    if is_int64:
        return np.float64(off) + np.float64(coeff) * x.astype(np.float64)
    return (np.float32(off) + np.float32(coeff) * x.astype(np.float32)).astype(np.float32).astype(np.float64)


def flags_of(rows, lo, hi, offsets=None, coeffs=None):
    """Boolean flags [n_rows, n]: integer rows against int64 bounds (x < L or x > H), or the restored values (offsets and
    restore coefficients given) against float64 thresholds (v < lo or v > hi)."""
    rows = np.asarray(rows)
    n_rows = rows.shape[0]
    lo = np.broadcast_to(np.asarray(lo), (n_rows,))
    hi = np.broadcast_to(np.asarray(hi), (n_rows,))
    out = np.zeros(rows.shape, bool)
    for r in range(n_rows):
        if offsets is None:
            out[r] = (rows[r] < np.int64(lo[r])) | (rows[r] > np.int64(hi[r]))
        else:
            v = restore(rows[r], offsets[r], coeffs[r], rows.dtype == np.int64)
            out[r] = (v < float(lo[r])) | (v > float(hi[r]))
    return out


def reference(flags, pad, status=None, sample0=0):
    """Ranges of boolean flags [n_rows, n] from numpy: (stream, first, last, nflag) with nflag -1 and no ranges for rows
    with a non-zero status.  Python integers for pad, so any pad >= 0 works."""
    flags = np.asarray(flags, bool)
    n_rows, n = flags.shape
    p = min(int(pad), n)
    gap = min(2 * int(pad) + 1, n)
    stream, first, last, nflag = [], [], [], np.zeros(n_rows, np.int64)
    for r in range(n_rows):
        if status is not None and status[r] != 0:
            nflag[r] = -1
            continue
        idx = np.flatnonzero(flags[r])
        nflag[r] = idx.size
        if idx.size == 0:
            continue
        cut = np.flatnonzero(np.diff(idx) > gap)
        s = idx[np.concatenate([[0], cut + 1])]
        e = idx[np.concatenate([cut, [idx.size - 1]])]
        stream.append(np.full(s.size, r, np.int64))
        first.append(np.maximum(s - p, 0) + sample0)
        last.append(np.minimum(e + p + 1, n) + sample0)
    cat = (lambda a: np.concatenate(a).astype(np.int64) if a else np.zeros(0, np.int64))
    return cat(stream), cat(first), cat(last), nflag
