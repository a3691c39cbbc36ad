"""The pure-Python reference the statistics of fab_row_stats are compared with bit for bit, and the wrappers of its host
emulation (hs_row_stats, hs_dbl_u256 in tests/hostsim/hostsim.cpp).

TEST HARNESS ONLY, like hostsim.py: runs the kernel bodies of flacarray_b200/csrc/fa_stats.h the way fab_row_stats drives
them, on the CPU.  Never imported by the product package.
"""
import ctypes as C
import math

import numpy as np

from hostsim import lib


def _ptr(a):
    return None if a is None else a.ctypes.data


def row_stats(rows, bin=None, offsets=None, gains=None, status=None, piece=0):
    """Emulated fab_row_stats on rows [n_rows, n] int32 / int64.  Returns ((count, min, max, mean, std) arrays
    [n_rows, nbins], pieces per bin)."""
    rows = np.ascontiguousarray(rows)
    is_int64 = rows.dtype == np.int64
    n_rows, n = rows.shape
    length = n if bin is None else min(int(bin), n)
    nbins = -(-n // length)
    restore = offsets is not None
    vdt = (np.float64 if is_int64 else np.float32) if restore else rows.dtype
    count = np.full((n_rows, nbins), -7, np.int64)
    mn = np.full((n_rows, nbins), 7, vdt)
    mx = np.full((n_rows, nbins), 7, vdt)
    mean = np.full((n_rows, nbins), 7.0)
    std = np.full((n_rows, nbins), 7.0)
    if restore:
        offsets = np.ascontiguousarray(offsets, vdt)
        gains = np.ascontiguousarray(gains, vdt)
    if status is not None:
        status = np.ascontiguousarray(status, np.int32)
    npc, ppb = C.c_int64(0), C.c_int64(0)
    rc = lib().hs_row_stats(rows.ctypes.data, 1 if is_int64 else 0, n_rows, n, 0 if bin is None else length, piece,
                            _ptr(offsets), _ptr(gains), _ptr(status), count.ctypes.data, mn.ctypes.data, mx.ctypes.data,
                            mean.ctypes.data, std.ctypes.data, C.byref(npc), C.byref(ppb))
    if rc:
        raise ValueError(f"fab_row_stats rejects these arguments (error {rc})")
    return (count, mn, mx, mean, std), ppb.value


def dbl_u256(v):
    """The emulated finisher's conversion of a non-negative integer < 2^256."""
    w = np.array([(v >> (64 * i)) & ((1 << 64) - 1) for i in range(4)], np.uint64)
    return lib().hs_dbl_u256(w.ctypes.data)


def restore_coeff(gain, is_int64):
    """fa_quant.h restore_coeff_f32 / _f64: 1 / gain in double, then the storage type."""
    g = float(gain)
    return float(np.float64(1.0 / g)) if is_int64 else float(np.float32(1.0 / g))


def restore(x, off, coeff, is_int64):
    """fa_quant.h restore_f32 / restore_f64 of one integer: off + coeff * x in the storage type, no FMA."""
    if is_int64:
        return np.float64(off) + np.float64(coeff) * np.float64(x)
    return np.float32(np.float32(off) + np.float32(np.float32(coeff) * np.float32(x)))


def reference(rows, bin=None, offsets=None, gains=None, status=None):
    """The statistics from Python integers and float(int): count, min, max, mean, std arrays [n_rows, nbins]."""
    rows = np.asarray(rows)
    is_int64 = rows.dtype == np.int64
    n_rows, n = rows.shape
    length = n if bin is None else min(int(bin), n)
    nbins = -(-n // length)
    restore_ = offsets is not None
    vdt = (np.float64 if is_int64 else np.float32) if restore_ else rows.dtype
    count = np.zeros((n_rows, nbins), np.int64)
    mn = np.zeros((n_rows, nbins), vdt)
    mx = np.zeros((n_rows, nbins), vdt)
    mean = np.zeros((n_rows, nbins))
    std = np.zeros((n_rows, nbins))
    for r in range(n_rows):
        if status is not None and status[r] != 0:
            count[r] = 0
            mean[r] = std[r] = np.nan
            mn[r] = mx[r] = np.nan if restore_ else 0
            continue
        vals = [int(v) for v in rows[r]]
        for b in range(nbins):
            seg = vals[b * length:(b + 1) * length]
            k = len(seg)
            s = sum(seg)
            q = sum(v * v for v in seg)
            mean_i = float(s) / float(k)
            std_i = math.sqrt(float(k * q - s * s)) / float(k)
            count[r, b] = k
            if not restore_:
                mn[r, b], mx[r, b] = min(seg), max(seg)
                mean[r, b], std[r, b] = mean_i, std_i
            else:
                off = float(offsets[r])
                coeff = restore_coeff(gains[r], is_int64)
                mean[r, b] = off + coeff * mean_i
                std[r, b] = abs(coeff) * std_i
                a, c = restore(min(seg), off, coeff, is_int64), restore(max(seg), off, coeff, is_int64)
                mn[r, b], mx[r, b] = min(a, c), max(a, c)
    return count, mn, mx, mean, std
