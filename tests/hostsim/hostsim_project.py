"""The numpy reference the projections of fab_project_rows are compared with bit for bit, and the wrapper of its host
emulation (hs_project_rows in tests/hostsim/hostsim_project.cpp: 32-row blocks, so that small arrays span several row
tiles).

TEST HARNESS ONLY, like hostsim.py: runs the kernel bodies of flacarray_b200/csrc/fa_project.h the way fab_project_rows
drives them, on the CPU.  Never imported by the product package.  hostsim_project.cpp is its own library, built with
hostsim.py's compiler and flags (hostsim.build builds hostsim.cpp only).
"""
import ctypes as C
import glob
import os
import subprocess

import numpy as np

import hostsim

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "hostsim_project.cpp")
_LIB = None
PIECE = 4096          # FAB_PROJECT_PIECE
THREADS = 32          # rows per emulated block


def build(path, flags=("-O2",)):
    """Compile the projection emulator library to `path` with the optimisation / instrumentation `flags`
    (hostsim.SANITIZE: an ASan + UBSan build to load in a process started with hostsim.sanitizer_env())."""
    subprocess.run([hostsim._CXX, *flags, "-std=c++20", "-ffp-contract=off", "-fPIC", "-shared", "-pthread", _SRC, "-o",
                    path], check=True, capture_output=True)


def lib(prebuilt=None):
    """The projection emulator library, built next to this file when older than its sources; `prebuilt`: load that
    build instead (e.g. one with sanitizers)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    so = prebuilt or os.path.join(_HERE, "libhostsim_project.so")
    deps = [_SRC] + glob.glob(os.path.join(_HERE, "..", "..", "flacarray_b200", "csrc", "*.h"))
    if prebuilt is None and (not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in deps)):
        tmp = f"{so}.{os.getpid()}.tmp"                 # test processes running side by side never load a partial file
        build(tmp)
        os.replace(tmp, so)
    L = C.CDLL(so)
    p, i64 = C.c_void_p, C.c_int64
    L.hs_project_rows.restype = C.c_int
    L.hs_project_rows.argtypes = [p, C.c_int, i64, i64, p, p, p, p, i64, p]
    _LIB = L
    return L


def _ptr(a):
    return None if a is None else a.ctypes.data


def project_rows(rows, templates, offsets=None, gains=None, status=None):
    """Emulated fab_project_rows on rows [n_rows, n] int32 / int64 (any element-aligned C-contiguous view) and templates
    [n_tmpl, n].  Returns out [n_rows, n_tmpl] float64; raises ValueError with the error bits of rejected arguments."""
    rows = np.asarray(rows)
    assert rows.ndim == 2 and rows.flags.c_contiguous
    is_int64 = rows.dtype == np.int64
    fdt = np.float64 if is_int64 else np.float32
    t = np.ascontiguousarray(templates, np.float64)
    t = t.reshape(1, -1) if t.ndim == 1 else t
    if offsets is not None:
        offsets = np.ascontiguousarray(offsets, fdt)
        gains = np.ascontiguousarray(gains, fdt)
    if status is not None:
        status = np.ascontiguousarray(status, np.int32)
    out = np.full((rows.shape[0], t.shape[0]), -7.0)
    rc = lib().hs_project_rows(rows.ctypes.data, 1 if is_int64 else 0, rows.shape[0], rows.shape[1], _ptr(offsets),
                               _ptr(gains), _ptr(status), t.ctypes.data, t.shape[0], out.ctypes.data)
    if rc:
        raise ValueError(f"fab_project_rows rejects these arguments ({rc})")
    return out


def reference(v, templates, ok=None):
    """The definition over values v [n_rows, n] (as to_array returns them; widened to float64 here) and templates
    [n_tmpl, n]: per piece of PIECE samples p = +0.0, p = p + T[t, i] * v[i] in ascending i, then out = +0.0, out = out +
    p in piece order, each multiply and add rounded on its own (numpy).  Zero padding to whole pieces changes no bit.
    Rows with ok False are NaN."""
    v = np.asarray(v).astype(np.float64)
    t = np.asarray(templates, np.float64)
    n_rows, n = v.shape
    n_tmpl = t.shape[0]
    npc = -(-n // PIECE)
    vp = np.zeros((n_rows, npc * PIECE))
    vp[:, :n] = v
    tp = np.zeros((n_tmpl, npc * PIECE))
    tp[:, :n] = t
    vp = vp.reshape(n_rows, npc, PIECE)
    tp = tp.reshape(n_tmpl, npc, PIECE)
    acc = np.zeros((n_rows, n_tmpl, npc))
    last = min(PIECE, n)             # beyond it every piece is padding only
    for i in range(last):
        acc = acc + tp[None, :, :, i] * vp[:, None, :, i]
    out = np.zeros((n_rows, n_tmpl))
    for j in range(npc):
        out = out + acc[:, :, j]
    if ok is not None:
        out[~np.asarray(ok, bool)] = np.nan
    return out
