"""Loader (and in-tree builder) of libflacarray_b200.so, the CUDA C-ABI library.

The product path has NO CPU fallback: if the shared library is missing, cannot be loaded, or no CUDA
device is usable, every call raises.  `build()` compiles the library in-tree with nvcc for sm_100a
(cross-compiles without a GPU); the resulting .so is git-ignored but ships to the GPU box.
"""
import ctypes as C
import os
import shutil
import subprocess
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("FLACARRAY_B200_SO") or os.path.join(_HERE, "libflacarray_b200.so")   # (override: kernel experiments)
_SOURCES = [os.path.join(_HERE, "csrc", f) for f in
            ("fa_api.cu", "fa_simt.h", "fa_bits.h", "fa_quant.h", "fa_encode.h", "fa_decode.h", "fa_decode_tile.h")]
_HEADER = os.path.join(os.path.dirname(_HERE), "include", "flacarray_b200.h")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-pthread", "-shared"]

_lib = None
_lock = threading.Lock()
_tls = threading.local()


def _nvcc():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    return None


def is_stale():
    if not os.path.exists(SO_PATH):
        return True
    t = os.path.getmtime(SO_PATH)
    return any(os.path.exists(s) and os.path.getmtime(s) > t for s in _SOURCES + [_HEADER])


def build(force=False, verbose=False):
    """Compile csrc/fa_api.cu -> libflacarray_b200.so for sm_100a.  Returns the path."""
    if not force and not is_stale():
        return SO_PATH
    nvcc = _nvcc()
    if nvcc is None:
        raise RuntimeError("nvcc not found: cannot build libflacarray_b200.so")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + [_SOURCES[0], "-o", SO_PATH]
    env = dict(os.environ)
    if os.path.exists("/usr/bin/g++"):
        cmd[1:1] = ["-ccbin", "/usr/bin/g++"]
    res = subprocess.run(cmd, capture_output=True, text=True, env=env)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return SO_PATH


_vp, _i64, _i32, _u32 = C.c_void_p, C.c_int64, C.c_int, C.c_uint32


def lib():
    """The loaded C-ABI library.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(SO_PATH):
            raise RuntimeError(
                f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(flacarray_b200 has no CPU fallback)")
        L = C.CDLL(SO_PATH)
        L.fab_create.restype = _i32
        L.fab_create.argtypes = [C.POINTER(_vp)]
        L.fab_destroy.argtypes = [_vp]
        L.fab_last_error.restype = C.c_char_p
        L.fab_last_error.argtypes = [_vp]
        L.fab_launch_count.restype = _i64
        L.fab_launch_count.argtypes = [_vp]
        L.fab_encode_bound.restype = _i64
        L.fab_encode_bound.argtypes = [_i64, _i64, _i32, _u32]
        L.fab_encode_workspace_bytes.restype = _i64
        L.fab_encode_workspace_bytes.argtypes = [_i64, _i64, _i32, _u32]
        L.fab_decode_workspace_bytes.restype = _i64
        L.fab_decode_workspace_bytes.argtypes = [_i64, _i64, _i32]
        L.fab_set_workspace.restype = _i32
        L.fab_set_workspace.argtypes = [_vp, _vp, _i64]
        L.fab_encode.restype = _i32
        L.fab_encode.argtypes = [_vp, _vp, _i32, _i64, _i64, _u32, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp]
        L.fab_decode.restype = _i32
        L.fab_decode.argtypes = [_vp, _vp, _vp, _vp, _i64, _i64, _i32, _i64, _i64, _vp, _vp, _vp, _i64, _i32, _vp]
        L.fab_decode_isolated.restype = _i32
        L.fab_decode_isolated.argtypes = [_vp, _vp, _vp, _vp, _i64, _i64, _i32, _i64, _i64, _vp, _vp, _vp, _i64, _i32, _vp, _vp]
        L.fab_verify.restype = _i32
        L.fab_verify.argtypes = [_vp, _vp, _vp, _vp, _i64, _i64, _i32, _i64, _i32, _vp, _vp]
        L.fab_decode_windows.restype = _i32
        L.fab_decode_windows.argtypes = [_vp, _vp, _vp, _vp, _i64, _i64, _i32, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _i64,
                                         _i32, _vp]
        L.fab_decode_windows_workspace_bytes.restype = _i64
        L.fab_decode_windows_workspace_bytes.argtypes = [_i64, _i64, _i64, _i64, _i32]
        L.fab_float_to_int.restype = _i32
        L.fab_float_to_int.argtypes = [_vp, _vp, _i32, _i64, _i64, _vp, _vp, _vp, _vp, _vp]
        L.fab_stream_std.restype = _i32
        L.fab_stream_std.argtypes = [_vp, _vp, _i32, _i64, _i64, _vp, _vp]
        L.fab_int_to_float.restype = _i32
        L.fab_int_to_float.argtypes = [_vp, _vp, _i32, _i64, _i64, _vp, _vp, _vp, _vp]
        L.fab_profile.argtypes = [_vp, _i32]
        L.fab_profile_ms.restype = C.c_double
        L.fab_profile_ms.argtypes = [_vp, _i32, C.POINTER(_i64)]
        L.fab_finish.restype = _i32
        L.fab_finish.argtypes = [_vp, _vp]
        _lib = L
    return _lib


# Every symbol include/flacarray_b200.h declares (checked by the CPU-side ABI test).
EXPORTED = [
    "encode_i32", "encode_i32_threaded", "encode_i64", "encode_i64_threaded", "decode_i32", "decode_i64",
    "float32_to_int32", "float64_to_int64", "int64_to_float64", "int32_to_float32",
    "fab_create", "fab_destroy", "fab_last_error", "fab_launch_count", "fab_encode_bound", "fab_encode",
    "fab_encode_workspace_bytes", "fab_decode_workspace_bytes", "fab_set_workspace",
    "fab_decode", "fab_decode_isolated", "fab_verify", "fab_decode_windows", "fab_decode_windows_workspace_bytes", "fab_stream_std", "fab_float_to_int", "fab_int_to_float", "fab_finish", "fab_profile", "fab_profile_ms",
]


class Context:
    """One fab_ctx per (thread, CUDA device)."""

    def __init__(self, device_index):
        import torch

        self.device_index = device_index
        self._h = _vp()
        with torch.cuda.device(device_index):
            rc = lib().fab_create(C.byref(self._h))
        if rc != 0 or not self._h:
            raise RuntimeError(f"flacarray_b200: cannot create a CUDA context on device {device_index} (code {rc})")

    @property
    def handle(self):
        return self._h

    def last_error(self):
        return lib().fab_last_error(self._h).decode()

    def launches(self):
        return int(lib().fab_launch_count(self._h))

    def set_workspace(self, tensor):
        """Hand the context a caller-owned device block (uint8 tensor, 256-byte aligned; None = back to the
        context-owned grow-only block).  With it no call allocates device memory: one that needs more fails."""
        ptr, n = (None, 0) if tensor is None else (tensor.data_ptr(), tensor.numel() * tensor.element_size())
        rc = lib().fab_set_workspace(self._h, ptr, n)
        if rc != 0:
            raise RuntimeError(f"fab_set_workspace failed (code {rc}): {self.last_error()}")
        self._ws = tensor      # keep the block alive as long as the context uses it

    def profile(self, enable):
        lib().fab_profile(self._h, 1 if enable else 0)

    def profile_ms(self, which):
        n = _i64(0)
        ms = lib().fab_profile_ms(self._h, which, C.byref(n))
        return float(ms), int(n.value)

    def __del__(self):
        try:
            if self._h:
                lib().fab_destroy(self._h)
                self._h = None
        except Exception:
            pass


def context(device=None):
    """Context for `device` (torch.device / index / None = current), cached per thread."""
    import torch

    if not torch.cuda.is_available():
        raise RuntimeError("flacarray_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    if device is None:
        idx = torch.cuda.current_device()
    elif isinstance(device, int):
        idx = device
    else:
        idx = device.index if device.index is not None else torch.cuda.current_device()
    cache = getattr(_tls, "ctx", None)
    if cache is None:
        cache = _tls.ctx = {}
    if idx not in cache:
        cache[idx] = Context(idx)
    return cache[idx]


def total_launches():
    cache = getattr(_tls, "ctx", None) or {}
    return sum(c.launches() for c in cache.values())
