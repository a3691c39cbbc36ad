"""Drop-in replacement for the reference's compiled extension `flacarray.libflacarray`.

Same function names, argument meaning, return shapes/dtypes and error behaviour as
/root/reference/src/flacarray/libflacarray/libflacarray.pyx:113-823, but every array operation runs in
hand-written sm_100a CUDA kernels behind the C ABI of include/flacarray_b200.h (ctypes).  PyTorch is
used only to own device memory and CUDA streams.

Inputs may be numpy arrays (host; results come back as numpy, staged through pinned memory) or CUDA
torch tensors (device-resident; results stay on the device as torch tensors).  `use_threads` and the
`*_threaded` variants are accepted and ignored: the work is always parallel on the GPU.
There is no CPU path: without the built library or without a CUDA device these functions raise.
"""
import ctypes as C
import os
import threading

import numpy as np
import torch

from . import _lib

flac_i32_dtype = np.dtype(np.int32)
flac_i64_dtype = np.dtype(np.int64)
compressed_dtype = np.dtype(np.uint8)
offset_dtype = np.dtype(np.int64)

_NP2TORCH = {
    np.dtype(np.int32): torch.int32, np.dtype(np.int64): torch.int64, np.dtype(np.float32): torch.float32,
    np.dtype(np.float64): torch.float64, np.dtype(np.uint8): torch.uint8, np.dtype(np.bool_): torch.bool,
}
_TORCH2NP = {v: k for k, v in _NP2TORCH.items()}
_FAB = {np.dtype(np.int32): 0, np.dtype(np.int64): 1, np.dtype(np.float32): 2, np.dtype(np.float64): 3}


def is_torch(x):
    return isinstance(x, torch.Tensor)


def np_dtype(x):
    """numpy dtype of a numpy array or torch tensor."""
    if is_torch(x):
        return _TORCH2NP[x.dtype]
    return np.dtype(x.dtype)


def _is_contiguous(x):
    if is_torch(x):
        return x.is_contiguous()
    return x.flags.c_contiguous


def _device():
    if not torch.cuda.is_available():
        raise RuntimeError("flacarray_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def to_device(x, device=None, dtype=None):
    """numpy / torch (any device) -> contiguous CUDA tensor (async H2D when the source is pinned)."""
    if device is None:
        device = x.device if (is_torch(x) and x.is_cuda) else _device()
    if is_torch(x):
        t = x
    else:
        a = np.ascontiguousarray(x)
        if not a.flags.writeable:
            a = a.copy()
        t = torch.from_numpy(a)
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    if not t.is_cuda:
        t = t.to(device, non_blocking=True)
    return t.contiguous()


def to_host(t):
    """CUDA tensor -> numpy (through a pinned staging tensor that keeps the memory alive)."""
    if not t.is_cuda:
        return t.numpy()
    h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    h.copy_(t, non_blocking=True)
    torch.cuda.current_stream(t.device).synchronize()
    return h.numpy()


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _stream(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _check(rc, ctx, stream, what):
    """Collect the device-side error mask; raise like the reference binding (pyx:325-328, :649-652)."""
    if rc == 0:
        rc = _lib.lib().fab_finish(ctx.handle, stream)
    if rc != 0:
        if rc & (1 << 21):
            raise RuntimeError("Cannot convert data with NaNs to integers")
        msg = f"{what} failed, return code = {rc}"
        if rc & (1 << 20):
            msg += f" ({ctx.last_error()})"
        raise RuntimeError(msg)


# -------------------------------------------------------------------------------------------------
# float <-> int (pyx:113-282)
# -------------------------------------------------------------------------------------------------

def _float_to_int(flatdata, n_stream, stream_size, quanta, fdt, idt, check_nan=False):
    on_dev = is_torch(flatdata) and flatdata.is_cuda
    d = to_device(flatdata, dtype=_NP2TORCH[fdt])
    dev = d.device
    with torch.cuda.device(dev):
        ctx = _lib.context(dev)
        q = None
        if quanta is not None and len(quanta) == n_stream:  # pyx:142-144: wrong length => computed from the data
            q = to_device(quanta, dev, _NP2TORCH[fdt])
        out = torch.empty(n_stream * stream_size, dtype=_NP2TORCH[idt], device=dev)
        off = torch.empty(n_stream, dtype=_NP2TORCH[fdt], device=dev)
        gain = torch.empty(n_stream, dtype=_NP2TORCH[fdt], device=dev)
        st = _stream(dev)
        rc = _lib.lib().fab_float_to_int(ctx.handle, _ptr(d), _FAB[fdt], n_stream, stream_size, _ptr(q), _ptr(out),
                                         _ptr(off), _ptr(gain), st)
        if rc == 0:
            rc = _lib.lib().fab_finish(ctx.handle, st)
        if not check_nan:
            rc &= ~(1 << 21)  # the compiled converter does not look for NaNs (utils.py:268 does, before calling it)
        if rc != 0:
            _check(rc, ctx, st, "Encoding")
    if on_dev:
        return out, off, gain
    return to_host(out), to_host(off), to_host(gain)


def stream_std_device(d, n_stream, stream_size):
    """Population standard deviation of every stream of a CUDA tensor [n_stream * stream_size] (float32 /
    float64), as a CUDA tensor of the same dtype: the device side of `precision` -> quanta (reference
    utils.py:282-296, np.std(data, axis=-1)).  One read of the input, double-precision moments."""
    dev = d.device
    fdt = np.dtype(np.float32) if d.dtype == torch.float32 else np.dtype(np.float64)
    with torch.cuda.device(dev):
        ctx = _lib.context(dev)
        out = torch.empty(n_stream, dtype=d.dtype, device=dev)
        st = _stream(dev)
        rc = _lib.lib().fab_stream_std(ctx.handle, _ptr(d), _FAB[fdt], n_stream, stream_size, _ptr(out), st)
        if rc != 0:
            _check(rc, ctx, st, "Standard deviation")
    return out


def stream_std(data):
    """np.std(data, axis=-1) on the device.  CUDA tensors are reduced in place; host arrays are staged through
    the device in chunks of whole streams (pinned double buffers), which beats a single-core host pass for anything
    but small arrays.  Returns a numpy array with the leading shape of `data`."""
    dt = np_dtype(data)
    shape = tuple(data.shape)
    stream_size = shape[-1]
    lead = shape[:-1]
    n_stream = 1 if len(lead) == 0 else int(np.prod(lead))
    tdt = _NP2TORCH[dt]
    if is_torch(data) and data.is_cuda:
        d = data.reshape((-1,))
        if not d.is_contiguous():
            d = d.contiguous()
        return to_host(stream_std_device(d, n_stream, stream_size)).reshape(lead)
    dev = _device()
    src = _as_host_tensor(data.numpy() if is_torch(data) else data).view(n_stream, stream_size)
    ranges = _chunk_ranges(n_stream, stream_size * src.element_size())
    if len(ranges) == 1:
        d = src.to(dev, non_blocking=True)
        return to_host(stream_std_device(d.view(-1), n_stream, stream_size)).reshape(lead)
    with torch.cuda.device(dev):
        cur = torch.cuda.current_stream(dev)
        s_in, _ = _side_streams(dev)

        def prep(feed, i):
            a, b = ranges[i]
            dc = torch.empty((b - a, stream_size), dtype=tdt, device=dev)
            feed.copy(dc, src[a:b])
            e = torch.cuda.Event()
            e.record(s_in)
            return dc, e

        parts = []
        for (a, b), (dc, ev) in zip(ranges, _Feeder(dev, s_in, prep, len(ranges))):
            cur.wait_event(ev)
            dc.record_stream(cur)
            parts.append(stream_std_device(dc.view(-1), b - a, stream_size))
            del dc
        return to_host(torch.cat(parts)).reshape(lead)


def quanta_from_std(rms, precision):
    """rms / 10**precision, the reference's expression (utils.py:285-296) evaluated by numpy on the host so that the
    quanta are bit-identical to what the reference derives from the same standard deviations (a scalar precision
    keeps the storage type of the data, an array of precisions goes through float64; torch's division by a scalar
    multiplies by the reciprocal and is 1 ulp off).  `rms`: numpy array or torch tensor (n_stream values cross the bus)."""
    if is_torch(rms):
        rms = to_host(rms)
    try:
        len(precision)
    except TypeError:
        return rms / 10**precision
    return rms / 10 ** np.asarray(precision).reshape(rms.shape)


def wrap_float32_to_int32(flatdata, n_stream, stream_size, quanta, check_nan=False):
    """pyx:113-161.  Returns (int32 flat, offsets float32[n], gains float32[n])."""
    return _float_to_int(flatdata, n_stream, stream_size, quanta, np.dtype(np.float32), np.dtype(np.int32), check_nan)


def wrap_float64_to_int64(flatdata, n_stream, stream_size, quanta, check_nan=False):
    """pyx:164-212."""
    return _float_to_int(flatdata, n_stream, stream_size, quanta, np.dtype(np.float64), np.dtype(np.int64), check_nan)


def _int_to_float(idata, n_stream, stream_size, offsets, gains, idt, fdt):
    on_dev = is_torch(idata) and idata.is_cuda
    d = to_device(idata, dtype=_NP2TORCH[idt])
    dev = d.device
    with torch.cuda.device(dev):
        ctx = _lib.context(dev)
        off = to_device(offsets, dev, _NP2TORCH[fdt])
        gain = to_device(gains, dev, _NP2TORCH[fdt])
        out = torch.empty(n_stream * stream_size, dtype=_NP2TORCH[fdt], device=dev)
        st = _stream(dev)
        rc = _lib.lib().fab_int_to_float(ctx.handle, _ptr(d), _FAB[idt], n_stream, stream_size, _ptr(off), _ptr(gain),
                                         _ptr(out), st)
        _check(rc, ctx, st, "Decoding")
    return out if on_dev else to_host(out)


def wrap_int32_to_float32(idata, n_stream, stream_size, offsets, gains):
    """pyx:215-247."""
    return _int_to_float(idata, n_stream, stream_size, offsets, gains, np.dtype(np.int32), np.dtype(np.float32))


def wrap_int64_to_float64(idata, n_stream, stream_size, offsets, gains):
    """pyx:250-282."""
    return _int_to_float(idata, n_stream, stream_size, offsets, gains, np.dtype(np.int64), np.dtype(np.float64))


# -------------------------------------------------------------------------------------------------
# encode (pyx:285-594)
# -------------------------------------------------------------------------------------------------

_scratch_tls = threading.local()   # per thread (like the C contexts): two threads never share a scratch buffer


def _scratch_map():
    """device index -> grow-only worst-case output buffer of the device-resident encode (this thread's)."""
    m = getattr(_scratch_tls, "bufs", None)
    if m is None:
        m = _scratch_tls.bufs = {}
    return m



_GUESS_MIN_BYTES = 8 << 20        # smaller inputs always take the scratch + exact copy route
_PROBE_MIN_BYTES = 1 << 30        # first calls at least this large probe the ratio on a subset of streams
_PROBE_FRACTION = 64


def _ratio_history():
    """(device, dtype, level) -> compression ratios of this thread's last device-resident encodes."""
    m = getattr(_scratch_tls, "ratios", None)
    if m is None:
        m = _scratch_tls.ratios = {}
    return m


def _scratch_out(dev, nbytes):
    # one buffer per (device, CUDA stream): the exact-size copy handed back to the caller is queued on the stream
    # the encode ran on, so only work on that same stream may reuse the scratch
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    key = (idx, torch.cuda.current_stream(dev).cuda_stream)
    bufs = _scratch_map()
    buf = bufs.get(key)
    if buf is None or buf.numel() < nbytes:
        bufs[key] = None
        buf = None
        buf = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=dev)
        bufs[key] = buf
    return buf


def release_scratch():
    """Drop the per-device worst-case output buffers of the device-resident encode (they are as large as
    the largest array encoded so far and are otherwise kept for reuse; the calling thread's)."""
    _scratch_map().clear()


_ENC_OVERFLOW = 1 << 11        # ERROR_ENCODE_COLLECT: the frames did not fit the output buffer


def _encode_device_raw(d, n_stream, stream_size, level, quanta=None, scratch=False, capacity=None):
    """fab_encode into a worst-case device buffer (a fresh one, or the per-device scratch), or -- when
    `capacity` is given -- into a fresh buffer of that many bytes; in that case None is returned if the
    compressed data did not fit (the kernels stop at the capacity and flag it; nothing is written past it).
    Returns (buffer, starts, nbytes, total, offsets, gains)."""
    dev = d.device
    dt = _TORCH2NP[d.dtype]
    with torch.cuda.device(dev):
        ctx = _lib.context(dev)
        L = _lib.lib()
        if level < 0 or level > 8:
            raise RuntimeError("Encoding failed, return code = 2")
        bound = L.fab_encode_bound(n_stream, stream_size, _FAB[dt], level)
        if capacity is not None:
            bound = min(int(capacity), bound)
            out = torch.empty(max(bound, 1), dtype=torch.uint8, device=dev)
        else:
            out = _scratch_out(dev, bound) if scratch else torch.empty(max(bound, 1), dtype=torch.uint8, device=dev)
        aux = torch.empty(2 * n_stream + 1, dtype=torch.int64, device=dev)
        starts, nbytes, total = aux[:n_stream], aux[n_stream:2 * n_stream], aux[2 * n_stream:]
        off = gain = None
        if dt.kind == "f":
            off = torch.empty(n_stream, dtype=d.dtype, device=dev)
            gain = torch.empty(n_stream, dtype=d.dtype, device=dev)
        st = _stream(dev)
        rc = L.fab_encode(ctx.handle, _ptr(d), _FAB[dt], n_stream, stream_size, level, _ptr(quanta), _ptr(off),
                          _ptr(gain), _ptr(out), bound, _ptr(starts), _ptr(nbytes), _ptr(total), st)
        if rc == 0 and capacity is not None:
            rc = L.fab_finish(ctx.handle, st)
            if rc == _ENC_OVERFLOW:
                return None
        _check(rc, ctx, st, "Encoding")
        n_total = int(total.item())
    return out, starts, nbytes, n_total, off, gain


def encode_device(d, n_stream, stream_size, level, quanta=None):
    """Device-level encode.  d: CUDA tensor (int32/int64/float32/float64), flat or 2-D.

    Returns CUDA tensors (compressed u8[total], starts i64[n], nbytes i64[n], offsets, gains); offsets /
    gains are None for integer input.  For float input the quantisation (utils.c:160-328) is fused in
    front of the encoder; `quanta` is None (auto) or a CUDA tensor [n_stream].
    """
    # The encoder needs a worst-case (~ raw size) output buffer, but a device-resident FlacArray should hold
    # the compressed bytes only.  First call for a (device, dtype, level): encode into a per-device
    # worst-case scratch and hand back an exact-size copy (stream-ordered: the copy is queued before the
    # next encode can reuse the scratch).  Later calls: encode straight into a buffer sized from the largest
    # of the recent compression ratios + 4 % and return a view of it -- no 2nd pass over the output; if the
    # data compresses worse than that the kernels flag the overflow and the call falls back to the scratch.
    raw = n_stream * stream_size * d.element_size()
    key = (d.device.index, d.dtype, int(level))
    hist = _ratio_history().setdefault(key, [])
    if not hist and raw >= _PROBE_MIN_BYTES and n_stream >= 2 * _PROBE_FRACTION:
        # large first call: learn the ratio from 1/64 of the streams rather than holding a worst-case
        # buffer as large as the input (cfg4: 66 GB next to 66 GB of samples)
        n_probe = n_stream // _PROBE_FRACTION
        _, _, _, t_probe, _, _ = _encode_device_raw(d.reshape(-1)[:n_probe * stream_size], n_probe, stream_size, level,
                                                    None if quanta is None else quanta[:n_probe], scratch=True)
        hist.append(t_probe / (n_probe * stream_size * d.element_size()))
    if hist and raw >= _GUESS_MIN_BYTES:
        res = _encode_device_raw(d, n_stream, stream_size, level, quanta,
                                 capacity=int(raw * max(hist) * 1.04) + (1 << 16))
        if res is not None:
            out, starts, nbytes, n_total, off, gain = res
            hist.append(n_total / raw)
            del hist[:-4]
            return out[:n_total], starts, nbytes, off, gain
    out, starts, nbytes, n_total, off, gain = _encode_device_raw(d, n_stream, stream_size, level, quanta, scratch=True)
    hist.append(n_total / max(raw, 1))
    del hist[:-4]
    return out[:n_total].clone(), starts, nbytes, off, gain


# -------------------------------------------------------------------------------------------------
# Host-buffer pipelines: H2D of chunk i+1, the kernels of chunk i and D2H of chunk i-1 overlap on three
# CUDA streams (the PCIe link is full duplex).  Chunks are whole streams, so every chunk is an
# independent call of the device path; only byte offsets have to be rebased on the host.
# -------------------------------------------------------------------------------------------------
_PIPE_CHUNK_BYTES = 192 << 20     # raw bytes per chunk
_PIPE_MIN_BYTES = 64 << 20        # smaller arrays go in one shot
_side = {}


def _side_streams(dev):
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    if key not in _side:
        _side[key] = (torch.cuda.Stream(dev), torch.cuda.Stream(dev))
    return _side[key]


_NO_RAMP = os.environ.get("FLACARRAY_B200_NO_RAMP", "") == "1"      # measurement switch


def _chunk_ranges(n_stream, bytes_per_stream):
    """Whole-stream chunks of the host pipelines.  The copy-in of the first chunk and the kernels + copy-out of the last
    one are the only parts nothing overlaps, so the pipeline starts and ends with a quarter- and a half-size chunk."""
    total = n_stream * bytes_per_stream
    if n_stream < 2 or total < _PIPE_MIN_BYTES:
        return [(0, n_stream)]
    full = max(1, _PIPE_CHUNK_BYTES // max(bytes_per_stream, 1))
    ramp = [max(1, full // 4), max(1, full // 2)]
    if not _NO_RAMP and full >= 4 and n_stream >= 2 * sum(ramp) + full:
        mid = n_stream - 2 * sum(ramp)
        nmid = max(1, -(-mid // full))
        sizes = ramp + [(mid * (i + 1)) // nmid - (mid * i) // nmid for i in range(nmid)] + ramp[::-1]
    else:
        nchunk = min(n_stream, max(2, -(-total // _PIPE_CHUNK_BYTES)))
        sizes = [(n_stream * (i + 1)) // nchunk - (n_stream * i) // nchunk for i in range(nchunk)]
    out, a = [], 0
    for n in sizes:
        if n > 0:
            out.append((a, a + n))
            a += n
    assert a == n_stream
    return out


_STAGE_MIN_BYTES = 1 << 20        # pageable pieces below this go straight to cudaMemcpy
_NO_STAGE = os.environ.get("FLACARRAY_B200_NO_STAGE", "") == "1"     # measurement switch
_feed_pool = None


def _feeder_pool():
    global _feed_pool
    if _feed_pool is None:
        from concurrent.futures import ThreadPoolExecutor

        _feed_pool = ThreadPoolExecutor(max_workers=1, thread_name_prefix="flacarray-h2d")
    return _feed_pool


_copy_pool = None
_NO_COPY_POOL = os.environ.get("FLACARRAY_B200_NO_COPY_POOL", "") == "1"    # measurement switch


def _host_copy(dst, src):
    """CPU copy into pinned memory on several cores.  torch's own copy is multi-threaded when it has
    intra-op threads; launchers such as torchrun set OMP_NUM_THREADS=1, and then the slices are copied
    by a small pool instead (Tensor.copy_ drops the GIL)."""
    global _copy_pool
    n = dst.numel()
    if torch.get_num_threads() >= 4 or n * dst.element_size() < (32 << 20) or _NO_COPY_POOL:
        dst.copy_(src)
        return
    if _copy_pool is None:
        from concurrent.futures import ThreadPoolExecutor

        _copy_pool = ThreadPoolExecutor(max_workers=max(1, min(8, os.cpu_count() or 1)),
                                        thread_name_prefix="flacarray-copy")
    d1, s1 = dst.reshape(-1), src.reshape(-1)
    parts = _copy_pool._max_workers
    step = -(-n // parts)
    futs = [_copy_pool.submit(d1[i:i + step].copy_, s1[i:i + step]) for i in range(0, n, step)]
    for f in futs:
        f.result()


class _Feeder:
    """Host -> device copies on the input side stream, issued by one helper thread a few chunks ahead of
    the kernels.  Pinned sources are copied in place.  Pageable sources (the usual numpy array) are
    first copied into one of two pinned staging buffers with torch's multi-threaded CPU copy -- a plain
    cudaMemcpy from pageable memory runs at a fraction of the PCIe rate and blocks the caller -- so
    staging chunk i+1 overlaps the transfer and the kernels of chunk i."""

    def __init__(self, dev, s_in, prep, n_items, depth=2):
        self.dev, self.s_in, self.prep, self.n, self.depth = dev, s_in, prep, n_items, depth
        self.stage = [None, None]
        self.stage_ev = [None, None]
        self.k = 0

    def copy(self, dst, src):
        nbytes = src.numel() * src.element_size()
        if nbytes < _STAGE_MIN_BYTES or _NO_STAGE or src.is_pinned():
            dst.copy_(src, non_blocking=True)
            return
        k = self.k
        self.k ^= 1
        if self.stage_ev[k] is not None:
            self.stage_ev[k].synchronize()          # the previous transfer out of this buffer is done
        if self.stage[k] is None or self.stage[k].numel() < nbytes:
            self.stage[k] = None
            self.stage[k] = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
        st = self.stage[k][:nbytes].view(src.dtype).view(src.shape)
        _host_copy(st, src)
        dst.copy_(st, non_blocking=True)
        e = torch.cuda.Event()
        e.record(self.s_in)
        self.stage_ev[k] = e

    def _run(self, i):
        with torch.cuda.device(self.dev), torch.cuda.stream(self.s_in):
            return self.prep(self, i)

    def __iter__(self):
        pool = _feeder_pool()
        futs = []
        nxt = 0
        try:
            for i in range(self.n):
                while nxt < self.n and nxt <= i + self.depth:
                    futs.append(pool.submit(self._run, nxt))
                    nxt += 1
                yield futs[i].result()
                futs[i] = None
        finally:
            for f in futs:
                if f is not None and not f.cancel():
                    try:
                        f.result()
                    except Exception:  # noqa: BLE001 - the first error is already on its way up
                        pass


def _as_host_tensor(a):
    a = np.ascontiguousarray(a)
    if not a.flags.writeable:
        a = a.copy()
    return torch.from_numpy(a)


def _encode_host(flat, n_stream, stream_size, level, quanta, dt, precision=None):
    """numpy [n_stream * stream_size] -> (compressed u8 numpy, starts, nbytes, offsets, gains) (numpy).

    precision (scalar or one value per stream, float input only): the quanta of every chunk of streams are derived
    on the device from the chunk's standard deviations right before it is encoded, so the host array crosses the
    bus once."""
    dev = _device()
    tdt = _NP2TORCH[dt]
    src = _as_host_tensor(flat)
    if src.dtype != tdt:
        src = src.to(tdt)
    src = src.view(n_stream, stream_size)
    isz = src.element_size()
    ranges = _chunk_ranges(n_stream, stream_size * isz)
    q = None
    if quanta is not None:
        q = to_device(quanta, dev, tdt)
    def chunk_quanta(dc, a, b):
        if precision is None:
            return None if q is None else q[a:b]
        pr = precision
        try:
            len(precision)
            pr = np.asarray(precision).reshape(-1)[a:b]
        except TypeError:
            pass
        return to_device(np.asarray(quanta_from_std(stream_std_device(dc.view(-1), b - a, stream_size), pr)).astype(dt), dev, tdt)

    if len(ranges) == 1:
        d = src.to(dev, non_blocking=True)
        comp, starts, nbytes, off, gain = encode_device(d.view(-1), n_stream, stream_size, level, chunk_quanta(d, 0, n_stream))
        return (to_host(comp), to_host(starts), to_host(nbytes), None if off is None else to_host(off),
                None if gain is None else to_host(gain))
    with torch.cuda.device(dev):
        cur = torch.cuda.current_stream(dev)
        s_in, s_out = _side_streams(dev)

        def prep(feed, i):
            a, b = ranges[i]
            dc = torch.empty((b - a, stream_size), dtype=tdt, device=dev)   # owned by s_in's pool
            feed.copy(dc, src[a:b])
            e = torch.cuda.Event()
            e.record(s_in)
            return dc, e

        raw_total = n_stream * stream_size * isz
        bound = int(_lib.lib().fab_encode_bound(n_stream, stream_size, _FAB[dt], level))
        host = None
        cap = 0
        pos = 0
        parts = []
        for (a, b), (dc, ev) in zip(ranges, _Feeder(dev, s_in, prep, len(ranges))):
            cur.wait_event(ev)
            dc.record_stream(cur)
            out, starts, nbytes, tot, off, gain = _encode_device_raw(dc.view(-1), b - a, stream_size, level,
                                                                     chunk_quanta(dc, a, b))
            del dc                # input chunk can go back to the pool
            if host is None:
                # capacity from the first chunk's ratio (+3 %); a wrong guess grows the buffer below
                cap = min(int(tot / ((b - a) * stream_size * isz) * raw_total * 1.03) + (1 << 20), bound)
                host = torch.empty(cap, dtype=torch.uint8, pin_memory=True)
            if pos + tot > cap:
                # the guess was too small: move what has arrived into a buffer sized from the ratio seen so far for the
                # remaining streams (+10 %), never more than the worst case.  No device buffer is kept alive for this:
                # device memory stays bounded by the chunk pipeline whatever the size of the input
                s_out.synchronize()
                done = b * stream_size * isz
                cap = min(max(int((pos + tot) / done * raw_total * 1.10) + (1 << 20), pos + tot), bound)
                bigger = torch.empty(cap, dtype=torch.uint8, pin_memory=True)
                bigger[:pos].copy_(host[:pos])
                host = bigger
            e = torch.cuda.Event()
            e.record(cur)
            out.record_stream(s_out)
            s_out.wait_event(e)
            with torch.cuda.stream(s_out):
                host[pos:pos + tot].copy_(out[:tot], non_blocking=True)
            del out               # (record_stream keeps it valid until the copy has run)
            parts.append((starts + pos, nbytes, off, gain))
            pos += tot
        starts = to_host(torch.cat([p[0] for p in parts]))
        nbytes = to_host(torch.cat([p[1] for p in parts]))
        off = gain = None
        if parts[0][2] is not None:
            off = to_host(torch.cat([p[2] for p in parts]))
            gain = to_host(torch.cat([p[3] for p in parts]))
        s_out.synchronize()
    return host[:pos].numpy(), starts, nbytes, off, gain


def _decode_host(compressed, h_starts, h_nbytes, n_stream, stream_size, first_sample, last_sample, is_int64,
                 offsets=None, gains=None):
    """Host compressed bytes -> host samples (numpy, flat); optional int->float restore on the device."""
    dev = _device()
    n_decode = stream_size
    if first_sample >= 0 and last_sample >= 0:
        n_decode = last_sample - first_sample
    h_starts = np.asarray(h_starts, dtype=np.int64).reshape(-1)
    h_nbytes = np.asarray(h_nbytes, dtype=np.int64).reshape(-1)
    restore = offsets is not None and gains is not None
    if is_int64:
        odt = torch.float64 if restore else torch.int64
    else:
        odt = torch.float32 if restore else torch.int32
    isz = 8 if is_int64 else 4
    hint = blocksize_hint(compressed, h_starts)
    src = _as_host_tensor(compressed)
    ranges = _chunk_ranges(n_stream, max(n_decode, 1) * isz)
    h_ends = h_starts + h_nbytes
    with torch.cuda.device(dev):
        cur = torch.cuda.current_stream(dev)
        s_in, s_out = _side_streams(dev)
        fdt = torch.float64 if is_int64 else torch.float32
        d_off = to_device(np.asarray(offsets).reshape(-1), dev, fdt) if restore else None
        d_gain = to_device(np.asarray(gains).reshape(-1), dev, fdt) if restore else None
        out_host = torch.empty((n_stream, max(n_decode, 0)), dtype=odt, pin_memory=True)

        def prep(feed, i):
            a, b = ranges[i]
            # the byte range covering this chunk's streams (keep masks select sparse subsets)
            lo = int(h_starts[a:b].min())
            hi = int(h_ends[a:b].max())
            dc = torch.empty(max(hi - lo, 1), dtype=torch.uint8, device=dev)
            feed.copy(dc[:hi - lo], src[lo:hi])
            d_st = torch.from_numpy(h_starts[a:b] - lo).to(dev, non_blocking=True)
            d_nb = torch.from_numpy(np.ascontiguousarray(h_nbytes[a:b])).to(dev, non_blocking=True)
            e = torch.cuda.Event()
            e.record(s_in)
            return dc, d_st, d_nb, e, int(h_nbytes[a:b].max())

        for (a, b), (dc, d_st, d_nb, e, max_nb) in zip(ranges, _Feeder(dev, s_in, prep, len(ranges))):
            cur.wait_event(e)
            for t in (dc, d_st, d_nb):
                t.record_stream(cur)
            out = decode_device(dc, d_st, d_nb, b - a, int(stream_size), int(first_sample), int(last_sample), is_int64,
                                max_nb, hint, None if d_off is None else d_off[a:b], None if d_gain is None else d_gain[a:b])
            del dc, d_st, d_nb
            e2 = torch.cuda.Event()
            e2.record(cur)
            out.record_stream(s_out)
            s_out.wait_event(e2)
            with torch.cuda.stream(s_out):
                out_host[a:b].view(-1).copy_(out.view(odt), non_blocking=True)
        s_out.synchronize()
    return out_host.view(-1).numpy()


def _wrap_encode(flatdata, n_stream, stream_size, level, dt):
    on_dev = is_torch(flatdata) and flatdata.is_cuda
    if not on_dev:
        if is_torch(flatdata):
            flatdata = flatdata.numpy()
        comp, starts, nbytes, _, _ = _encode_host(flatdata, int(n_stream), int(stream_size), int(level), None, dt)
        return comp, starts, nbytes
    d = to_device(flatdata, dtype=_NP2TORCH[dt])
    comp, starts, nbytes, _, _ = encode_device(d, int(n_stream), int(stream_size), int(level))
    return comp, starts, nbytes


def wrap_encode_i32(flatdata, n_stream, stream_size, level):
    """pyx:285-343.  Returns (compressed bytes, flat starts, flat nbytes)."""
    return _wrap_encode(flatdata, n_stream, stream_size, level, flac_i32_dtype)


def wrap_encode_i32_threaded(flatdata, n_stream, stream_size, level):
    """pyx:346-404 (the GPU path is always parallel)."""
    return _wrap_encode(flatdata, n_stream, stream_size, level, flac_i32_dtype)


def wrap_encode_i64(flatdata, n_stream, stream_size, level):
    """pyx:407-465."""
    return _wrap_encode(flatdata, n_stream, stream_size, level, flac_i64_dtype)


def wrap_encode_i64_threaded(flatdata, n_stream, stream_size, level):
    """pyx:468-526."""
    return _wrap_encode(flatdata, n_stream, stream_size, level, flac_i64_dtype)


def encode_flac(data, level, use_threads=False):
    """Compress an integer array to a FLAC representation (pyx:529-594).

    Returns (compressed bytestream, stream starting bytes, stream nbytes); starts / nbytes have the
    leading shape of `data` (or (1,) for a single stream).
    """
    dt = np_dtype(data)
    if dt != flac_i32_dtype and dt != flac_i64_dtype:
        raise RuntimeError("Only 32bit or 64bit integer data is supported")
    if not _is_contiguous(data):
        raise RuntimeError("Only C-contiguous arrays are supported")
    if level < 0 or level > 8:
        raise RuntimeError("FLAC only supports compression levels 0-8")
    shape = tuple(data.shape)
    stream_size = shape[-1]
    if len(shape[:-1]) == 0:
        n_stream = 1
        starts_shape = (1,)
    else:
        n_stream = int(np.prod(shape[:-1]))
        starts_shape = shape[:-1]
    flatdata = data.reshape((-1,))
    if dt == flac_i32_dtype:
        compressed, flatstarts, flatnbytes = wrap_encode_i32(flatdata, n_stream, stream_size, level)
    else:
        compressed, flatstarts, flatnbytes = wrap_encode_i64(flatdata, n_stream, stream_size, level)
    return (compressed, flatstarts.reshape(starts_shape), flatnbytes.reshape(starts_shape))


# -------------------------------------------------------------------------------------------------
# decode (pyx:597-823)
# -------------------------------------------------------------------------------------------------

def blocksize_hint(compressed, starts):
    """Nominal FLAC blocksize from the first stream's STREAMINFO (sizes the device frame table)."""
    try:
        s0 = int(np.asarray(starts.cpu() if is_torch(starts) else starts).reshape(-1)[0])
        head = compressed[s0:s0 + 12]
        head = head.cpu().numpy() if is_torch(head) else np.asarray(head)
        if head.size >= 12 and bytes(head[:4]) == b"fLaC":
            return (int(head[8]) << 8) | int(head[9])
    except Exception:
        pass
    return 0


def decode_device(comp, starts, nbytes, n_stream, stream_size, first_sample, last_sample, is_int64, max_nbytes,
                  bs_hint, offsets=None, gains=None):
    """Device-level decode.  All arrays are CUDA tensors; returns a flat CUDA tensor.

    With offsets/gains the int->float restore (utils.c:330-368) is applied on the device.
    """
    dev = comp.device
    n_decode = stream_size
    if first_sample >= 0 and last_sample >= 0:
        n_decode = last_sample - first_sample
    with torch.cuda.device(dev):
        ctx = _lib.context(dev)
        out = torch.empty(n_stream * max(n_decode, 0), dtype=torch.int64 if is_int64 else torch.int32, device=dev)
        st = _stream(dev)
        rc = _lib.lib().fab_decode(ctx.handle, _ptr(comp), _ptr(starts), _ptr(nbytes), n_stream, stream_size,
                                   1 if is_int64 else 0, first_sample, last_sample, _ptr(out), _ptr(offsets),
                                   _ptr(gains), int(max_nbytes), int(bs_hint), st)
        _check(rc, ctx, st, "Decoding")
    if offsets is not None and gains is not None:
        out = out.view(torch.float64 if is_int64 else torch.float32)
    return out


def _check_sample_range(stream_size, first_sample, last_sample):
    """decompress.c:207-222 / pyx:769-777: the window [first, last) must lie inside the stream."""
    if first_sample >= 0 and last_sample >= 0:
        if last_sample > stream_size:
            raise RuntimeError("last_sample is beyond end of stream")
        if first_sample > stream_size - 1:
            raise RuntimeError("first_sample is beyond last element of stream")
        if first_sample >= last_sample:
            raise RuntimeError("first_sample is larger than last_sample")


def _check_byte_windows(h_starts, h_nbytes, n_compressed):
    """Every (start, nbytes) window must lie inside the compressed buffer: the kernels index it directly (a stale
    index array would otherwise turn into out-of-bounds device reads instead of an error)."""
    if h_starts.size == 0:
        return
    if h_starts.size != h_nbytes.size:
        raise RuntimeError("starts and nbytes should have the same number of elements")
    if int(h_starts.min()) < 0 or int(h_nbytes.min()) < 0 or int((h_starts + h_nbytes).max()) > int(n_compressed):
        raise RuntimeError("stream starts / nbytes point outside the compressed buffer")


def _wrap_decode(compressed, starts, nbytes, n_stream, stream_size, first_sample, last_sample, is_int64):
    on_dev = is_torch(compressed) and compressed.is_cuda
    h_starts = starts.cpu().numpy() if is_torch(starts) else np.asarray(starts)
    h_nbytes = nbytes.cpu().numpy() if is_torch(nbytes) else np.asarray(nbytes)
    _check_byte_windows(h_starts.reshape(-1), h_nbytes.reshape(-1), compressed.numel() if is_torch(compressed) else compressed.size)
    if not on_dev:
        if is_torch(compressed):
            compressed = compressed.numpy()
        return _decode_host(compressed, h_starts, h_nbytes, int(n_stream), int(stream_size), int(first_sample),
                            int(last_sample), is_int64)
    max_nb = int(h_nbytes.max()) if h_nbytes.size else 0
    hint = blocksize_hint(compressed, h_starts)
    d_starts = to_device(h_starts, compressed.device, torch.int64)
    d_nbytes = to_device(h_nbytes, compressed.device, torch.int64)
    return decode_device(compressed, d_starts, d_nbytes, int(n_stream), int(stream_size), int(first_sample),
                         int(last_sample), is_int64, max_nb, hint)


def wrap_decode_i32(compressed, starts, nbytes, n_stream, stream_size, first_sample, last_sample, use_threads):
    """pyx:597-653.  Returns the flat int32 array."""
    return _wrap_decode(compressed, starts, nbytes, n_stream, stream_size, first_sample, last_sample, False)


def wrap_decode_i64(compressed, starts, nbytes, n_stream, stream_size, first_sample, last_sample, use_threads):
    """pyx:655-711."""
    return _wrap_decode(compressed, starts, nbytes, n_stream, stream_size, first_sample, last_sample, True)


def decode_flac(compressed, starts, nbytes, stream_size, first_sample=-1, last_sample=-1, use_threads=False,
                is_int64=False):
    """Decompress a FLAC compressed bytestream (pyx:713-823)."""
    if np_dtype(compressed) != compressed_dtype:
        raise RuntimeError("Compressed data should be of type uint8")
    if not _is_contiguous(compressed):
        raise RuntimeError("Only C-contiguous arrays are supported")
    if np_dtype(starts) != offset_dtype:
        raise RuntimeError("starts data should be of type int64")
    if not _is_contiguous(starts):
        raise RuntimeError("Only C-contiguous arrays are supported")
    if np_dtype(nbytes) != offset_dtype:
        raise RuntimeError("nbytes data should be of type int64")
    if not _is_contiguous(nbytes):
        raise RuntimeError("Only C-contiguous arrays are supported")
    if stream_size <= 0:
        raise RuntimeError("You must specify the non-zero output stream size")
    if len(compressed.shape) != 1:
        raise RuntimeError("Compressed byte array should be one dimensional")

    n_decode = stream_size
    _check_sample_range(stream_size, first_sample, last_sample)
    if first_sample >= 0 and last_sample >= 0:
        n_decode = last_sample - first_sample

    output_shape = tuple(starts.shape) + (n_decode,)
    n_stream = int(np.prod(starts.shape))
    flat_starts = starts.reshape((-1,))
    flat_nbytes = nbytes.reshape((-1,))
    if is_int64:
        flat_output = wrap_decode_i64(compressed, flat_starts, flat_nbytes, n_stream, stream_size, first_sample,
                                      last_sample, use_threads)
    else:
        flat_output = wrap_decode_i32(compressed, flat_starts, flat_nbytes, n_stream, stream_size, first_sample,
                                      last_sample, use_threads)
    return flat_output.reshape(output_shape)


# -------------------------------------------------------------------------------------------------
# Fused entry points used by compress.py / decompress.py (no integer intermediate in host memory)
# -------------------------------------------------------------------------------------------------

def encode_flac_float(data, level, quanta, precision=None):
    """float32/float64 [..., stream_size] -> (compressed, starts, nbytes, offsets, gains).

    Equivalent to utils.float_to_int (utils.c:160-328) followed by encode_flac, with the quantisation
    fused into the encoder's frame load.  `quanta`: None (derive from the data range) or an array with
    one value per stream.  `precision` (instead of quanta; scalar or one value per stream): quanta =
    std(stream) / 10**precision (utils.py:282-296) with the standard deviation reduced on the device.
    """
    dt = np_dtype(data)
    shape = tuple(data.shape)
    stream_size = shape[-1]
    if len(shape[:-1]) == 0:
        n_stream, lead = 1, (1,)
    else:
        n_stream, lead = int(np.prod(shape[:-1])), shape[:-1]
    on_dev = is_torch(data) and data.is_cuda
    if quanta is not None:
        quanta = quanta.reshape((-1,))
        if (quanta.numel() if is_torch(quanta) else quanta.size) != n_stream:
            quanta = None
    if not on_dev:
        if is_torch(data):
            data = data.numpy()
        comp, starts, nbytes, off, gain = _encode_host(data.reshape((-1,)), n_stream, stream_size, int(level), quanta, dt,
                                                       precision=precision)
        return comp, starts.reshape(lead), nbytes.reshape(lead), off, gain
    d = to_device(data.reshape((-1,)), dtype=_NP2TORCH[dt])
    if precision is not None:
        quanta = np.asarray(quanta_from_std(stream_std_device(d, n_stream, stream_size), precision)).astype(dt).reshape(-1)
    q = None if quanta is None else to_device(quanta, d.device, _NP2TORCH[dt])
    comp, starts, nbytes, off, gain = encode_device(d, n_stream, stream_size, int(level), q)
    return comp, starts.reshape(lead), nbytes.reshape(lead), off, gain


def decode_flac_float(compressed, starts, nbytes, stream_size, offsets, gains, first_sample=-1, last_sample=-1,
                      is_int64=False):
    """decode_flac followed by utils.int_to_float (utils.c:330-368) without leaving the device."""
    n_decode = stream_size
    _check_sample_range(stream_size, first_sample, last_sample)
    if first_sample >= 0 and last_sample >= 0:
        n_decode = last_sample - first_sample
    output_shape = tuple(starts.shape) + (n_decode,)
    n_stream = int(np.prod(starts.shape))
    on_dev = is_torch(compressed) and compressed.is_cuda
    h_starts = (starts.cpu().numpy() if is_torch(starts) else np.asarray(starts)).reshape(-1)
    h_nbytes = (nbytes.cpu().numpy() if is_torch(nbytes) else np.asarray(nbytes)).reshape(-1)
    _check_byte_windows(h_starts, h_nbytes, compressed.numel() if is_torch(compressed) else compressed.size)
    if not on_dev:
        if is_torch(compressed):
            compressed = compressed.numpy()
        out = _decode_host(compressed, h_starts, h_nbytes, n_stream, int(stream_size), int(first_sample), int(last_sample),
                           is_int64, offsets, gains)
        return out.reshape(output_shape)
    max_nb = int(h_nbytes.max()) if h_nbytes.size else 0
    hint = blocksize_hint(compressed, h_starts)
    comp = compressed
    d_starts = to_device(h_starts, comp.device, torch.int64)
    d_nbytes = to_device(h_nbytes, comp.device, torch.int64)
    fdt = torch.float64 if is_int64 else torch.float32
    off = to_device(offsets.reshape((-1,)), comp.device, fdt)
    gain = to_device(gains.reshape((-1,)), comp.device, fdt)
    out = decode_device(comp, d_starts, d_nbytes, n_stream, int(stream_size), int(first_sample), int(last_sample),
                        is_int64, max_nb, hint, off, gain)
    return out.reshape(output_shape)


# -------------------------------------------------------------------------------------------------
# Per-stream sample windows (fab_decode_windows; no reference equivalent)
# -------------------------------------------------------------------------------------------------

def _window_records(n_stream, stream_size, streams, first, last):
    """Host validation of window records (flat stream indices, [first, last) each); returns three int64 arrays."""
    s = np.asarray(streams.cpu() if is_torch(streams) else streams)
    f = np.asarray(first.cpu() if is_torch(first) else first)
    l_ = np.asarray(last.cpu() if is_torch(last) else last)
    for name, a in (("streams", s), ("first", f), ("last", l_)):
        if a.size and not np.issubdtype(a.dtype, np.integer):
            raise RuntimeError(f"window {name} must be integers, not {a.dtype}")
    s = s.reshape(-1).astype(np.int64)
    f = f.reshape(-1).astype(np.int64) if f.ndim else np.full(s.size, int(f), np.int64)
    l_ = l_.reshape(-1).astype(np.int64) if l_.ndim else np.full(s.size, int(l_), np.int64)
    if not (s.size == f.size == l_.size):
        raise RuntimeError(f"streams, first and last must have the same length (got {s.size}, {f.size} and {l_.size})")
    if s.size:
        if int(s.min()) < 0 or int(s.max()) >= n_stream:
            bad = int(s[(s < 0) | (s >= n_stream)][0])
            raise RuntimeError(f"window stream index {bad} is out of range for {n_stream} streams")
        if int(f.min()) < 0 or int(l_.max()) > stream_size:
            i = int(np.nonzero((f < 0) | (l_ > stream_size))[0][0])
            raise RuntimeError(f"window {i} [{int(f[i])}, {int(l_[i])}) lies outside the stream of {stream_size} samples")
        if bool((f > l_).any()):
            i = int(np.nonzero(f > l_)[0][0])
            raise RuntimeError(f"window {i}: first sample {int(f[i])} is larger than last sample {int(l_[i])}")
    return s, f, l_


def decode_windows_device(comp, starts, nbytes, n_stream, stream_size, is_int64, win_stream, win_first, win_last, win_out,
                          out, max_nbytes, bs_hint, offsets=None, gains=None):
    """Device-level fab_decode_windows.  Every array is a CUDA tensor; `out` receives the windows at win_out."""
    dev = comp.device
    with torch.cuda.device(dev):
        ctx = _lib.context(dev)
        st = _stream(dev)
        rc = _lib.lib().fab_decode_windows(ctx.handle, _ptr(comp), _ptr(starts), _ptr(nbytes), n_stream, stream_size,
                                           1 if is_int64 else 0, _ptr(win_stream), _ptr(win_first), _ptr(win_last),
                                           _ptr(win_out), int(win_stream.numel()), _ptr(out), _ptr(offsets), _ptr(gains),
                                           int(max_nbytes), int(bs_hint), st)
        _check(rc, ctx, st, "Decoding")
    return out


def decode_windows(compressed, starts, nbytes, stream_size, streams, first, last, offsets=None, gains=None,
                   is_int64=False):
    """Decode window i = samples [first[i], last[i]) of stream streams[i] for every i in one call.

    streams: flat (C-order) indices into starts / nbytes; first / last: arrays or scalars broadcast against streams.
    Windows may be empty, overlap, repeat and come in any order.  With offsets and gains (one per stream) the samples
    are restored to float32 / float64.  Returns (data, woff): data is 1-D, window i is data[woff[i]:woff[i + 1]], and woff
    is a host int64 array of n + 1 entries.  data is a CUDA tensor when `compressed` is one (the decode stays on the
    device), else a numpy array.  Only the frames the windows touch are decoded, and every referenced stream is indexed
    once however many windows it has.
    """
    if np_dtype(compressed) != compressed_dtype:
        raise RuntimeError("Compressed data should be of type uint8")
    if len(compressed.shape) != 1 or not _is_contiguous(compressed):
        raise RuntimeError("Compressed byte array should be one dimensional and C-contiguous")
    if stream_size <= 0:
        raise RuntimeError("You must specify the non-zero output stream size")
    if (offsets is None) != (gains is None):
        raise RuntimeError("Offsets and gains must be given together")
    h_starts = (starts.cpu().numpy() if is_torch(starts) else np.asarray(starts)).reshape(-1).astype(np.int64)
    h_nbytes = (nbytes.cpu().numpy() if is_torch(nbytes) else np.asarray(nbytes)).reshape(-1).astype(np.int64)
    n_stream = h_starts.size
    _check_byte_windows(h_starts, h_nbytes, compressed.numel() if is_torch(compressed) else compressed.size)
    s, f, l_ = _window_records(n_stream, int(stream_size), streams, first, last)
    restore = offsets is not None
    woff = np.zeros(s.size + 1, np.int64)
    np.cumsum(l_ - f, out=woff[1:])
    total = int(woff[-1])
    if is_int64:
        odt = torch.float64 if restore else torch.int64
    else:
        odt = torch.float32 if restore else torch.int32
    idt = torch.int64 if is_int64 else torch.int32
    on_dev = is_torch(compressed) and compressed.is_cuda
    if s.size == 0:
        if on_dev:
            return torch.empty(0, dtype=odt, device=compressed.device), woff
        return np.zeros(0, dtype=_TORCH2NP[odt]), woff
    # the device only sees the referenced streams, each once
    uniq, inv = np.unique(s, return_inverse=True)
    inv = inv.reshape(-1).astype(np.int64)
    u_starts, u_nbytes = h_starts[uniq], h_nbytes[uniq]
    fdt = torch.float64 if is_int64 else torch.float32
    h_off = h_gain = None
    if restore:
        h_off = np.asarray(offsets.cpu() if is_torch(offsets) else offsets).reshape(-1)[uniq]
        h_gain = np.asarray(gains.cpu() if is_torch(gains) else gains).reshape(-1)[uniq]
    hint = blocksize_hint(compressed, u_starts)
    if on_dev:
        dev = compressed.device
        out = torch.empty(max(total, 1), dtype=idt, device=dev)
        d_off = to_device(h_off, dev, fdt) if restore else None
        d_gain = to_device(h_gain, dev, fdt) if restore else None
        decode_windows_device(compressed, to_device(u_starts, dev, torch.int64), to_device(u_nbytes, dev, torch.int64),
                              uniq.size, int(stream_size), is_int64, to_device(inv, dev, torch.int64),
                              to_device(f, dev, torch.int64), to_device(l_, dev, torch.int64),
                              to_device(woff[:-1], dev, torch.int64), out, int(u_nbytes.max()), hint, d_off, d_gain)
        return out[:total].view(odt), woff
    return _decode_windows_host(compressed, u_starts, u_nbytes, int(stream_size), inv, f, l_, woff, is_int64, hint, idt, odt,
                                h_off, h_gain), woff


def _decode_windows_host(compressed, u_starts, u_nbytes, stream_size, inv, f, l_, woff, is_int64, hint, idt, odt, h_off,
                         h_gain):
    """Host compressed bytes: the referenced streams' bytes go to the device in staged copies, in groups of streams
    (_chunk_ranges) when they exceed one chunk; every group decodes its windows into one packed device output."""
    if is_torch(compressed):
        compressed = compressed.numpy()
    dev = _device()
    total = int(woff[-1])
    n_u = u_starts.size
    restore = h_off is not None
    order = np.argsort(inv, kind="stable")          # windows grouped by stream slot
    bounds = np.searchsorted(inv[order], np.arange(n_u + 1))
    ranges = _chunk_ranges(n_u, max(1, int(u_nbytes.sum()) // n_u))
    src = _as_host_tensor(compressed)
    with torch.cuda.device(dev):
        cur = torch.cuda.current_stream(dev)
        s_in, _ = _side_streams(dev)
        fdt = torch.float64 if is_int64 else torch.float32
        out = torch.empty(max(total, 1), dtype=idt, device=dev)
        d_wout = to_device(woff[:-1], dev, torch.int64)

        def prep(feed, i):
            a, b = ranges[i]
            st, nb = u_starts[a:b], u_nbytes[a:b]
            lo, hi = int(st.min()), int((st + nb).max())
            if hi - lo == int(nb.sum()):                 # back to back (any order): one contiguous range
                part, rel = src[lo:hi], st - lo
            else:                                        # gather the streams' bytes into one buffer first
                rel = np.zeros(b - a, np.int64)
                np.cumsum(nb[:-1], out=rel[1:])
                part = torch.from_numpy(np.concatenate([compressed[int(x):int(x) + int(n)] for x, n in zip(st, nb)]))
            dc = torch.empty(max(part.numel(), 1), dtype=torch.uint8, device=dev)
            feed.copy(dc[:part.numel()], part)
            sel = order[bounds[a]:bounds[b]]
            dw = [torch.from_numpy(np.ascontiguousarray(x)).to(dev, non_blocking=True)
                  for x in (rel, nb, inv[sel] - a, f[sel], l_[sel], sel.astype(np.int64))]
            e = torch.cuda.Event()
            e.record(s_in)
            return dc, dw, e, int(nb.max())

        d_off = to_device(h_off, dev, fdt) if restore else None
        d_gain = to_device(h_gain, dev, fdt) if restore else None
        for (a, b), (dc, dw, e, max_nb) in zip(ranges, _Feeder(dev, s_in, prep, len(ranges))):
            cur.wait_event(e)
            for t in [dc] + dw:
                t.record_stream(cur)
            d_st, d_nb, d_ws, d_wf, d_wl, d_sel = dw
            d_wo = d_wout[d_sel]
            decode_windows_device(dc, d_st, d_nb, b - a, stream_size, is_int64, d_ws, d_wf, d_wl, d_wo, out, max_nb, hint,
                                  None if d_off is None else d_off[a:b], None if d_gain is None else d_gain[a:b])
            del dc, dw, d_st, d_nb, d_ws, d_wf, d_wl, d_sel, d_wo
        host = to_host(out[:total].view(odt))
    return host
