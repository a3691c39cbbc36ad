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
import collections
import ctypes as C
import math
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
        parts = []
        for a, b, dc in _staged(dev, ranges, _rows_prep(src, dev)):
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
    the kernels (_staged).  Pinned sources are copied in place.  Pageable sources (the usual numpy array) are
    first copied into one of two pinned staging buffers with torch's multi-threaded CPU copy -- a plain
    cudaMemcpy from pageable memory runs at a fraction of the PCIe rate and blocks the caller -- so
    staging chunk i+1 overlaps the transfer and the kernels of chunk i."""

    def __init__(self, s_in):
        self.s_in = s_in
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


def _staged(dev, ranges, prep):
    """The host -> device side of every host-buffer pipeline.  For each group of streams [a, b) in `ranges`, the helper
    thread runs prep(feed, a, b) on the input side stream, up to two groups ahead of the caller: prep issues the group's
    copies through feed.copy and returns what the group's kernels read.  Yields (a, b, *what prep returned) once the
    current stream is ordered after those copies.  No reference to a yielded group is kept here, so its device buffers
    go back to the caching allocator as soon as the caller drops them after queuing its kernels (record_stream keeps
    them valid until those kernels have run)."""
    cur = torch.cuda.current_stream(dev)
    s_in = _side_streams(dev)[0]
    feed = _Feeder(s_in)

    def run(a, b):
        with torch.cuda.device(dev), torch.cuda.stream(s_in):
            bufs = prep(feed, a, b)
            e = torch.cuda.Event()
            e.record(s_in)
        return e, bufs

    def take(fut):
        e, bufs = fut.result()
        cur.wait_event(e)
        for t in bufs:
            if is_torch(t):
                t.record_stream(cur)
        return bufs

    pool = _feeder_pool()
    futs = collections.deque()
    nxt = 0
    try:
        for i, (a, b) in enumerate(ranges):
            while nxt < len(ranges) and nxt <= i + 2:
                futs.append(pool.submit(run, *ranges[nxt]))
                nxt += 1
            yield (a, b, *take(futs.popleft()))
    finally:
        for f in futs:
            if not f.cancel():
                try:
                    f.result()
                except Exception:  # noqa: BLE001 - the first error is already on its way up
                    pass


def _as_host_tensor(a):
    a = np.ascontiguousarray(a)
    if not a.flags.writeable:
        a = a.copy()
    return torch.from_numpy(a)


def _rows_prep(src, dev):
    """_staged prep: rows [a, b) of a host tensor."""
    def prep(feed, a, b):
        dc = torch.empty((b - a,) + tuple(src.shape[1:]), dtype=src.dtype, device=dev)   # owned by s_in's pool
        feed.copy(dc, src[a:b])
        return (dc,)
    return prep


def _group_bytes(comp, starts, nbytes):
    """The host bytes that stage one group of streams, and the streams' starts rebased into them.  The covering range
    [min start, max end) is one plain copy; when it is more than twice the streams' own bytes (a sparse keep mask,
    windows over scattered streams) only the streams' bytes are gathered."""
    lo, hi = int(starts.min()), int((starts + nbytes).max())
    if hi - lo <= 2 * int(nbytes.sum()):
        return comp[lo:hi], starts - lo
    rel = np.zeros(starts.size, np.int64)
    np.cumsum(nbytes[:-1], out=rel[1:])
    return np.concatenate([comp[int(s):int(s) + int(n)] for s, n in zip(starts, nbytes)]), rel


def _bytes_prep(compressed, h_starts, h_nbytes, dev):
    """_staged prep: the bytes of streams [a, b) of a host compressed buffer -> (device bytes, the streams' starts in
    them, their nbytes, the largest of those nbytes)."""
    comp = _as_host_tensor(compressed.numpy() if is_torch(compressed) else compressed).numpy()

    def prep(feed, a, b):
        part, rel = _group_bytes(comp, h_starts[a:b], h_nbytes[a:b])
        dc = torch.empty(max(part.size, 1), dtype=torch.uint8, device=dev)
        feed.copy(dc[:part.size], torch.from_numpy(part))
        d_st = torch.from_numpy(rel).to(dev, non_blocking=True)
        d_nb = torch.from_numpy(np.ascontiguousarray(h_nbytes[a:b])).to(dev, non_blocking=True)
        return dc, d_st, d_nb, int(h_nbytes[a:b].max())
    return prep


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
        s_out = _side_streams(dev)[1]
        raw_total = n_stream * stream_size * isz
        bound = int(_lib.lib().fab_encode_bound(n_stream, stream_size, _FAB[dt], level))
        host = None
        cap = 0
        pos = 0
        parts = []
        for a, b, dc in _staged(dev, ranges, _rows_prep(src, dev)):
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
                  bs_hint, offsets=None, gains=None, status=None):
    """Device-level decode.  All arrays are CUDA tensors; returns a flat CUDA tensor.

    With offsets/gains the int->float restore (utils.c:330-368) is applied on the device.  With `status` (int32 CUDA
    tensor [n_stream]) the decode isolates failures per stream (fab_decode_isolated): each stream's error bits go to
    its status entry, failed rows are filled with 0 / NaN, and only call-level errors raise.
    """
    dev = comp.device
    n_decode = stream_size
    if first_sample >= 0 and last_sample >= 0:
        n_decode = last_sample - first_sample
    with torch.cuda.device(dev):
        ctx = _lib.context(dev)
        out = torch.empty(n_stream * max(n_decode, 0), dtype=torch.int64 if is_int64 else torch.int32, device=dev)
        st = _stream(dev)
        if status is None:
            rc = _lib.lib().fab_decode(ctx.handle, _ptr(comp), _ptr(starts), _ptr(nbytes), n_stream, stream_size,
                                       1 if is_int64 else 0, first_sample, last_sample, _ptr(out), _ptr(offsets),
                                       _ptr(gains), int(max_nbytes), int(bs_hint), st)
        else:
            rc = _lib.lib().fab_decode_isolated(ctx.handle, _ptr(comp), _ptr(starts), _ptr(nbytes), n_stream, stream_size,
                                                1 if is_int64 else 0, first_sample, last_sample, _ptr(out), _ptr(offsets),
                                                _ptr(gains), int(max_nbytes), int(bs_hint), _ptr(status), st)
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


def _stream_index(compressed, starts, nbytes):
    """The front door of every decode and verify: flat int64 host copies of starts and nbytes, checked against the
    compressed buffer, whether that buffer is on the device, and the blocksize hint of the call."""
    h_starts = np.asarray(starts.cpu().numpy() if is_torch(starts) else starts, dtype=np.int64).reshape(-1)
    h_nbytes = np.asarray(nbytes.cpu().numpy() if is_torch(nbytes) else nbytes, dtype=np.int64).reshape(-1)
    _check_byte_windows(h_starts, h_nbytes, compressed.numel() if is_torch(compressed) else compressed.size)
    return h_starts, h_nbytes, is_torch(compressed) and compressed.is_cuda, blocksize_hint(compressed, h_starts)


def _decode_groups(compressed, h_starts, h_nbytes, on_dev, hint, dev, ranges, stream_size, first_sample, last_sample,
                   is_int64, d_off=None, d_gain=None, status=None):
    """The per-group decode shared by every whole-stream decode: for each group of streams [a, b) in `ranges` yields
    (a, b, the group's flat CUDA output).  Device bytes are decoded in place; host bytes reach the device through
    _staged.  d_off / d_gain (restore) and status (per-stream isolation) are CUDA tensors over all n streams, and each
    group gets its slice.  A group's output goes back to the caching allocator when the caller drops it."""
    def part(t, a, b):
        return None if t is None else t[a:b]

    if on_dev:
        d_st, d_nb = to_device(h_starts, dev, torch.int64), to_device(h_nbytes, dev, torch.int64)
        for a, b in ranges:
            yield a, b, decode_device(compressed, d_st[a:b], d_nb[a:b], b - a, stream_size, first_sample, last_sample,
                                      is_int64, int(h_nbytes[a:b].max()) if b > a else 0, hint, part(d_off, a, b),
                                      part(d_gain, a, b), part(status, a, b))
        return
    for a, b, dc, d_st, d_nb, max_nb in _staged(dev, ranges, _bytes_prep(compressed, h_starts, h_nbytes, dev)):
        out = decode_device(dc, d_st, d_nb, b - a, stream_size, first_sample, last_sample, is_int64, max_nb, hint,
                            part(d_off, a, b), part(d_gain, a, b), part(status, a, b))
        del dc, d_st, d_nb
        yield a, b, out


def _decode(compressed, starts, nbytes, n_stream, stream_size, first_sample, last_sample, is_int64, offsets=None,
            gains=None, isolate=False):
    """Decode streams [0, n_stream) into one flat array: a CUDA tensor for device bytes; numpy for host bytes, which go
    to the device in groups of streams while the previous group's samples come back.  With offsets and gains the
    samples are restored to floats on the device.  Returns (flat, status): with `isolate` status is the int32 numpy
    per-stream status (each group fills its slice), else None."""
    h_starts, h_nbytes, on_dev, hint = _stream_index(compressed, starts, nbytes)
    dev = compressed.device if on_dev else _device()
    n_decode = last_sample - first_sample if (first_sample >= 0 and last_sample >= 0) else stream_size
    fdt = torch.float64 if is_int64 else torch.float32
    with torch.cuda.device(dev):
        status = _status_tensor(dev, n_stream) if isolate else None
        d_off = None if offsets is None else to_device(offsets, dev, fdt).reshape(-1)
        d_gain = None if gains is None else to_device(gains, dev, fdt).reshape(-1)
        if on_dev:
            # one group: the whole decode is one call and its output is the result
            (_, _, out), = _decode_groups(compressed, h_starts, h_nbytes, True, hint, dev, [(0, n_stream)], stream_size,
                                          first_sample, last_sample, is_int64, d_off, d_gain, status)
        else:
            odt = fdt if d_off is not None else (torch.int64 if is_int64 else torch.int32)
            out_host = torch.empty((n_stream, max(n_decode, 0)), dtype=odt, pin_memory=True)
            cur = torch.cuda.current_stream(dev)
            s_out = _side_streams(dev)[1]
            ranges = _chunk_ranges(n_stream, max(n_decode, 1) * (8 if is_int64 else 4))
            for a, b, out in _decode_groups(compressed, h_starts, h_nbytes, False, hint, dev, ranges, stream_size,
                                            first_sample, last_sample, is_int64, d_off, d_gain, status):
                e = torch.cuda.Event()
                e.record(cur)
                out.record_stream(s_out)
                s_out.wait_event(e)
                with torch.cuda.stream(s_out):
                    out_host[a:b].view(-1).copy_(out.view(odt), non_blocking=True)
            s_out.synchronize()
            out = out_host.view(-1).numpy()
    return out, None if status is None else to_host(status)


def wrap_decode_i32(compressed, starts, nbytes, n_stream, stream_size, first_sample, last_sample, use_threads):
    """pyx:597-653.  Returns the flat int32 array."""
    return _decode(compressed, starts, nbytes, int(n_stream), int(stream_size), int(first_sample), int(last_sample),
                   False)[0]


def wrap_decode_i64(compressed, starts, nbytes, n_stream, stream_size, first_sample, last_sample, use_threads):
    """pyx:655-711."""
    return _decode(compressed, starts, nbytes, int(n_stream), int(stream_size), int(first_sample), int(last_sample),
                   True)[0]


def check_on_error(on_error):
    """True for on_error="fill" (per-stream fault isolation), False for "raise"; anything else is a ValueError."""
    if isinstance(on_error, str) and on_error in ("raise", "fill"):
        return on_error == "fill"
    raise ValueError(f"on_error must be 'raise' or 'fill', not {on_error!r}")


def _status_tensor(dev, n_stream):
    """Device int32 [n_stream] for the per-stream status of an isolated decode or a verify."""
    return torch.empty(max(n_stream, 1), dtype=torch.int32, device=dev)[:n_stream]


def decode_flac(compressed, starts, nbytes, stream_size, first_sample=-1, last_sample=-1, use_threads=False,
                is_int64=False, on_error="raise"):
    """Decompress a FLAC compressed bytestream (pyx:713-823).

    on_error="fill": a stream that cannot be decoded does not fail the call; returns (array, status) where status
    (int32 numpy, shaped like starts) holds 0 or the stream's ERROR_DECODE_INIT / ERROR_DECODE_PROCESS bit and the rows
    of failed streams are 0.
    """
    isolate = check_on_error(on_error)
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

    lead = tuple(starts.shape)
    out, status = _decode(compressed, starts.reshape((-1,)), nbytes.reshape((-1,)), int(np.prod(lead)), int(stream_size),
                          int(first_sample), int(last_sample), is_int64, isolate=isolate)
    out = out.reshape(lead + (n_decode,))
    return (out, status.reshape(lead)) if isolate else out


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
                      is_int64=False, on_error="raise"):
    """decode_flac followed by utils.int_to_float (utils.c:330-368) without leaving the device.  on_error="fill" as in
    decode_flac, with the rows of failed streams set to NaN."""
    isolate = check_on_error(on_error)
    n_decode = stream_size
    _check_sample_range(stream_size, first_sample, last_sample)
    if first_sample >= 0 and last_sample >= 0:
        n_decode = last_sample - first_sample
    lead = tuple(starts.shape)
    out, status = _decode(compressed, starts, nbytes, int(np.prod(lead)), int(stream_size), int(first_sample),
                          int(last_sample), is_int64, offsets, gains, isolate)
    out = out.reshape(lead + (n_decode,))
    return (out, status.reshape(lead)) if isolate else out


# -------------------------------------------------------------------------------------------------
# Verify: decode and check every frame, store no samples (fab_verify; no reference equivalent)
# -------------------------------------------------------------------------------------------------

def verify_device(comp, starts, nbytes, n_stream, stream_size, is_int64, max_nbytes, bs_hint, status):
    """Device-level fab_verify: CUDA tensors in, `status` (int32 CUDA tensor [n_stream]) filled."""
    dev = comp.device
    with torch.cuda.device(dev):
        ctx = _lib.context(dev)
        st = _stream(dev)
        rc = _lib.lib().fab_verify(ctx.handle, _ptr(comp), _ptr(starts), _ptr(nbytes), n_stream, stream_size,
                                   1 if is_int64 else 0, int(max_nbytes), int(bs_hint), _ptr(status), st)
        _check(rc, ctx, st, "Verifying")
    return status


def verify_flac(compressed, starts, nbytes, stream_size, is_int64=False):
    """Decode and check every frame of every stream without storing samples.  Returns an int32 numpy array shaped like
    `starts`: 0, or the ERROR_DECODE_INIT / ERROR_DECODE_PROCESS bit of a stream that decoding would reject.  Host bytes
    go to the device in groups of streams; no samples come back."""
    if np_dtype(compressed) != compressed_dtype:
        raise RuntimeError("Compressed data should be of type uint8")
    if len(compressed.shape) != 1 or not _is_contiguous(compressed):
        raise RuntimeError("Compressed byte array should be one dimensional and C-contiguous")
    if stream_size <= 0:
        raise RuntimeError("You must specify the non-zero output stream size")
    shape = tuple(starts.shape)
    h_starts, h_nbytes, on_dev, hint = _stream_index(compressed, starts, nbytes)
    n_stream = h_starts.size
    if n_stream == 0:
        return np.zeros(shape, np.int32)
    dev = compressed.device if on_dev else _device()
    status = _status_tensor(dev, n_stream)
    if on_dev:
        verify_device(compressed, to_device(h_starts, dev, torch.int64), to_device(h_nbytes, dev, torch.int64), n_stream,
                      int(stream_size), is_int64, int(h_nbytes.max()), hint, status)
        return to_host(status).reshape(shape)
    ranges = _chunk_ranges(n_stream, max(1, int(h_nbytes.sum()) // n_stream))
    with torch.cuda.device(dev):
        for a, b, dc, d_st, d_nb, max_nb in _staged(dev, ranges, _bytes_prep(compressed, h_starts, h_nbytes, dev)):
            verify_device(dc, d_st, d_nb, b - a, int(stream_size), is_int64, max_nb, hint, status[a:b])
            del dc, d_st, d_nb
    return to_host(status).reshape(shape)


# -------------------------------------------------------------------------------------------------
# Statistics: count, min, max, mean and std per stream and bin, reduced from the decoded integers on the device
# (fab_row_stats; no reference equivalent)
# -------------------------------------------------------------------------------------------------
_STATS_GROUP_BYTES = 4 << 30      # decoded integers of one group of device-resident streams (see DESIGN.md section 6)
_MAX_BIN = (1 << 32) - 1          # a bin's exact sums are sized for at most this many samples

StreamStats = collections.namedtuple("StreamStats", ["count", "min", "max", "mean", "std"])


def check_bin(bin, n_decode):
    """The bin length of a stats call over n_decode samples: None is one bin of all of them, else an integer >= 1 (a bin
    longer than the range is one bin).  Raises ValueError for anything else and for bins of more than 2^32 - 1."""
    if bin is not None and (isinstance(bin, bool) or not isinstance(bin, (int, np.integer)) or int(bin) < 1):
        raise ValueError(f"bin must be None or an integer >= 1, not {bin!r}")
    length = n_decode if bin is None else min(int(bin), n_decode)
    if length > _MAX_BIN:
        raise ValueError(f"a bin of {length} samples is longer than the 2^32 - 1 samples a bin may hold")
    return length


def _stats_ranges(n_stream, row_bytes, cap):
    """Whole-stream groups of device-resident streams whose decoded rows take at most `cap` bytes (one stream at least)."""
    per = max(1, cap // max(row_bytes, 1))
    return [(a, min(a + per, n_stream)) for a in range(0, n_stream, per)]


def row_stats_device(rows, is_int64, n_rows, n, bin, offsets, gains, status, count, mn, mx, mean, std):
    """Device-level fab_row_stats over CUDA tensors; bin = 0 is one bin per row."""
    dev = rows.device
    with torch.cuda.device(dev):
        ctx = _lib.context(dev)
        st = _stream(dev)
        rc = _lib.lib().fab_row_stats(ctx.handle, _ptr(rows), 1 if is_int64 else 0, n_rows, n, bin, _ptr(offsets),
                                      _ptr(gains), _ptr(status), _ptr(count), _ptr(mn), _ptr(mx), _ptr(mean), _ptr(std), st)
        if rc != 0:
            _check(rc, ctx, st, "Statistics")


def stats_flac(compressed, starts, nbytes, stream_size, first_sample, last_sample, bin, offsets=None, gains=None,
               is_int64=False, isolate=False):
    """count, min, max, mean and std of samples [first_sample, last_sample) of every stream, per bin of `bin` samples
    (None: one bin), without storing the decoded array: groups of streams are decoded to integers on the device and
    reduced there by fab_row_stats; only the statistics come back.  Offsets and gains (both or neither) give the float
    statistics of the restored samples.  Returns (StreamStats of numpy arrays [n_stream, nbins], status): status is the
    int32 per-stream status with `isolate` (failed streams are filled), else None and a failed decode raises."""
    h_starts, h_nbytes, on_dev, hint = _stream_index(compressed, starts, nbytes)
    n_stream = h_starts.size
    n_decode = last_sample - first_sample
    length = check_bin(bin, n_decode)
    nbins = -(-n_decode // length)
    dev = compressed.device if on_dev else _device()
    fdt = torch.float64 if is_int64 else torch.float32
    restore = offsets is not None
    vdt = fdt if restore else (torch.int64 if is_int64 else torch.int32)
    vsz = 8 if is_int64 else 4
    m = n_stream * nbins
    with torch.cuda.device(dev):
        # every result in one device buffer, so that they come back in one copy
        res = torch.empty(24 * m + 2 * vsz * m + 4 * n_stream + 8, dtype=torch.uint8, device=dev)
        count = res[:8 * m].view(torch.int64)
        mean = res[8 * m:16 * m].view(torch.float64)
        std = res[16 * m:24 * m].view(torch.float64)
        mn = res[24 * m:24 * m + vsz * m].view(vdt)
        mx = res[24 * m + vsz * m:24 * m + 2 * vsz * m].view(vdt)
        status = res[24 * m + 2 * vsz * m:24 * m + 2 * vsz * m + 4 * n_stream].view(torch.int32) if isolate else None
        d_off = to_device(offsets, dev, fdt).reshape(-1) if restore else None
        d_gain = to_device(gains, dev, fdt).reshape(-1) if restore else None
        row_bytes = n_decode * vsz
        if on_dev:
            ranges = _stats_ranges(n_stream, row_bytes, _STATS_GROUP_BYTES)
        else:
            ranges = _chunk_ranges(n_stream, row_bytes)
        full = first_sample == 0 and last_sample == stream_size
        for a, b, rows in _decode_groups(compressed, h_starts, h_nbytes, on_dev, hint, dev, ranges, stream_size,
                                         -1 if full else first_sample, -1 if full else last_sample, is_int64,
                                         status=status):
            o0, o1 = a * nbins, b * nbins
            row_stats_device(rows, is_int64, b - a, n_decode, 0 if bin is None else length,
                             None if d_off is None else d_off[a:b], None if d_gain is None else d_gain[a:b],
                             None if status is None else status[a:b], count[o0:o1], mn[o0:o1], mx[o0:o1], mean[o0:o1],
                             std[o0:o1])
            del rows
        h = to_host(res)
    vnp = _TORCH2NP[vdt]
    out = StreamStats(h[:8 * m].view(np.int64), h[24 * m:24 * m + vsz * m].view(vnp),
                      h[24 * m + vsz * m:24 * m + 2 * vsz * m].view(vnp), h[8 * m:16 * m].view(np.float64),
                      h[16 * m:24 * m].view(np.float64))
    out = StreamStats(*(v.reshape(n_stream, nbins) for v in out))
    st = h[24 * m + 2 * vsz * m:24 * m + 2 * vsz * m + 4 * n_stream].view(np.int32) if isolate else None
    return out, st


# -------------------------------------------------------------------------------------------------
# Weighted sums across streams: per-sample sums of weighted streams per group, folded from the decoded integers on the
# device (fab_combine_rows; no reference equivalent)
# -------------------------------------------------------------------------------------------------

def check_combine_args(n_stream, weights, groups, n_groups):
    """The weights (float64, default 1), output row of every stream (int64, -1 = left out; None = all in row 0) and the
    number of output rows of a combine over n_stream streams, flat.  Raises ValueError for a size that is not n_stream,
    non-integer or boolean groups, a group below -1 or at least n_groups, and n_groups < 0."""
    def host(a):
        return a.cpu().numpy() if is_torch(a) else np.asarray(a)

    if weights is None:
        w = np.ones(n_stream)
    else:
        w = host(weights)
        if w.dtype == np.bool_ or w.dtype.kind not in "iuf":
            raise ValueError(f"weights must be real numbers, not {w.dtype}")
        w = w.astype(np.float64).reshape(-1)
        if w.size != n_stream:
            raise ValueError(f"weights has {w.size} entries for {n_stream} streams")
    if groups is None:
        if n_groups is not None:
            raise ValueError("n_groups needs groups")
        return w, np.zeros(n_stream, np.int64), 1
    g = host(groups)
    if g.dtype.kind not in "iu":
        raise ValueError(f"groups must be integers, not {g.dtype}")
    g = g.astype(np.int64).reshape(-1)
    if g.size != n_stream:
        raise ValueError(f"groups has {g.size} entries for {n_stream} streams")
    if n_groups is None:
        n_groups = int(g.max()) + 1 if g.size else 0
    elif isinstance(n_groups, bool) or not isinstance(n_groups, (int, np.integer)) or int(n_groups) < 0:
        raise ValueError(f"n_groups must be an integer >= 0, not {n_groups!r}")
    n_groups = int(n_groups)
    if g.size and (int(g.min()) < -1 or int(g.max()) >= n_groups):
        raise ValueError(f"groups must lie in [-1, {n_groups}), found [{int(g.min())}, {int(g.max())}]")
    return w, g, n_groups


def combine_device(rows, is_int64, n_rows, n, offsets, gains, status, weights, seg, seg_out, n_seg, out, n_out):
    """Device-level fab_combine_rows over CUDA tensors."""
    dev = rows.device
    with torch.cuda.device(dev):
        ctx = _lib.context(dev)
        st = _stream(dev)
        rc = _lib.lib().fab_combine_rows(ctx.handle, _ptr(rows), 1 if is_int64 else 0, n_rows, n, _ptr(offsets),
                                         _ptr(gains), _ptr(status), _ptr(weights), _ptr(seg), _ptr(seg_out), n_seg,
                                         _ptr(out), n_out, st)
        if rc != 0:
            _check(rc, ctx, st, "Combining")


def _segments(labels, ranges):
    """Segments of every decode group: consecutive rows of `labels` (sorted) with the same label.  Returns the
    concatenated row bounds (rebased to each group, n_seg + 1 per group), output rows, and each group's offsets into
    them."""
    bounds, outs, where = [], [], []
    nb = no = 0
    for a, b in ranges:
        lab = labels[a:b]
        cut = np.flatnonzero(lab[1:] != lab[:-1]) + 1
        bd = np.concatenate([[0], cut, [b - a]]).astype(np.int64)
        bounds.append(bd)
        outs.append(lab[bd[:-1]])
        where.append((nb, no, bd.size - 1))
        nb += bd.size
        no += bd.size - 1
    return np.concatenate(bounds), np.concatenate(outs).astype(np.int64), where


def combine_flac(compressed, starts, nbytes, stream_size, first_sample, last_sample, weights, groups, n_groups,
                 offsets=None, gains=None, is_int64=False, isolate=False):
    """Per-sample weighted sums of samples [first_sample, last_sample) over the streams of each group, without storing
    the decoded array: the streams with groups >= 0 are decoded to integers on the device in (group, storage index)
    order, group by group of streams, and fab_combine_rows folds each group's rows into its output row.  `weights`,
    `groups` and `n_groups` as check_combine_args returns them.  Returns (out [n_groups, n] float64: a CUDA tensor for
    device bytes, else numpy; status): status is the int32 numpy per-stream status with `isolate` (0 for streams left
    out), else None and a failed decode raises."""
    h_starts, h_nbytes, on_dev, hint = _stream_index(compressed, starts, nbytes)
    n_stream = h_starts.size
    n_decode = last_sample - first_sample
    sel = np.flatnonzero(groups >= 0)
    order = sel[np.argsort(groups[sel], kind="stable")]      # by group, storage order within a group
    m = order.size
    dev = compressed.device if on_dev else _device()
    fdt = torch.float64 if is_int64 else torch.float32
    restore = offsets is not None
    st_all = np.zeros(n_stream, np.int32) if isolate else None
    with torch.cuda.device(dev):
        out = torch.zeros((n_groups, n_decode), dtype=torch.float64, device=dev)
        if m and n_groups:
            row_bytes = n_decode * (8 if is_int64 else 4)
            if on_dev:
                ranges = _stats_ranges(m, row_bytes, _STATS_GROUP_BYTES)
            else:
                ranges = _chunk_ranges(m, row_bytes)
            labels = groups[order]
            bounds, outs, where = _segments(labels, ranges)
            d_w = to_device(weights[order], dev, torch.float64)
            d_bounds = to_device(bounds, dev, torch.int64)
            d_outs = to_device(outs, dev, torch.int64)
            d_off = to_device(np.asarray(offsets).reshape(-1)[order], dev, fdt) if restore else None
            d_gain = to_device(np.asarray(gains).reshape(-1)[order], dev, fdt) if restore else None
            status = _status_tensor(dev, m) if isolate else None
            full = first_sample == 0 and last_sample == stream_size
            for (a, b, rows), (nb, no, n_seg) in zip(
                    _decode_groups(compressed, h_starts[order], h_nbytes[order], on_dev, hint, dev, ranges, stream_size,
                                   -1 if full else first_sample, -1 if full else last_sample, is_int64, status=status),
                    where):
                combine_device(rows, is_int64, b - a, n_decode, None if d_off is None else d_off[a:b],
                               None if d_gain is None else d_gain[a:b], None if status is None else status[a:b],
                               d_w[a:b], d_bounds[nb:nb + n_seg + 1], d_outs[no:no + n_seg], n_seg, out, n_groups)
                del rows
            ctx = _lib.context(dev)
            _check(0, ctx, _stream(dev), "Combining")
            if isolate:
                st_all[order] = to_host(status)
        if not on_dev:
            out = to_host(out)
    return out, st_all


# -------------------------------------------------------------------------------------------------
# Projections onto templates: per-stream inner products with a few templates, folded from the decoded integers on the
# device (fab_project_rows; no reference equivalent)
# -------------------------------------------------------------------------------------------------
PROJECT_PIECE = 4096              # FAB_PROJECT_PIECE: samples per partial, part of the result's definition


def check_project_args(templates, n):
    """The number of templates and whether they came 1-D, for templates over n samples (numpy, array-like or any torch
    tensor; nothing is copied).  Raises ValueError for templates that are not real numbers or are boolean, are neither
    1-D nor 2-D, whose last axis is not n, or that hold no template."""
    if is_torch(templates):
        shape = tuple(templates.shape)
        real = not (templates.dtype == torch.bool or templates.is_complex())
        kind = str(templates.dtype)
    else:
        a = np.asarray(templates)
        shape = a.shape
        real = a.dtype.kind in "iuf"
        kind = str(a.dtype)
    if not real:
        raise ValueError(f"templates must be real numbers, not {kind}")
    if len(shape) not in (1, 2):
        raise ValueError(f"templates must be 1-D (n,) or 2-D (n_templates, n), not of shape {shape}")
    if shape[-1] != n:
        raise ValueError(f"templates have {shape[-1]} samples for a range of {n}")
    n_tmpl = 1 if len(shape) == 1 else shape[0]
    if n_tmpl == 0:
        raise ValueError("templates hold no template")
    return n_tmpl, len(shape) == 1


def _templates_on(templates, dev):
    """The templates as one contiguous float64 [n_tmpl, n] CUDA tensor on dev (one copy)."""
    if is_torch(templates):
        t = templates.to(device=dev, dtype=torch.float64)
    else:
        t = to_device(np.ascontiguousarray(templates, np.float64), dev, torch.float64)
    return t.reshape(-1, t.shape[-1]).contiguous()


def project_device(rows, is_int64, n_rows, n, offsets, gains, status, templates, n_tmpl, out):
    """Device-level fab_project_rows over CUDA tensors: out [n_rows, n_tmpl] float64."""
    dev = rows.device
    with torch.cuda.device(dev):
        ctx = _lib.context(dev)
        st = _stream(dev)
        rc = _lib.lib().fab_project_rows(ctx.handle, _ptr(rows), 1 if is_int64 else 0, n_rows, n, _ptr(offsets),
                                         _ptr(gains), _ptr(status), _ptr(templates), n_tmpl, _ptr(out), st)
        if rc != 0:
            _check(rc, ctx, st, "Projecting")


def project_flac(compressed, starts, nbytes, stream_size, first_sample, last_sample, templates, offsets=None,
                 gains=None, is_int64=False, isolate=False):
    """Inner products of samples [first_sample, last_sample) of every stream with every template, without storing the
    decoded array: groups of streams are decoded to integers on the device and fab_project_rows projects each group's
    rows.  `templates` as check_project_args accepts them, over last_sample - first_sample samples.  Returns (out
    [n_stream, n_tmpl] float64: a CUDA tensor for device bytes, else numpy; status): status is the int32 numpy
    per-stream status with `isolate` (failed streams: NaN), else None and a failed decode raises."""
    h_starts, h_nbytes, on_dev, hint = _stream_index(compressed, starts, nbytes)
    n_stream = h_starts.size
    n_decode = last_sample - first_sample
    dev = compressed.device if on_dev else _device()
    fdt = torch.float64 if is_int64 else torch.float32
    restore = offsets is not None
    with torch.cuda.device(dev):
        t = _templates_on(templates, dev)
        n_tmpl = t.shape[0]
        out = torch.empty((n_stream, n_tmpl), dtype=torch.float64, device=dev)
        status = _status_tensor(dev, n_stream) if isolate else None
        d_off = to_device(offsets, dev, fdt).reshape(-1) if restore else None
        d_gain = to_device(gains, dev, fdt).reshape(-1) if restore else None
        row_bytes = n_decode * (8 if is_int64 else 4)
        if on_dev:
            ranges = _stats_ranges(n_stream, row_bytes, _STATS_GROUP_BYTES)
        else:
            ranges = _chunk_ranges(n_stream, row_bytes)
        full = first_sample == 0 and last_sample == stream_size
        for a, b, rows in _decode_groups(compressed, h_starts, h_nbytes, on_dev, hint, dev, ranges, stream_size,
                                         -1 if full else first_sample, -1 if full else last_sample, is_int64,
                                         status=status):
            project_device(rows, is_int64, b - a, n_decode, None if d_off is None else d_off[a:b],
                           None if d_gain is None else d_gain[a:b], None if status is None else status[a:b], t, n_tmpl,
                           out[a:b])
            del rows
        st_h = to_host(status) if isolate else None
        if not on_dev:
            out = to_host(out)
    return out, st_h


# -------------------------------------------------------------------------------------------------
# Ranges of out-of-threshold samples: glitch and saturation intervals per stream, found in the decoded integers on the
# device (fab_flag_count / fab_flag_write; no reference equivalent)
# -------------------------------------------------------------------------------------------------
FlagRanges = collections.namedtuple("FlagRanges", ["stream", "first", "last", "nflagged"])

_I64_MIN, _I64_MAX = -(1 << 63), (1 << 63) - 1


def _threshold(t, n_stream, name):
    """A threshold as given: None, a Python int, or a flat numpy array (integer or float) of 1 or n_stream values.
    Raises ValueError for booleans, non-numbers, NaN and a size that is neither a scalar nor one per stream."""
    if t is None:
        return None
    if isinstance(t, (bool, np.bool_)):
        raise ValueError(f"{name} must be a number or one number per stream, not a boolean")
    if isinstance(t, int):
        return t                                   # exact, whatever its size
    a = t.cpu().numpy() if is_torch(t) else np.asarray(t)
    if a.dtype.kind not in "iuf":
        raise ValueError(f"{name} must be a number or one number per stream, not {a.dtype}")
    if a.ndim and a.size != n_stream:
        raise ValueError(f"{name} has {a.size} entries for {n_stream} streams")
    if a.dtype.kind == "f" and np.isnan(a).any():
        raise ValueError(f"{name} must not be NaN")
    return a.reshape(-1)


def _int_bounds(lo, hi, n_stream):
    """int64 [L, H] per stream for integer streams: x is flagged iff x < L or x > H (L > H: every sample).  Integers are
    used as they are; a float lo means x < ceil(lo) and a float hi x > floor(hi), in Python integers, so the rule holds
    at +-2^63."""
    def each(t, up):
        if t is None:
            return [_I64_MAX if up else _I64_MIN] * n_stream
        out = []
        for v in ([t] if isinstance(t, int) else t.tolist()):
            if isinstance(v, float) and math.isinf(v):
                v = _I64_MAX + 1 if v > 0 else _I64_MIN - 1     # beyond every int64 on that side
            elif isinstance(v, float):
                v = math.floor(v) if up else math.ceil(v)
            out.append(int(v))
        return out * n_stream if len(out) == 1 else out

    L, H = np.empty(n_stream, np.int64), np.empty(n_stream, np.int64)
    for k, (lv, hv) in enumerate(zip(each(lo, False), each(hi, True))):
        if lv > hv or lv > _I64_MAX or hv < _I64_MIN:
            lv, hv = 1, 0
        L[k], H[k] = max(lv, _I64_MIN), min(hv, _I64_MAX)
    return L, H


def check_flag_args(n_stream, lo, hi, pad, is_float):
    """The per-stream thresholds and the pad of a flag_ranges call over n_stream streams: float64 lo / hi (None: -inf /
    +inf) for float streams, int64 bounds [L, H] for integer streams (see _int_bounds), and pad as an int.  Raises
    ValueError when both thresholds are None, for NaN, boolean or non-numeric thresholds, a per-stream threshold of the
    wrong size, and a pad that is negative, boolean or not an integer."""
    if lo is None and hi is None:
        raise ValueError("flag_ranges needs lo, hi or both")
    lo, hi = _threshold(lo, n_stream, "lo"), _threshold(hi, n_stream, "hi")
    if isinstance(pad, (bool, np.bool_)) or not isinstance(pad, (int, np.integer)) or int(pad) < 0:
        raise ValueError(f"pad must be an integer >= 0, not {pad!r}")
    pad = int(pad)
    if not is_float:
        L, H = _int_bounds(lo, hi, n_stream)
        return L, H, pad

    def flt(t, inf):
        if t is None:
            return np.full(n_stream, inf)
        a = np.asarray(float(t) if isinstance(t, int) else t, np.float64).reshape(-1)
        return np.ascontiguousarray(np.broadcast_to(a, (n_stream,)))

    return flt(lo, -np.inf), flt(hi, np.inf), pad


def flag_count_device(rows, is_int64, n_rows, n, lo, hi, offsets, gains, status, pad, work, nflag, nrange):
    """Device-level fab_flag_count over CUDA tensors (work: the uint8 workspace)."""
    dev = rows.device
    with torch.cuda.device(dev):
        ctx = _lib.context(dev)
        st = _stream(dev)
        rc = _lib.lib().fab_flag_count(ctx.handle, _ptr(rows), 1 if is_int64 else 0, n_rows, n, _ptr(lo), _ptr(hi),
                                       _ptr(offsets), _ptr(gains), _ptr(status), pad, _ptr(work), work.numel(),
                                       _ptr(nflag), _ptr(nrange), st)
        if rc != 0:
            _check(rc, ctx, st, "Flagging")


def flag_write_device(rows, is_int64, n_rows, n, status, pad, work, base, sample0, first, last):
    """Device-level fab_flag_write over CUDA tensors, after flag_count_device on the same rows and workspace."""
    dev = rows.device
    with torch.cuda.device(dev):
        ctx = _lib.context(dev)
        st = _stream(dev)
        rc = _lib.lib().fab_flag_write(ctx.handle, _ptr(rows), 1 if is_int64 else 0, n_rows, n, _ptr(status), pad,
                                       _ptr(work), work.numel(), _ptr(base), sample0, _ptr(first), _ptr(last), st)
        if rc != 0:
            _check(rc, ctx, st, "Flagging")


def flag_ranges_flac(compressed, starts, nbytes, stream_size, first_sample, last_sample, lo, hi, pad, offsets=None,
                     gains=None, is_int64=False, isolate=False):
    """Ranges of out-of-threshold samples in [first_sample, last_sample) of every stream, without storing the decoded
    array: groups of streams are decoded to integers on the device, fab_flag_count counts each group's ranges, one copy
    of the counts sizes the group's output and fab_flag_write fills it.  The ranges stay on the device until one copy at
    the end.  lo, hi and pad as check_flag_args returns them (float thresholds with offsets and gains, integer bounds
    without).  Returns (stream, first, last, nflag, status) as numpy arrays, first / last as sample indices of the
    stream; status is the int32 per-stream status with `isolate` (failed streams: no ranges, nflag -1), else None and a
    failed decode raises."""
    h_starts, h_nbytes, on_dev, hint = _stream_index(compressed, starts, nbytes)
    n_stream = h_starts.size
    n_decode = last_sample - first_sample
    dev = compressed.device if on_dev else _device()
    fdt = torch.float64 if is_int64 else torch.float32
    restore = offsets is not None
    tdt = torch.float64 if restore else torch.int64
    with torch.cuda.device(dev):
        counts = torch.empty(2 * n_stream, dtype=torch.int64, device=dev)
        nflag, nrange = counts[:n_stream], counts[n_stream:]
        status = _status_tensor(dev, n_stream) if isolate else None
        d_lo, d_hi = to_device(lo, dev, tdt), to_device(hi, dev, tdt)
        d_off = to_device(offsets, dev, fdt).reshape(-1) if restore else None
        d_gain = to_device(gains, dev, fdt).reshape(-1) if restore else None
        row_bytes = n_decode * (8 if is_int64 else 4)
        if on_dev:
            ranges = _stats_ranges(n_stream, row_bytes, _STATS_GROUP_BYTES)
        else:
            ranges = _chunk_ranges(n_stream, row_bytes)
        ws = int(_lib.lib().fab_flag_ranges_workspace_bytes(max(b - a for a, b in ranges), n_decode,
                                                             1 if is_int64 else 0))
        work = torch.empty(ws, dtype=torch.uint8, device=dev)
        full = first_sample == 0 and last_sample == stream_size
        parts = []
        for a, b, rows in _decode_groups(compressed, h_starts, h_nbytes, on_dev, hint, dev, ranges, stream_size,
                                         -1 if full else first_sample, -1 if full else last_sample, is_int64,
                                         status=status):
            sa = None if status is None else status[a:b]
            flag_count_device(rows, is_int64, b - a, n_decode, d_lo[a:b], d_hi[a:b],
                              None if d_off is None else d_off[a:b], None if d_gain is None else d_gain[a:b], sa, pad,
                              work, nflag[a:b], nrange[a:b])
            nr = to_host(nrange[a:b])                  # sizes the group's output
            m = int(nr.sum())
            if m:
                base = to_device(np.concatenate([[0], np.cumsum(nr)[:-1]]).astype(np.int64), dev, torch.int64)
                out = torch.empty(2 * m, dtype=torch.int64, device=dev)
                flag_write_device(rows, is_int64, b - a, n_decode, sa, pad, work, base, first_sample, out[:m], out[m:])
                parts.append(out)
            del rows
        h = to_host(torch.cat([*parts, counts]))
        st_h = to_host(status) if isolate else None
    firsts, lasts, o = [], [], 0
    for t in parts:
        m = t.numel() // 2
        firsts.append(h[o:o + m])
        lasts.append(h[o + m:o + 2 * m])
        o += 2 * m
    nfl, nrg = h[o:o + n_stream], h[o + n_stream:o + 2 * n_stream]
    stream = np.repeat(np.arange(n_stream, dtype=np.int64), nrg)
    cat = (lambda v: np.concatenate(v) if v else np.zeros(0, np.int64))
    return stream, cat(firsts), cat(lasts), nfl.copy(), st_h


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
    h_starts, h_nbytes, on_dev, hint = _stream_index(compressed, starts, nbytes)
    n_stream = h_starts.size
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
    dev = _device()
    total = int(woff[-1])
    n_u = u_starts.size
    restore = h_off is not None
    order = np.argsort(inv, kind="stable")          # windows grouped by stream slot
    bounds = np.searchsorted(inv[order], np.arange(n_u + 1))
    ranges = _chunk_ranges(n_u, max(1, int(u_nbytes.sum()) // n_u))
    stream_bytes = _bytes_prep(compressed, u_starts, u_nbytes, dev)

    def prep(feed, a, b):
        sel = order[bounds[a]:bounds[b]]
        return stream_bytes(feed, a, b) + tuple(torch.from_numpy(np.ascontiguousarray(x)).to(dev, non_blocking=True)
                                                for x in (inv[sel] - a, f[sel], l_[sel], sel.astype(np.int64)))

    with torch.cuda.device(dev):
        fdt = torch.float64 if is_int64 else torch.float32
        out = torch.empty(max(total, 1), dtype=idt, device=dev)
        d_wout = to_device(woff[:-1], dev, torch.int64)
        d_off = to_device(h_off, dev, fdt) if restore else None
        d_gain = to_device(h_gain, dev, fdt) if restore else None
        for a, b, dc, d_st, d_nb, max_nb, d_ws, d_wf, d_wl, d_sel in _staged(dev, ranges, prep):
            decode_windows_device(dc, d_st, d_nb, b - a, stream_size, is_int64, d_ws, d_wf, d_wl, d_wout[d_sel], out,
                                  max_nb, hint, None if d_off is None else d_off[a:b],
                                  None if d_gain is None else d_gain[a:b])
            del dc, d_st, d_nb, d_ws, d_wf, d_wl, d_sel
        host = to_host(out[:total].view(odt))
    return host
