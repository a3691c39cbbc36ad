"""array_decompress / array_decompress_slice: same contract as
/root/reference/src/flacarray/decompress.py:18-205 (keep mask, sample window, single-stream
flattening rules, error messages); array_decompress_windows: many per-stream sample windows in one decode.
The FLAC decode and the int->float restore run on the device."""
import numpy as np

from .libflacarray import decode_flac, decode_flac_float, decode_windows, is_torch
from .utils import ensure_one_element, function_timer, keep_select, select_keep_indices


def _host(x):
    return x.cpu().numpy() if is_torch(x) else x


def _result_dtype(is_int64, restored):
    if restored:
        return np.float64 if is_int64 else np.float32
    return np.int64 if is_int64 else np.int32


@function_timer
def array_decompress_slice(
    compressed,
    stream_size,
    stream_starts,
    stream_nbytes,
    stream_offsets=None,
    stream_gains=None,
    keep=None,
    first_stream_sample=None,
    last_stream_sample=None,
    is_int64=False,
    use_threads=False,
    no_flatten=False,
):
    """Decompress a window of selected streams and restore the original data type.

    Contract of the reference's decompress.py:18-141: `keep` (boolean mask shaped like stream_starts) selects the
    streams, [first_stream_sample, last_stream_sample) the samples (None = whole stream); offsets and gains -- both
    or neither -- turn the integers back into floats.  A single stream may be described by scalars or 1-element
    arrays and then comes back flattened unless `no_flatten`.  Returns (array, indices): `indices` lists the index
    tuples of the kept streams in storage order, or is None without `keep`.
    """
    if (stream_offsets is None) != (stream_gains is None):
        which = "gains" if stream_gains is None else "offsets"
        given = "offsets" if stream_gains is None else "gains"
        raise RuntimeError(f"When specifying {given}, you must also provide the {which}")
    restored = stream_offsets is not None
    first = -1 if first_stream_sample is None else first_stream_sample
    last = -1 if last_stream_sample is None else last_stream_sample

    # one stream given as scalars / 1-element arrays: promote, remember to flatten the result
    single = not (isinstance(stream_starts, np.ndarray) or is_torch(stream_starts)) or tuple(stream_starts.shape) == (1,)
    if single:
        fdt = np.float64 if is_int64 else np.float32
        stream_starts = ensure_one_element(stream_starts, np.int64)
        stream_nbytes = ensure_one_element(stream_nbytes, np.int64)
        if restored:
            stream_offsets = ensure_one_element(stream_offsets, fdt)
            stream_gains = ensure_one_element(stream_gains, fdt)

    starts, nbytes, indices = keep_select(keep, _host(stream_starts), _host(stream_nbytes))
    offsets = select_keep_indices(None if not restored else _host(stream_offsets), indices)
    gains = select_keep_indices(None if not restored else _host(stream_gains), indices)

    if starts.size == 0:
        # an all-False mask: the reference hands back an empty (0, n) array
        n = last - first if (first >= 0 and last >= 0) else stream_size
        arr = np.zeros(tuple(starts.shape) + (n,), dtype=_result_dtype(is_int64, restored))
    elif restored:
        arr = decode_flac_float(compressed, starts, nbytes, stream_size, offsets, gains, first_sample=first,
                                last_sample=last, is_int64=is_int64)
    else:
        arr = decode_flac(compressed, starts, nbytes, stream_size, first_sample=first, last_sample=last,
                          use_threads=use_threads, is_int64=is_int64)
    if single and not no_flatten:
        arr = arr.reshape((-1,))
    return arr, indices


@function_timer
def array_decompress(
    compressed,
    stream_size,
    stream_starts,
    stream_nbytes,
    stream_offsets=None,
    stream_gains=None,
    first_stream_sample=None,
    last_stream_sample=None,
    is_int64=False,
    use_threads=False,
    no_flatten=False,
):
    """Decompress a FLAC encoded array and restore the original data type."""
    arr, _ = array_decompress_slice(
        compressed,
        stream_size,
        stream_starts,
        stream_nbytes,
        stream_offsets=stream_offsets,
        stream_gains=stream_gains,
        keep=None,
        first_stream_sample=first_stream_sample,
        last_stream_sample=last_stream_sample,
        is_int64=is_int64,
        use_threads=use_threads,
        no_flatten=no_flatten,
    )
    return arr


@function_timer
def array_decompress_windows(
    compressed,
    stream_size,
    stream_starts,
    stream_nbytes,
    streams,
    first,
    last,
    stream_offsets=None,
    stream_gains=None,
    is_int64=False,
):
    """Decompress many sample windows, each of its own stream, in one call.

    Window i is samples [first[i], last[i]) of the stream with flat C-order index streams[i] into stream_starts;
    `first` and `last` may be scalars (broadcast against `streams`).  Windows may be empty, overlap, repeat and come in
    any order.  Offsets and gains -- both or neither -- restore the floats as array_decompress does.  Only the frames
    the windows touch are decoded.

    Returns (data, offsets): `data` is 1-D in the restored dtype (a CUDA tensor when `compressed` is one, else numpy)
    and `offsets` an int64 numpy array of shape (n + 1,); window i is data[offsets[i]:offsets[i + 1]].
    """
    if (stream_offsets is None) != (stream_gains is None):
        which = "gains" if stream_gains is None else "offsets"
        given = "offsets" if stream_gains is None else "gains"
        raise RuntimeError(f"When specifying {given}, you must also provide the {which}")
    if not (isinstance(stream_starts, np.ndarray) or is_torch(stream_starts)):
        stream_starts = ensure_one_element(stream_starts, np.int64)
        stream_nbytes = ensure_one_element(stream_nbytes, np.int64)
        if stream_offsets is not None:
            fdt = np.float64 if is_int64 else np.float32
            stream_offsets = ensure_one_element(stream_offsets, fdt)
            stream_gains = ensure_one_element(stream_gains, fdt)
    return decode_windows(compressed, stream_starts, stream_nbytes, stream_size, streams, first, last,
                          offsets=stream_offsets, gains=stream_gains, is_int64=is_int64)
