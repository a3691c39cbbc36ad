"""array_decompress / array_decompress_slice: same contract as
/root/reference/src/flacarray/decompress.py:18-205 (keep mask, sample window, single-stream
flattening rules, error messages), plus on_error="fill" (per-stream fault isolation);
array_decompress_windows: many per-stream sample windows in one decode; array_verify: check streams without
decoding them out; array_stats: per-stream and per-bin statistics without decoding the array out; array_combine:
per-sample weighted sums across streams without decoding the array out; array_flag_ranges: per-stream ranges of samples
outside thresholds without decoding the array out; array_project: per-stream projections onto templates without decoding
the array out.  The FLAC decode, the int->float restore, the statistics, the sums, the range search and the projections
run on the device."""
import numpy as np

from .libflacarray import (FlagRanges, StreamStats, check_bin, check_combine_args, check_flag_args, check_on_error,
                           check_project_args, combine_flac, decode_flac, decode_flac_float, decode_windows,
                           flag_ranges_flac, is_torch, project_flac, stats_flac, verify_flac)
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
    on_error="raise",
):
    """Decompress a window of selected streams and restore the original data type.

    Contract of the reference's decompress.py:18-141: `keep` (boolean mask shaped like stream_starts) selects the
    streams, [first_stream_sample, last_stream_sample) the samples (None = whole stream); offsets and gains -- both
    or neither -- turn the integers back into floats.  A single stream may be described by scalars or 1-element
    arrays and then comes back flattened unless `no_flatten`.  Returns (array, indices): `indices` lists the index
    tuples of the kept streams in storage order, or is None without `keep`.

    on_error: "raise" (default) fails the whole call when any stream cannot be decoded.  "fill" decodes every stream it
    can and returns (array, indices, status): status is an int32 numpy array of array.shape[:-1] ((1,) for a flattened
    single stream), in the same row order, holding 0 or the stream's ERROR_DECODE_INIT (1 << 13) / ERROR_DECODE_PROCESS
    (1 << 14) bit; the rows of failed streams are 0 (integers) or NaN (floats).  Call-level errors still raise.
    """
    isolate = check_on_error(on_error)
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
        if isolate:
            arr = (arr, np.zeros(tuple(starts.shape), np.int32))
    elif restored:
        arr = decode_flac_float(compressed, starts, nbytes, stream_size, offsets, gains, first_sample=first,
                                last_sample=last, is_int64=is_int64, on_error=on_error)
    else:
        arr = decode_flac(compressed, starts, nbytes, stream_size, first_sample=first, last_sample=last,
                          use_threads=use_threads, is_int64=is_int64, on_error=on_error)
    status = None
    if isolate:
        arr, status = arr
    if single and not no_flatten:
        arr = arr.reshape((-1,))
    if isolate:
        return arr, indices, status
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
    on_error="raise",
):
    """Decompress a FLAC encoded array and restore the original data type.

    on_error="fill" returns (array, status) instead of failing on a damaged stream (see array_decompress_slice)."""
    res = array_decompress_slice(
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
        on_error=on_error,
    )
    if check_on_error(on_error):
        return res[0], res[2]
    return res[0]


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


@function_timer
def array_verify(compressed, stream_size, stream_starts, stream_nbytes, is_int64=False):
    """Check every stream without decoding it out: every frame is decoded and checked (CRC-8 / CRC-16, syntax, frame
    chain, sample count) exactly as a full decode would, and no samples are stored or copied back.

    Returns an int32 numpy array shaped like stream_starts ((1,) for a single stream given as scalars): 0 for a stream a
    full decode accepts, else its ERROR_DECODE_INIT (1 << 13) / ERROR_DECODE_PROCESS (1 << 14) bit.  Host-resident bytes
    are copied to the device in groups of streams.
    """
    if not (isinstance(stream_starts, np.ndarray) or is_torch(stream_starts)):
        stream_starts = ensure_one_element(stream_starts, np.int64)
        stream_nbytes = ensure_one_element(stream_nbytes, np.int64)
    return verify_flac(compressed, stream_starts, stream_nbytes, stream_size, is_int64=is_int64)


def stats_slice(compressed, stream_size, stream_starts, stream_nbytes, stream_offsets=None, stream_gains=None, keep=None,
                first_stream_sample=None, last_stream_sample=None, bin=None, is_int64=False, no_flatten=False,
                on_error="raise"):
    """array_stats with the index tuples of the kept streams and FlacArray's flattening rule: returns (StreamStats,
    indices, status), status None unless on_error="fill"."""
    isolate = check_on_error(on_error)
    if (stream_offsets is None) != (stream_gains is None):
        raise RuntimeError("Offsets and gains must be given together")
    restored = stream_offsets is not None
    first = 0 if first_stream_sample is None else int(first_stream_sample)
    last = int(stream_size) if last_stream_sample is None else int(last_stream_sample)
    if first < 0 or last > stream_size:
        raise ValueError(f"sample range [{first}, {last}) lies outside the stream of {stream_size} samples")
    if last <= first:
        raise ValueError(f"sample range [{first}, {last}) is empty")
    length = check_bin(bin, last - first)
    nbins = -(-(last - first) // length)

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
    lead = tuple(starts.shape)
    tail = () if bin is None else (nbins,)
    if starts.size == 0:
        vdt = _result_dtype(is_int64, restored)
        z = lead + tail
        stats = StreamStats(np.zeros(z, np.int64), np.zeros(z, vdt), np.zeros(z, vdt), np.zeros(z), np.zeros(z))
        status = np.zeros(lead, np.int32)
    else:
        stats, status = stats_flac(compressed, starts, nbytes, stream_size, first, last, bin, offsets, gains, is_int64,
                                   isolate)
        stats = StreamStats(*(v.reshape(lead + tail) for v in stats))
        status = None if status is None else status.reshape(lead)
    if single and not no_flatten:
        stats = StreamStats(*(v.reshape(tail) for v in stats))
    return stats, indices, (status if isolate else None)


@function_timer
def array_stats(
    compressed,
    stream_size,
    stream_starts,
    stream_nbytes,
    stream_offsets=None,
    stream_gains=None,
    keep=None,
    first_stream_sample=None,
    last_stream_sample=None,
    bin=None,
    is_int64=False,
    on_error="raise",
):
    """Per-stream and per-bin statistics of the decompressed samples without materialising them.

    Streams and samples are selected as in array_decompress_slice (`keep`, [first_stream_sample, last_stream_sample),
    offsets and gains both or neither).  `bin`: None for one bin over the whole sample range, or an integer B >= 1 that
    cuts the range into ceil(n / B) bins of B samples (the last one may be shorter); a bin may hold at most 2^32 - 1
    samples.  Returns StreamStats(count, min, max, mean, std): each array has the shape array_decompress_slice's result
    would have with the sample axis replaced by the bin axis (dropped when bin is None).  count is int64, min / max are
    in the array's dtype and equal to the decoded samples' min / max, mean and std (population, ddof = 0) are float64:
    the sums are exact integers, then mean = S / n and std = sqrt(n*Q - S^2) / n are each rounded once, and floats go
    through the restore's offset and coefficient.

    Compressed bytes on the device are decoded there in groups of streams; host bytes are copied to the device in
    groups.  Only the statistics come back.  on_error="fill" returns (stats, status) as array_decompress does: a stream
    that cannot be decoded gets count 0, NaN mean / std and NaN (floats) or 0 (integers) min / max.
    """
    stats, _, status = stats_slice(compressed, stream_size, stream_starts, stream_nbytes, stream_offsets=stream_offsets,
                                   stream_gains=stream_gains, keep=keep, first_stream_sample=first_stream_sample,
                                   last_stream_sample=last_stream_sample, bin=bin, is_int64=is_int64, on_error=on_error)
    return (stats, status) if status is not None else stats


@function_timer
def array_combine(
    compressed,
    stream_size,
    stream_starts,
    stream_nbytes,
    stream_offsets=None,
    stream_gains=None,
    weights=None,
    groups=None,
    n_groups=None,
    first_stream_sample=None,
    last_stream_sample=None,
    is_int64=False,
    on_error="raise",
):
    """Per-sample weighted sums across streams (common modes, pair differences, group averages) without materialising
    the decoded array.

    `groups` gives every stream the output row it adds into: an integer array with one entry per stream, shaped like
    stream_starts or flat in C order; -1 leaves a stream out (it is neither copied nor decoded).  None puts every stream
    in one group and the result is 1-D, (n,); otherwise it is (n_groups, n), n_groups defaulting to groups.max() + 1 (give
    it so that callers without streams in some group get results of the same shape).  `weights`: one float64 per stream
    (default 1.0), used as given.  Samples [first_stream_sample, last_stream_sample) of every stream are combined, and
    offsets and gains (both or neither) restore floats as array_decompress does.

    With x_k the row array_decompress returns for stream k, each output row g is the fold over the streams k of group g
    in storage order, in plain IEEE double (multiply and add each rounded, no FMA):
        acc = +0.0;  acc = acc + w_k * float64(x_k)
    float32 widens exactly and int64 converts with round to nearest even, so
    `for k: acc += w[k] * x[k].astype(np.float64)` in numpy gives the same bits, whatever the residency or the grouping
    of streams into device calls.

    The result is float64: a CUDA tensor when the compressed bytes are on the device, else numpy.  on_error="fill"
    returns (combined, status) with the int32 status shaped like stream_starts: a stream that cannot be decoded adds
    nothing and reports its ERROR_DECODE_* bit.  Streams with group -1 are not examined and report 0 (array_verify checks
    every stream).  A weights or groups size that is not the stream count, non-integer or boolean groups, a group below -1
    or at least n_groups, n_groups < 0, an empty sample range and an unknown on_error raise ValueError before any device
    is used.
    """
    isolate = check_on_error(on_error)
    if (stream_offsets is None) != (stream_gains is None):
        raise RuntimeError("Offsets and gains must be given together")
    first = 0 if first_stream_sample is None else int(first_stream_sample)
    last = int(stream_size) if last_stream_sample is None else int(last_stream_sample)
    if first < 0 or last > stream_size:
        raise ValueError(f"sample range [{first}, {last}) lies outside the stream of {stream_size} samples")
    if last <= first:
        raise ValueError(f"sample range [{first}, {last}) is empty")
    single = not (isinstance(stream_starts, np.ndarray) or is_torch(stream_starts))
    if single:
        stream_starts = ensure_one_element(stream_starts, np.int64)
        stream_nbytes = ensure_one_element(stream_nbytes, np.int64)
    lead = tuple(stream_starts.shape)
    n_stream = int(np.prod(lead))
    w, g, n_out = check_combine_args(n_stream, weights, groups, n_groups)
    offsets = None if stream_offsets is None else _host(stream_offsets)
    gains = None if stream_gains is None else _host(stream_gains)
    out, status = combine_flac(compressed, _host(stream_starts), _host(stream_nbytes), stream_size, first, last, w, g,
                               n_out, offsets, gains, is_int64, isolate)
    if groups is None:
        out = out.reshape(last - first)
    if isolate:
        return out, status.reshape(lead)
    return out


@function_timer
def array_flag_ranges(
    compressed,
    stream_size,
    stream_starts,
    stream_nbytes,
    stream_offsets=None,
    stream_gains=None,
    lo=None,
    hi=None,
    pad=0,
    keep=None,
    first_stream_sample=None,
    last_stream_sample=None,
    is_int64=False,
    on_error="raise",
):
    """Per-stream ranges of samples outside [lo, hi] (glitches, samples at the ADC rails, excursions beyond N sigma)
    without materialising the decoded array.

    A sample whose value v (the value array_decompress returns) satisfies v < lo or v > hi is flagged; a threshold equal
    to v does not flag it.  `lo` and `hi` are each None (no bound on that side), a scalar, or one value per stream shaped
    like stream_starts or flat; at least one must be given, and lo > hi flags every sample.  Float arrays compare the
    restored value, widened to float64, with the float64 threshold.  Integer arrays compare exactly: integer thresholds
    are used as they are, a float lo means x < ceil(lo) and a float hi x > floor(hi).

    Within samples [first_stream_sample, last_stream_sample) of each stream selected by `keep` (a boolean mask shaped
    like stream_starts), every flagged sample j is widened to [j - pad, j + pad + 1); windows that overlap or touch are
    merged (flagged samples j1 < j2 that follow each other share a range iff j2 - j1 <= 2 * pad + 1) and each range is
    clipped to the sample range.  Returns FlagRanges(stream, first, last, nflagged) of int64 numpy arrays: one entry of
    stream / first / last per range, sorted by (stream, first), with stream the flat C-order index into stream_starts
    and first / last absolute sample indices, so array_decompress_windows(..., stream, first, last) cuts the ranges
    out; nflagged, shaped like stream_starts, counts each stream's flagged samples before widening (-1 for streams
    `keep` leaves out).  Compressed bytes on the device are decoded there in groups of streams; host bytes are copied
    to the device in groups.

    on_error="fill" returns (ranges, status) with the int32 status shaped like stream_starts: a stream that cannot be
    decoded gives no ranges and nflagged -1; streams left out report 0.  Both thresholds None, NaN, boolean or
    non-numeric thresholds, a per-stream threshold of the wrong size, a negative, boolean or non-integer pad, an empty
    sample range and an unknown on_error raise ValueError before any device is used.  A pad longer than the stream is
    allowed.
    """
    isolate = check_on_error(on_error)
    if (stream_offsets is None) != (stream_gains is None):
        raise RuntimeError("Offsets and gains must be given together")
    restored = stream_offsets is not None
    first = 0 if first_stream_sample is None else int(first_stream_sample)
    last = int(stream_size) if last_stream_sample is None else int(last_stream_sample)
    if first < 0 or last > stream_size:
        raise ValueError(f"sample range [{first}, {last}) lies outside the stream of {stream_size} samples")
    if last <= first:
        raise ValueError(f"sample range [{first}, {last}) is empty")
    if not (isinstance(stream_starts, np.ndarray) or is_torch(stream_starts)):
        stream_starts = ensure_one_element(stream_starts, np.int64)
        stream_nbytes = ensure_one_element(stream_nbytes, np.int64)
    lead = tuple(stream_starts.shape)
    n_stream = int(np.prod(lead))
    lo, hi, pad = check_flag_args(n_stream, lo, hi, pad, restored)
    if keep is None:
        sel = np.arange(n_stream, dtype=np.int64)
    else:
        k = np.asarray(_host(keep))
        if k.dtype != np.bool_ or k.size != n_stream:
            raise ValueError(f"keep must be a boolean mask with one entry per stream ({n_stream})")
        sel = np.flatnonzero(k.reshape(-1))
    nflagged = np.full(n_stream, -1, np.int64)
    status = np.zeros(n_stream, np.int32)
    stream = first_out = last_out = np.zeros(0, np.int64)
    if sel.size:
        def pick(a):
            return None if a is None else np.asarray(_host(a)).reshape(-1)[sel]

        stream, first_out, last_out, nfl, st = flag_ranges_flac(
            compressed, pick(stream_starts), pick(stream_nbytes), int(stream_size), first, last, lo[sel], hi[sel], pad,
            pick(stream_offsets), pick(stream_gains), is_int64, isolate)
        stream = sel[stream]
        nflagged[sel] = nfl
        if isolate:
            status[sel] = st
    res = FlagRanges(stream, first_out, last_out, nflagged.reshape(lead))
    return (res, status.reshape(lead)) if isolate else res


def project_slice(compressed, stream_size, stream_starts, stream_nbytes, templates, stream_offsets=None,
                  stream_gains=None, keep=None, first_stream_sample=None, last_stream_sample=None, is_int64=False,
                  no_flatten=False, on_error="raise"):
    """array_project with the index tuples of the kept streams and FlacArray's flattening rule: returns (projections,
    indices, status), status None unless on_error="fill"."""
    isolate = check_on_error(on_error)
    if (stream_offsets is None) != (stream_gains is None):
        raise RuntimeError("Offsets and gains must be given together")
    restored = stream_offsets is not None
    first = 0 if first_stream_sample is None else int(first_stream_sample)
    last = int(stream_size) if last_stream_sample is None else int(last_stream_sample)
    if first < 0 or last > stream_size:
        raise ValueError(f"sample range [{first}, {last}) lies outside the stream of {stream_size} samples")
    if last <= first:
        raise ValueError(f"sample range [{first}, {last}) is empty")
    n_tmpl, one_d = check_project_args(templates, last - first)

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
    lead = tuple(starts.shape)
    tail = () if one_d else (n_tmpl,)
    if starts.size == 0:
        out = np.zeros(lead + tail)
        if is_torch(compressed) and compressed.is_cuda:
            import torch

            out = torch.zeros(lead + tail, dtype=torch.float64, device=compressed.device)
        status = np.zeros(lead, np.int32)
    else:
        out, status = project_flac(compressed, starts, nbytes, stream_size, first, last, templates, offsets, gains,
                                   is_int64, isolate)
        out = out.reshape(lead + tail)
        status = None if status is None else status.reshape(lead)
    if single and not no_flatten:
        out = out.reshape(tail)
    return out, indices, (status if isolate else None)


@function_timer
def array_project(
    compressed,
    stream_size,
    stream_starts,
    stream_nbytes,
    templates,
    stream_offsets=None,
    stream_gains=None,
    keep=None,
    first_stream_sample=None,
    last_stream_sample=None,
    is_int64=False,
    on_error="raise",
):
    """Per-stream projections onto templates (common-mode couplings, baseline coefficients, lock-in amplitudes) without
    materialising the decoded array: P[s, t] = sum_i T[t, i] * x_s[i].

    Streams and samples are selected as in array_decompress_slice (`keep`, [first_stream_sample, last_stream_sample),
    offsets and gains both or neither).  `templates`: (n,) or (n_templates, n) real numbers over the n selected samples,
    numpy or any torch tensor; they are copied once to the device as float64.  Returns float64 projections with the shape
    array_decompress_slice's result would have, the sample axis replaced by the template axis (dropped for 1-D
    templates): a CUDA tensor when the compressed bytes are on the device, else numpy.

    With v the row array_decompress returns, widened to float64 (float32 exactly, int64 with round to nearest even), the
    samples are cut into pieces of PROJECT_PIECE = 4096 counted from first_stream_sample, and in plain IEEE double
    (multiply and add each rounded, no FMA):
        per piece j: p_j = +0.0; p_j = p_j + T[t, i] * v[i] in ascending i;  then P = +0.0; P = P + p_j in piece order
    so the result has the same bits whatever the residency or the grouping of streams into device calls.

    on_error="fill" returns (projections, status) as array_stats does: a stream that cannot be decoded gets NaN.
    Templates that are not real numbers or are boolean, that are neither 1-D nor 2-D, whose last axis is not n or that
    hold no template, an empty sample range and an unknown on_error raise ValueError before any device is used.
    """
    out, _, status = project_slice(compressed, stream_size, stream_starts, stream_nbytes, templates,
                                   stream_offsets=stream_offsets, stream_gains=stream_gains, keep=keep,
                                   first_stream_sample=first_stream_sample, last_stream_sample=last_stream_sample,
                                   is_int64=is_int64, on_error=on_error)
    return (out, status) if status is not None else out
