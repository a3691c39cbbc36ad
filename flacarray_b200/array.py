"""FlacArray: FLAC-compressed N-d array, drop-in for /root/reference/src/flacarray/array.py:19-884.

Same constructor keywords, properties, slicing semantics (`__getitem__`, array.py:279-449), `to_array`
(keep mask / stream_slice / keep_indices, array.py:518-584), `from_array` (array.py:586-637) and byte
bookkeeping (`stream_starts`, `stream_nbytes`, global offsets via an all-gather of byte counts,
mpi.py:156-187).  Compression and decompression run on the GPU.

Documented differences (SURVEY App. C): properties that raise AttributeError in the reference (Q3:
`global_process_nbytes`, `nstreams`, `global_nstreams`, `global_stream_nbytes`) return the intended
values; an all-integer key returns the selected sample instead of a zero (Q4).  `to_array` keeps the
reference behaviour of forwarding `stream_slice.start/.stop` unnormalised (Q5).
"""
import copy

import numpy as np

from .compress import array_compress
from .decompress import array_decompress_slice, array_decompress_windows
from .libflacarray import is_torch
from .mpi import global_array_properties, global_bytes
from .utils import log


def _nbytes_of(compressed):
    if is_torch(compressed):
        return int(compressed.numel())
    return int(compressed.nbytes)


class FlacArray:
    """FLAC compressed array representation (see the reference class docstring, array.py:20-77)."""

    def __init__(
        self,
        other,
        shape=None,
        global_shape=None,
        compressed=None,
        dtype=None,
        stream_starts=None,
        stream_nbytes=None,
        stream_offsets=None,
        stream_gains=None,
        mpi_comm=None,
        mpi_dist=None,
    ):
        if other is not None:
            self._shape = copy.deepcopy(other._shape)
            self._global_shape = copy.deepcopy(other._global_shape)
            self._compressed = other._compressed.clone() if is_torch(other._compressed) else copy.deepcopy(other._compressed)
            self._dtype = np.dtype(other._dtype)
            self._stream_starts = copy.deepcopy(other._stream_starts)
            self._stream_nbytes = copy.deepcopy(other._stream_nbytes)
            self._stream_offsets = copy.deepcopy(other._stream_offsets)
            self._stream_gains = copy.deepcopy(other._stream_gains)
            self._mpi_dist = copy.deepcopy(other._mpi_dist)
            self._mpi_comm = other._mpi_comm
        else:
            self._shape = tuple(shape)
            self._global_shape = tuple(global_shape)
            self._compressed = compressed
            self._dtype = np.dtype(dtype)
            self._stream_starts = stream_starts
            self._stream_nbytes = stream_nbytes
            self._stream_offsets = stream_offsets
            self._stream_gains = stream_gains
            self._mpi_comm = mpi_comm
            self._mpi_dist = mpi_dist
        self._init_params()

    def _init_params(self):
        if len(self._shape) == 1:
            self._flatten_single = True
            self._local_shape = (1, self._shape[0])
        else:
            self._flatten_single = False
            self._local_shape = self._shape
        self._local_nbytes = _nbytes_of(self._compressed)
        (
            self._global_nbytes,
            self._global_proc_nbytes,
            self._global_stream_starts,
        ) = global_bytes(self._local_nbytes, self._stream_starts, self._mpi_comm)
        self._leading_shape = self._local_shape[:-1]
        self._global_leading_shape = self._global_shape[:-1]
        self._stream_size = self._local_shape[-1]
        self._local_nstreams = int(np.prod(self._leading_shape))
        self._global_nstreams = int(np.prod(self._global_leading_shape))
        self._typestr = self._dtype_str(self._dtype)
        self._is_int64 = self._dtype == np.dtype(np.int64) or self._dtype == np.dtype(np.float64)

    @staticmethod
    def _dtype_str(dt):
        for name in ("float64", "float32", "int64", "int32"):
            if dt == np.dtype(name):
                return name
        raise RuntimeError(f"Unsupported dtype '{dt}'")

    # ---- shapes ----
    @property
    def shape(self):
        """The shape of the local, uncompressed array."""
        return self._shape

    @property
    def global_shape(self):
        """The global shape of array across any communicator."""
        return self._global_shape

    @property
    def leading_shape(self):
        return self._leading_shape

    @property
    def global_leading_shape(self):
        return self._global_leading_shape

    @property
    def stream_size(self):
        """The uncompressed length of each stream."""
        return self._stream_size

    # ---- compressed data ----
    @property
    def nbytes(self):
        """Compressed bytes on the local process."""
        return self._local_nbytes

    @property
    def global_nbytes(self):
        return self._global_nbytes

    @property
    def global_process_nbytes(self):
        return self._global_proc_nbytes

    @property
    def nstreams(self):
        return self._local_nstreams

    @property
    def global_nstreams(self):
        return self._global_nstreams

    @property
    def compressed(self):
        """The concatenated raw bytes of all streams on the local process."""
        return self._compressed

    @property
    def stream_starts(self):
        return self._stream_starts

    @property
    def stream_nbytes(self):
        return self._stream_nbytes

    @property
    def global_stream_starts(self):
        return self._global_stream_starts

    @property
    def global_stream_nbytes(self):
        return self._stream_nbytes

    @property
    def stream_offsets(self):
        return self._stream_offsets

    @property
    def stream_gains(self):
        return self._stream_gains

    @property
    def mpi_comm(self):
        return self._mpi_comm

    @property
    def mpi_dist(self):
        return self._mpi_dist

    @property
    def dtype(self):
        return self._dtype

    @property
    def typestr(self):
        return self._typestr

    # ---- indexing: one resolver turns any key into (keep mask, sample window, result shape) ----
    def _resolve_key(self, raw_key):
        """Normalise an indexing key.

        Same selection rules as the reference's __getitem__ (array.py:279-449): integers and slices (any step) on the
        leading axes, an integer or a contiguous slice on the sample axis, missing axes mean "everything", a 1-D array
        is addressed by its sample axis alone.  Returns (keep, first, last, shape): `keep` is a boolean mask over the
        leading axes (None when nothing is selected), [first, last) the sample window and `shape` the shape of the
        result.  Streams always come back in storage order (a negative step does not reverse them -- array.py:287).
        Supersets: negative integers count from the end, an out-of-range integer selects nothing instead of raising.
        """
        key = raw_key if isinstance(raw_key, tuple) else (raw_key,)
        if self._flatten_single:
            if len(key) != 1:
                raise ValueError(f"Slice key {raw_key} is not valid for single, flattened stream.")
            key = (0,) + key
        ndim = len(self._local_shape)
        if len(key) > ndim:
            raise ValueError(f"Invalid slice key {raw_key}, too many dimensions")
        key = key + (slice(None),) * (ndim - len(key))

        picked = []          # per leading axis: the indices it keeps
        shape = []           # axes of the result (integer keys drop theirs)
        for n, k in zip(self._leading_shape, key[:-1]):
            if isinstance(k, (int, np.integer)):
                i = int(k) + (n if k < 0 else 0)
                inside = 0 <= i < n
                picked.append(np.array([i] if inside else [], dtype=np.int64))
                if not inside:
                    shape.append(0)
            elif isinstance(k, slice):
                idx = np.arange(n, dtype=np.int64)[k]
                picked.append(idx)
                shape.append(idx.size)
            else:
                raise ValueError("Leading dimensions support integer indices and slices.")
        if self._flatten_single:
            shape = []

        size = self._stream_size
        k = key[-1]
        if k is None:
            k = slice(None)
        if isinstance(k, slice):
            first, last, step = k.indices(size)
            if step != 1:
                raise ValueError("Only stride==1 supported on stream slices")
            last = max(last, first)
            shape.append(last - first)
        elif isinstance(k, (int, np.integer)):
            first = int(k) + (size if k < 0 else 0)
            last = first + 1
            if not 0 <= first < size:
                first = last = 0          # nothing to decode: the result is zeros of the leading shape
        else:
            raise ValueError("Stream dimension supports contiguous slices or single indices.")

        keep = None
        if last > first and all(ix.size for ix in picked):
            keep = np.zeros(self._leading_shape, dtype=bool)
            keep[np.ix_(*picked)] = True
        return keep, first, last, tuple(shape)

    def __getitem__(self, raw_key):
        """Decompress a slice of data on the fly (array.py:409-449)."""
        keep, first, last, shape = self._resolve_key(raw_key)
        if keep is None:
            return np.zeros(shape, dtype=self._dtype)
        arr, _ = array_decompress_slice(
            self._compressed,
            self._stream_size,
            self._stream_starts,
            self._stream_nbytes,
            stream_offsets=self._stream_offsets,
            stream_gains=self._stream_gains,
            keep=keep,
            first_stream_sample=first,
            last_stream_sample=last,
            is_int64=self._is_int64,
        )
        return arr.reshape(shape)

    def __delitem__(self, key):
        raise RuntimeError("Cannot delete individual streams")

    def __setitem__(self, key, value):
        raise RuntimeError("Cannot modify individual byte streams")

    def __repr__(self):
        where = ""
        if self._mpi_comm is not None:
            lo, hi = self._mpi_dist[self._mpi_comm.rank]
            where = f" | Rank {self._mpi_comm.rank:04d} {lo}-{hi - 1} |"
        return f"<FlacArray{where} {self._typestr} shape={self._shape} bytes={self._local_nbytes}>"

    def __eq__(self, other):
        """Same data in the same layout (array.py:469-516): shapes, dtype, stream starts and the compressed BYTES must
        be identical, offsets / gains equal to floating-point tolerance."""
        def host(x):
            return x.cpu().numpy() if is_torch(x) else x

        for name in ("_shape", "_dtype", "_global_shape"):
            if getattr(self, name) != getattr(other, name):
                log.debug(f"FlacArray.__eq__: {name[1:]} differs")
                return False
        for name in ("_stream_starts", "_compressed"):
            if not np.array_equal(host(getattr(self, name)), host(getattr(other, name))):
                log.debug(f"FlacArray.__eq__: {name[1:]} differs")
                return False
        for name in ("_stream_offsets", "_stream_gains"):
            mine, theirs = getattr(self, name), getattr(other, name)
            if (mine is None) != (theirs is None) or (mine is not None and not np.allclose(host(mine), host(theirs))):
                log.debug(f"FlacArray.__eq__: {name[1:]} differs")
                return False
        return True

    def to_array(self, keep=None, stream_slice=None, keep_indices=False, use_threads=False):
        """Decompress local data into an array (array.py:518-584)."""
        first_samp = None
        last_samp = None
        if stream_slice is not None:
            if stream_slice.step is not None and stream_slice.step != 1:
                raise RuntimeError("Only stream slices with a step size of 1 are supported")
            first_samp = stream_slice.start
            last_samp = stream_slice.stop
        arr, indices = array_decompress_slice(
            self._compressed,
            self._stream_size,
            self._stream_starts,
            self._stream_nbytes,
            stream_offsets=self._stream_offsets,
            stream_gains=self._stream_gains,
            keep=keep,
            first_stream_sample=first_samp,
            last_stream_sample=last_samp,
            is_int64=self._is_int64,
            use_threads=use_threads,
            no_flatten=(not self._flatten_single),
        )
        if keep is not None and keep_indices:
            return (arr, indices)
        return arr

    def to_windows(self, streams, first, last):
        """Decompress many sample windows of local streams in one call.

        Window i is samples [first[i], last[i]) of stream streams[i].  `streams` is either flat C-order indices over
        the leading shape or a tuple of index arrays, one per leading axis (as np.nonzero returns); a 1-D array has the
        single stream 0.  `first` / `last` may be scalars.  Returns (data, offsets) like array_decompress_windows:
        window i is data[offsets[i]:offsets[i + 1]] in the array's dtype.
        """
        if isinstance(streams, tuple):
            if len(streams) != len(self._leading_shape):
                raise RuntimeError(
                    f"streams has {len(streams)} index arrays for {len(self._leading_shape)} leading axes")
            idx = [np.asarray(a, dtype=np.int64).reshape(-1) for a in streams]
            if len({a.size for a in idx}) > 1:
                raise RuntimeError("the index arrays of streams must have the same length")
            for ax, (a, n) in enumerate(zip(idx, self._leading_shape)):
                if a.size and (int(a.min()) < 0 or int(a.max()) >= n):
                    raise RuntimeError(f"window stream index out of range on leading axis {ax} of length {n}")
            streams = np.ravel_multi_index(tuple(idx), self._leading_shape) if idx and idx[0].size else np.zeros(0, np.int64)
        starts = np.asarray(self._stream_starts).reshape(-1)
        nbytes = np.asarray(self._stream_nbytes).reshape(-1)
        offsets = None if self._stream_offsets is None else np.asarray(self._stream_offsets).reshape(-1)
        gains = None if self._stream_gains is None else np.asarray(self._stream_gains).reshape(-1)
        return array_decompress_windows(self._compressed, self._stream_size, starts, nbytes, streams, first, last,
                                        stream_offsets=offsets, stream_gains=gains, is_int64=self._is_int64)

    @classmethod
    def from_array(cls, arr, level=5, quanta=None, precision=None, mpi_comm=None, use_threads=False):
        """Construct a FlacArray from an array (array.py:586-637).

        `arr` may be a numpy array or a CUDA torch tensor; in the latter case the compressed bytes stay
        on the device.  With `mpi_comm` the array is this rank's block of the leading axis.
        """
        global_props = global_array_properties(tuple(arr.shape), mpi_comm=mpi_comm)
        global_shape = global_props["shape"]
        mpi_dist = global_props["dist"]
        compressed, starts, nbytes, offsets, gains = array_compress(
            arr, level=level, quanta=quanta, precision=precision, use_threads=use_threads
        )
        if is_torch(starts):
            starts = starts.cpu().numpy()
            nbytes = nbytes.cpu().numpy()
            if offsets is not None:
                offsets = offsets.cpu().numpy()
                gains = gains.cpu().numpy()
        from .libflacarray import np_dtype

        return FlacArray(
            None,
            shape=tuple(arr.shape),
            global_shape=global_shape,
            compressed=compressed,
            dtype=np_dtype(arr),
            stream_starts=starts,
            stream_nbytes=nbytes,
            stream_offsets=offsets,
            stream_gains=gains,
            mpi_comm=mpi_comm,
            mpi_dist=mpi_dist,
        )

    # ---- file I/O (array.py:639-884): format version 1 group layout, see io_common.py ----
    def _write_group(self, grp):
        from . import __version__
        from .io_common import write_compressed

        write_compressed(
            grp, self._leading_shape, self._global_leading_shape, self._stream_size, self._stream_starts,
            self._global_stream_starts, self._stream_nbytes, self._stream_offsets, self._stream_gains, self._compressed,
            2 if self._is_int64 else 1, self._local_nbytes, self._global_nbytes, self._global_proc_nbytes,
            self._mpi_comm, self._mpi_dist, software_version=__version__)

    @classmethod
    def _read_group(cls, grp, keep, mpi_comm, mpi_dist, no_flatten):
        from .io_common import read_compressed
        from .utils import compressed_dtype

        (local_shape, global_shape, compressed, n_channels, starts, nbytes, offsets, gains, mpi_dist, _) = read_compressed(
            grp, keep=keep, mpi_comm=mpi_comm, mpi_dist=mpi_dist)
        if compressed is None:
            raise RuntimeError("No streams selected on this process")
        dt = compressed_dtype(n_channels, offsets, gains)
        if len(local_shape) == 2 and local_shape[0] == 1 and not no_flatten:
            shape = (local_shape[1],)
        else:
            shape = local_shape
        return FlacArray(None, shape=shape, global_shape=global_shape, compressed=compressed, dtype=dt,
                         stream_starts=starts, stream_nbytes=nbytes, stream_offsets=offsets, stream_gains=gains,
                         mpi_comm=mpi_comm, mpi_dist=mpi_dist)

    def write_hdf5(self, hgrp):
        """Write the compressed representation to an open HDF5 group (array.py:639-681)."""
        self._write_group(hgrp)

    @classmethod
    def read_hdf5(cls, hgrp, keep=None, mpi_comm=None, mpi_dist=None, no_flatten=False):
        """Construct a FlacArray from an HDF5 group (array.py:683-764)."""
        return cls._read_group(hgrp, keep, mpi_comm, mpi_dist, no_flatten)

    def write_zarr(self, zgrp):
        """Write the compressed representation to an open zarr group (array.py:766-803)."""
        self._write_group(zgrp)

    @classmethod
    def read_zarr(cls, zgrp, keep=None, mpi_comm=None, mpi_dist=None, no_flatten=False):
        """Construct a FlacArray from a zarr group (array.py:805-884)."""
        return cls._read_group(zgrp, keep, mpi_comm, mpi_dist, no_flatten)
