"""flacarray_b200: B200-native (sm_100a CUDA) implementation of flacarray's FLAC encode/decode hot path.

Public names follow hpc4cmb/flacarray: FlacArray, array_compress, array_decompress[_slice],
float_to_int, int_to_float; array_decompress_windows (and FlacArray.to_windows), array_verify (and FlacArray.verify),
array_stats (and FlacArray.stats), array_combine (and FlacArray.combine), array_flag_ranges (and
FlacArray.flag_ranges), array_project (and FlacArray.project) and on_error="fill" (per-stream fault isolation) are additions.
The compiled extension of the reference (`flacarray.libflacarray`) is replaced by `flacarray_b200.libflacarray` (ctypes over libflacarray_b200.so).  No CPU fallback.
"""
__version__ = "0.1.0"

from .array import FlacArray  # noqa: F401
from .compress import array_compress  # noqa: F401
from .decompress import (array_combine, array_decompress, array_decompress_slice, array_decompress_windows,  # noqa: F401
                         array_flag_ranges, array_project, array_stats, array_verify)
from .libflacarray import FlagRanges, StreamStats  # noqa: F401
from .utils import float_to_int, int_to_float  # noqa: F401
