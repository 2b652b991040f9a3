"""B200-native exact pattern matching: the Boyer-Moore scan path of
AnupBS28/PARALLEL_IMPLEMENTATION_OF_STRING_MATCHING_ALGORITHMS_OPENCL rebuilt as hand-written
sm_100a CUDA behind a C ABI (include/bmx.h).  See DESIGN.md and INTEGRATION.md."""
from . import _lib, synth  # noqa: F401
from ._lib import BmxError, LIB_PATH  # noqa: F401
from .host import (Dictionary, Exchange, MultiGpu, Scanner, build_tables, device_count, find_first, find_first_device,  # noqa: F401
                   partition_words, search, search_device, search_multi, search_multi_device, search_partitions,
                   search_ranges, search_ranges_device, version)

__all__ = [
    "BmxError", "Dictionary", "Exchange", "LIB_PATH", "MultiGpu", "Scanner", "build_tables", "device_count", "find_first",
    "find_first_device", "partition_words",
    "search", "search_device", "search_multi", "search_multi_device", "search_partitions", "search_ranges",
    "search_ranges_device", "version", "synth",
]
