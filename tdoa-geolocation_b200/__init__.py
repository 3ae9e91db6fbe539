"""tdoa-geolocation_b200 -- B200-native drop-in for the processing stage of
KX0U-Jim/tdoa-geolocation (processor.go): hand-written sm_100a CUDA kernels behind a
C ABI (include/tdoa_b200.h, built as libtdoa_b200.so), plus this thin host-side mirror
of the reference's TDOAProcessor interface.

The directory name is not a Python identifier; import it with
    importlib.import_module("tdoa-geolocation_b200")
or through the repo-root shim `tdoa_b200`.
"""
from ._native import (  # noqa: F401
    Engine,
    TdoaError,
    Peak,
    MODE_SOURCE,
    MODE_BINARY,
    MODE_EXTENDED,
    KIND_REF,
    KIND_TGT,
    default_config,
    library_path,
    load_library,
    host_alloc,
    comm_unique_id,
    PEAK_DTYPE,
    PEAK_EDGE,
    PEAK_EMPTY,
)
from .processor import Station, TDOAProcessor  # noqa: F401
from . import sharding  # noqa: F401
from . import analyzer  # noqa: F401

__all__ = [
    "Engine", "TdoaError", "Peak", "MODE_SOURCE", "MODE_BINARY", "MODE_EXTENDED", "KIND_REF", "KIND_TGT",
    "default_config", "library_path", "load_library", "host_alloc", "comm_unique_id", "PEAK_DTYPE", "PEAK_EDGE", "PEAK_EMPTY", "Station", "TDOAProcessor", "sharding", "analyzer",
]
