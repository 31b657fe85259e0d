"""pcpx — B200-native neighbourhood engine behind pcp's API (Python test / bench driver).

The product is ``lib/libpcpx.so`` (CUDA C++ for sm_100a behind the C ABI in ``include/pcpx.h``)
and the C++17 drop-in headers in ``include/pcpx/``.  This package is a thin ctypes binding over
the SAME C ABI, used by ``tests/`` and ``bench.py``.  The directory name carries a hyphen, so
import it with::

    import importlib; pcpx = importlib.import_module("point-cloud-processing_b200")

There is no CPU fallback: importing works without a GPU (so that the exported symbols can be
checked), but every compute call fails loudly when the library or a CUDA device is missing.
"""
from .capi import (  # noqa: F401
    LIB_PATH,
    NO_NEIGHBOUR,
    NOISE,
    Index,
    PcpxError,
    bilateral_filter_normals,
    bilateral_filter_points,
    device_count,
    exported_symbols,
    extract_bands,
    lib,
    normals_from_neighbourhoods,
    orient_normals_graph,
    set_tuning,
    wlop,
)
from . import sharding, synth  # noqa: F401
