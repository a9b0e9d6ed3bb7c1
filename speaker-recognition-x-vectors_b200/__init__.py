"""B200-native x-vector embedding extractor — drop-in for the reference's extraction path.

    from xvec_b200 import XVectorModel, TdnnLayer        # (alias of this package, see /xvec_b200.py)

The compute lives in libxvec_b200.so (hand-written sm_100a CUDA, C ABI in include/xvec_b200.h).
"""
from . import _lib, layout, ops  # noqa: F401
from .layout import balanced_batches, build_layout, bucket_batches, lpt_partition, sliding_windows, window_layout  # noqa: F401
from .tdnn_layer import TdnnLayer, get_time_context, tap_offsets  # noqa: F401
from .xvector import XVectorModel  # noqa: F401
from .extractor import HostExtractor  # noqa: F401
from . import io_csv, scoring, sharding  # noqa: F401
from .io_csv import read_xvector_csv, write_xvector_csv  # noqa: F401

TDNN = TdnnLayer  # BASELINE.json's north_star calls the layer "TDNN"

__all__ = ["TdnnLayer", "TDNN", "XVectorModel", "get_time_context", "tap_offsets", "build_layout", "bucket_batches",
           "lpt_partition", "balanced_batches", "sliding_windows", "window_layout", "ops", "layout", "HostExtractor", "io_csv", "scoring", "sharding", "read_xvector_csv", "write_xvector_csv"]
