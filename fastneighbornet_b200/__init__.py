"""fastneighbornet_b200 — B200-native Neighbor-Net hot path behind the FastNeighborNet interface.

The package is a thin host-side mirror of the reference's operator interface
(NetMakerOriginal.runNeighborNet, CircularSplitWeights.getWeights) over the C-ABI
library libfastnn.so (include/fastnn.h).  There is no CPU fallback: importing works
anywhere, computing needs the built library and a B200.
"""
from .api import (  # noqa: F401
    FastNNError,
    Context,
    NeighborNetCanonical,
    NeighborNetLocal,
    NeighborNetRandom,
    default_opts,
    device_count,
    lib,
    lib_path,
    order,
    rowsums,
    seq_sum,
    split_weights,
    split_weights_budget,
    csw_matvec,
    weighted_splits,
    network_splits,
    network,
    bootstrap,
    read_phylip,
    read_alignment,
    distances,
    MODELS,
    write_nexus,
    java_double_str,
    release_cache,
)
from . import synth  # noqa: F401
