"""vega_b200 — B200-native (sm_100a) shuffle + aggregation engine behind vega's RDD operator API.

The product is vega_b200/libvega_b200.so (C ABI in include/vega_b200.h, CUDA kernels in
vega_b200/csrc/).  This package is the host-side mirror of the reference's operator
interface for the path (rdd.py) plus the one-process-per-GPU exchange (dist.py).
Importing works without a GPU (so the C ABI can be inspected); computing does not.
"""
from ._lib import (LIB_PATH, SYMBOLS, VegaB200Error, lib)  # noqa: F401
from .rdd import Context, Grouped, JoinedRdd, OuterJoinedRdd, PairRdd, Rdd, Shuffle, ShuffledRdd, slice_starts  # noqa: F401

__all__ = ["Context", "PairRdd", "Rdd", "Shuffle", "ShuffledRdd", "JoinedRdd", "OuterJoinedRdd", "Grouped", "slice_starts",
           "VegaB200Error", "lib", "LIB_PATH", "SYMBOLS"]
