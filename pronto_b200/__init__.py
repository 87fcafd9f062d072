"""pronto_b200 -- B200-native batched RBIS EKF hot path (openhumanoids/pronto's 21-state filter).

The product is librbis_b200.so (CUDA sm_100a, C ABI in include/rbis_batch.h); this package is the
Python host mirror used by tests, bench.py and the multi-GPU driver.  No CPU compute path exists.
"""
from . import capi  # noqa: F401
from .batch import (MeasStream, RBISBatch, SynthSpec, make_ops, measure_fp64_peak, record_fields, record_layout,  # noqa: F401
                    reduce_chunks)

__all__ = ["capi", "RBISBatch", "MeasStream", "make_ops", "record_fields", "record_layout", "reduce_chunks", "measure_fp64_peak"]
