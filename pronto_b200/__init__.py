"""pronto_b200 -- B200-native batched RBIS EKF hot path (openhumanoids/pronto's 21-state filter).

The product is librbis_b200.so (CUDA sm_100a, C ABI in include/rbis_batch.h); this package is the
Python host mirror used by tests, bench.py and the multi-GPU driver.  No CPU compute path exists.
"""
from . import capi  # noqa: F401
from .batch import (MeasStream, RBISBatch, SynthSpec, filter_states_from_record, innovation_layout, make_ops,  # noqa: F401
                    measure_fp64_peak, record_cov_blocks, record_fields, record_layout, reduce_chunks)

__all__ = ["capi", "RBISBatch", "MeasStream", "make_ops", "record_fields", "record_layout", "record_cov_blocks",
           "filter_states_from_record", "innovation_layout", "reduce_chunks", "measure_fp64_peak"]
