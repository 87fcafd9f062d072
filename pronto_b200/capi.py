"""ctypes binding of librbis_b200.so (the C ABI declared in include/rbis_batch.h).

This module only loads the library and declares prototypes; it performs no arithmetic.  If the
shared library is missing it raises: there is no CPU fallback anywhere in this package.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "librbis_b200.so")

NUM_STATES = 21
COV_ELEMS = 441
MAX_MEAS = 9
MAX_STREAMS = 8
NUM_STATS = 96

MEM_HOST, MEM_DEVICE = 0, 1
MEM_F32_ROWS = 4  # rbis_batch_run_fused: imu / z / quat are float32 arrays (widened exactly on the device)
OP_IMU, OP_MEAS, OP_SNAPSHOT, OP_RESTORE, OP_RECORD = 0, 1, 2, 3, 4
REC_FIELDS = 47  # record fields: 0..20 vec, 21..24 quat w,x,y,z, 25 loglik, 26..46 covariance diagonal
REC_BLOCKS = 7   # record covariance blocks: state indices 3b..3b+2 (omega, v, chi, p, a, gyro bias, accel bias)
INNOV_NIS, INNOV_Y, INNOV_S_DIAG = 1, 2, 4  # rbis_innovation_t::fields: NIS (1 entry), y (m entries), S(a,a) (m entries)
R_SHARED_FULL, R_PER_FILTER_DIAG, R_PER_ROW_FULL = 0, 1, 2
STREAM_SKIP_NAN_ROWS = 1  # rbis_stream_t::flags: a filter whose row holds a NaN in a value the update reads skips that update

c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)
c_int64_p = C.POINTER(C.c_int64)


class Config(C.Structure):
    _fields_ = [
        ("g_val", C.c_double),
        ("chi_tol", C.c_double),
        ("ctor_folds_chi", C.c_int32),
        ("renormalize_quat", C.c_int32),
        ("snapshot_slots", C.c_int32),
        ("device", C.c_int32),
        ("launch_groups", C.c_int32),
        ("dense_only", C.c_int32),
        ("mapping", C.c_int32),
        ("lane_filters_per_cta", C.c_int32),
        ("piece_ops", C.c_int32),
        ("synth_materialize", C.c_int32),
    ]


class Stream(C.Structure):
    _fields_ = [
        ("m", C.c_int32),
        ("has_orientation", C.c_int32),
        ("r_mode", C.c_int32),
        ("sensor_id", C.c_int32),
        ("idx", C.c_int32 * MAX_MEAS),
        ("flags", C.c_int32),
        ("z", C.c_void_p),
        ("quat", C.c_void_p),
        ("R", C.c_void_p),
        ("rows", C.c_int64),
    ]


class SynthStream(C.Structure):
    _fields_ = [
        ("m", C.c_int32),
        ("has_orientation", C.c_int32),
        ("channel", C.c_int32),
        ("channel_rot", C.c_int32),
        ("mean", C.c_void_p),
        ("mean_quat", C.c_void_p),
        ("step", C.c_void_p),
        ("sigma", C.c_double * MAX_MEAS),
        ("sigma_rot", C.c_double * 3),
        ("rows", C.c_int64),
    ]


class Synth(C.Structure):
    _fields_ = [
        ("seed", C.c_uint64),
        ("first_filter", C.c_int64),
        ("mode", C.c_int32),
        ("n_streams", C.c_int32),
        ("imu_mean", C.c_void_p),
        ("imu_step", C.c_void_p),
        ("imu_rows", C.c_int64),
        ("sigma_gyro", C.c_double),
        ("sigma_accel", C.c_double),
        ("dt", C.c_double),
        ("streams", C.POINTER(SynthStream)),
    ]


class FilterState(C.Structure):
    _fields_ = [("utime", C.c_int64), ("quat", C.c_double * 4), ("num_states", C.c_int32), ("reserved0", C.c_int32),
                ("state", C.c_double * NUM_STATES), ("num_cov_elements", C.c_int32), ("reserved1", C.c_int32),
                ("cov", C.c_double * COV_ELEMS)]


class IndexedMeasurement(C.Structure):
    _fields_ = [("utime", C.c_int64), ("state_utime", C.c_int64), ("measured_dim", C.c_int32), ("measured_cov_dim", C.c_int32),
                ("z_effective", C.c_double * MAX_MEAS), ("z_indices", C.c_int32 * MAX_MEAS), ("reserved", C.c_int32),
                ("R_effective", C.c_double * (MAX_MEAS * MAX_MEAS))]


class KvhPacket(C.Structure):
    _fields_ = [("utime", C.c_int64), ("packet_count", C.c_int64), ("delta_rotation", C.c_double * 3), ("linear_acceleration", C.c_double * 3)]


class ImuPacket(C.Structure):
    _fields_ = [("utime_raw", C.c_int64), ("utime_batch", C.c_int64), ("utime", C.c_int64), ("utime_delta", C.c_int64),
                ("packet_count", C.c_int64), ("delta_rotation", C.c_double * 3), ("linear_acceleration", C.c_double * 3)]


class Record(C.Structure):
    _fields_ = [
        ("fields", C.c_uint64),
        ("out", C.c_void_p),
        ("rows", C.c_int64),
        ("mem", C.c_int32),
        ("cov_blocks", C.c_int32),
    ]


class Innovation(C.Structure):
    _fields_ = [
        ("fields", C.c_uint32),
        ("m", C.c_int32),
        ("out", C.c_void_p),
        ("rows", C.c_int64),
    ]


class Op(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("stream", C.c_int32),
        ("row", C.c_int64),
        ("utime", C.c_int64),
        ("dt", C.c_double),
    ]


# every symbol include/rbis_batch.h declares: name -> (restype, argtypes)
PROTOTYPES = {
    "rbis_last_error": (C.c_char_p, []),
    "rbis_default_config": (None, [C.POINTER(Config)]),
    "rbis_batch_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int64, C.POINTER(Config)]),
    "rbis_batch_destroy": (C.c_int, [C.c_void_p]),
    "rbis_batch_synchronize": (C.c_int, [C.c_void_p]),
    "rbis_batch_num_filters": (C.c_int64, [C.c_void_p]),
    "rbis_batch_stream": (C.c_void_p, [C.c_void_p]),
    "rbis_batch_launch_count": (C.c_int64, [C.c_void_p]),
    "rbis_batch_last_kernel_variant": (C.c_int, [C.c_void_p]),
    "rbis_batch_notch_configure": (C.c_int, [C.c_void_p, C.c_double, C.c_double, C.c_int, C.c_int64]),
    "rbis_batch_notch_filter": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int]),
    "rbis_smooth_plan": (C.c_int64, [C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rbis_batch_smooth_backward": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_void_p, C.c_double]),
    "rbis_batch_get_snapshot": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "rbis_batch_set_state": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int]),
    "rbis_batch_get_state": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, c_int64_p, C.c_int]),
    "rbis_batch_set_filter": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double]),
    "rbis_batch_get_filter": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, c_double_p]),
    "rbis_batch_set_process_noise": (C.c_int, [C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_double]),
    "rbis_batch_set_process_noise_per_filter": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "rbis_batch_ins_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_int64, C.c_int]),
    "rbis_batch_indexed_update": (C.c_int, [C.c_void_p, C.c_int, c_int32_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int]),
    "rbis_batch_indexed_orient_update": (C.c_int, [C.c_void_p, C.c_int, c_int32_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int]),
    "rbis_batch_set_column_map": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64]),
    "rbis_batch_set_record": (C.c_int, [C.c_void_p, C.POINTER(Record)]),
    "rbis_batch_set_innovations": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(Innovation)]),
    "rbis_batch_run_fused": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(Op), C.c_void_p, C.c_int64, C.c_int, C.POINTER(Stream), C.c_int]),
    "rbis_batch_synthesize": (C.c_int, [C.c_void_p, C.POINTER(Synth), C.c_void_p, C.c_void_p, C.c_void_p]),
    "rbis_batch_run_fused_synth": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(Op), C.c_int, C.POINTER(Stream), C.POINTER(Synth)]),
    "rbis_batch_get_filter_states": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.POINTER(FilterState)]),
    "rbis_batch_set_filter_states": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.POINTER(FilterState)]),
    "rbis_record_filter_states": (C.c_int, [C.c_uint64, C.c_int32, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                            C.POINTER(FilterState)]),
    "rbis_stream_from_indexed_measurement": (C.c_int, [C.POINTER(IndexedMeasurement), C.POINTER(Stream), C.c_void_p]),
    "rbis_stream_from_indexed_measurements": (C.c_int, [C.POINTER(IndexedMeasurement), C.c_int64, C.POINTER(Stream), C.c_void_p]),
    "rbis_kvh_stream_create": (C.c_int, [C.POINTER(C.c_void_p)]),
    "rbis_kvh_stream_destroy": (C.c_int, [C.c_void_p]),
    "rbis_kvh_decode_batch": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.POINTER(KvhPacket), C.POINTER(ImuPacket), c_int32_p, C.POINTER(ImuPacket), c_int32_p]),
    "rbis_kvh_imu_step": (C.c_int, [C.POINTER(ImuPacket), C.c_int64, c_double_p, c_double_p, C.c_double, c_int64_p, c_double_p, c_double_p, c_double_p]),
    "rbis_planner_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int64, C.c_int32, C.c_int64, C.c_int64, C.c_int64]),
    "rbis_planner_destroy": (C.c_int, [C.c_void_p]),
    "rbis_planner_add_update": (C.c_int, [C.c_void_p, C.POINTER(Op), C.c_int]),
    "rbis_planner_pending": (C.c_int64, [C.c_void_p]),
    "rbis_planner_take": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, c_int64_p]),
    "rbis_planner_counters": (C.c_int, [C.c_void_p, c_int64_p]),
    "rbis_batch_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, c_int64_p, C.c_void_p, C.c_int]),
    "rbis_batch_stats_enqueue": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, c_int64_p]),
    "rbis_batch_stats_snapshot_enqueue": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, c_int64_p,
                                                     C.POINTER(C.c_int32)]),
    "rbis_batch_stats_records_enqueue": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                                    C.c_void_p, c_int64_p, C.POINTER(C.c_int32)]),
    "rbis_batch_stats_innovations_enqueue": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_int64, C.c_int, C.c_void_p, C.c_void_p,
                                                        c_int64_p, C.POINTER(C.c_int32)]),
    "rbis_batch_stats_allreduce": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]),
    "rbis_batch_window_neg_loglik": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int,
                                               C.c_void_p, C.c_void_p, C.c_int]),
    "rbis_batch_record": (C.c_int, [C.c_void_p, c_int32_p]),
    "rbis_batch_wait": (C.c_int, [C.c_void_p, C.c_int32]),
    "rbis_stats_reduce_chunks": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p]),
    "rbis_measure_fp64_peak": (C.c_int, [C.c_int, C.c_int, c_double_p, c_double_p]),
}

_lib = None


def load():
    """Load librbis_b200.so (built by __graft_entry__.build()); raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
            "pronto_b200 has no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (restype, argtypes) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


class RBISError(RuntimeError):
    pass


def check(rc):
    if rc != 0:
        raise RBISError(f"rbis error {rc}: {load().rbis_last_error().decode()}")
