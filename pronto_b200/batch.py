"""Thin Python host mirror of the batch API (tests, bench and the multi-GPU driver use it).

All arithmetic happens in librbis_b200.so (CUDA, sm_100a).  Arrays may be numpy (host memory) or
torch CUDA tensors (device memory, used in place); layouts are those of include/rbis_batch.h
(structure of arrays, filter index fastest).
"""
import ctypes as C

import numpy as np

from . import capi

OP_DTYPE = np.dtype([("kind", "<i4"), ("stream", "<i4"), ("row", "<i8"), ("utime", "<i8"), ("dt", "<f8")], align=True)
assert OP_DTYPE.itemsize == C.sizeof(capi.Op)


def _is_torch(a):
    return type(a).__module__.startswith("torch")


def _ptr(a, shape=None, name="array"):
    """(address, mem) of a float64 contiguous numpy array or torch CUDA tensor."""
    if a is None:
        return None, None
    if _is_torch(a):
        import torch

        if a.dtype != torch.float64 or not a.is_contiguous():
            raise ValueError(f"{name}: need a contiguous float64 tensor")
        if shape is not None and tuple(a.shape) != tuple(shape):
            raise ValueError(f"{name}: shape {tuple(a.shape)} != {tuple(shape)}")
        return a.data_ptr(), (capi.MEM_DEVICE if a.is_cuda else capi.MEM_HOST)
    if not isinstance(a, np.ndarray) or a.dtype != np.float64 or not a.flags.c_contiguous:
        raise ValueError(f"{name}: need a C-contiguous float64 numpy array")
    if shape is not None and tuple(a.shape) != tuple(shape):
        raise ValueError(f"{name}: shape {a.shape} != {tuple(shape)}")
    return a.ctypes.data, capi.MEM_HOST


def _ptr_rows(a, name):
    """(address, mem, is_f32) of a sensor-row array for run_fused: float64 or float32, numpy or torch."""
    if _is_torch(a):
        import torch

        if a.dtype not in (torch.float64, torch.float32) or not a.is_contiguous():
            raise ValueError(f"{name}: need a contiguous float64 or float32 tensor")
        return a.data_ptr(), (capi.MEM_DEVICE if a.is_cuda else capi.MEM_HOST), a.dtype == torch.float32
    if not isinstance(a, np.ndarray) or a.dtype not in (np.float64, np.float32) or not a.flags.c_contiguous:
        raise ValueError(f"{name}: need a C-contiguous float64 or float32 numpy array")
    return a.ctypes.data, capi.MEM_HOST, a.dtype == np.float32


def _common_mem(mems, what):
    mems = [m for m in mems if m is not None]
    if not mems:
        return capi.MEM_HOST
    if any(m != mems[0] for m in mems):
        raise ValueError(f"{what}: all arrays of one call must live in the same memory space")
    return mems[0]


class MeasStream:
    """Constant part + data of an RBISIndexed[PlusOrientation]Measurement stream
    (MSE/rbis_update_interface.hpp:84-120): index set, z rows, R, optional orientation rows.

    R: one m x m matrix for every row; or [rows][m][m], row r's matrix for the update that reads row r
    (RBIS_R_PER_ROW_FULL); or [m][N] per-filter diagonals with per_filter_diag=True.

    skip_nan_rows=True (RBIS_STREAM_SKIP_NAN_ROWS): a filter whose row holds a NaN in a value the update reads (z[row, :, n],
    without the chi entries of an orientation stream) did not receive that row and skips the update, bit for bit as if its
    MEAS op were deleted from the program.  run_fused only."""

    def __init__(self, idx, z, R, quat=None, per_filter_diag=False, sensor_id=0, skip_nan_rows=False):
        self.idx = [int(i) for i in idx]
        self.z, self.R, self.quat = z, R, quat
        self.per_filter_diag = bool(per_filter_diag)
        self.sensor_id = int(sensor_id)
        self.skip_nan_rows = bool(skip_nan_rows)


class SynthSpec:
    """Noise-free rows + noise description of one time chunk (rbis_synth_t): what rbis_batch_run_fused_synth /
    rbis_batch_synthesize turn into per-filter input rows on the device.

    imu_mean [rows][6], imu_step [rows]; streams: list of dicts with mean [rows][m], step [rows], sigma [m], channel and,
    for orientation streams, mean_quat [rows][4], sigma_rot [3], channel_rot.  sigma_gyro / sigma_accel < 0: per filter
    sqrt(q / dt) from the handle's process noise."""

    def __init__(self, seed, imu_mean, imu_step, streams=(), sigma_gyro=-1.0, sigma_accel=-1.0, dt=1e-3, mode=0, first_filter=0):
        f8 = lambda a: np.ascontiguousarray(a, dtype=np.float64)
        i8 = lambda a: np.ascontiguousarray(a, dtype=np.int64)
        self.keep = []
        self.c = capi.Synth()
        self.c.seed, self.c.first_filter, self.c.mode = int(seed) & (2 ** 64 - 1), int(first_filter), int(mode)
        im, ist = f8(imu_mean).reshape(-1, 6), i8(imu_step).reshape(-1)
        assert im.shape[0] == ist.shape[0]
        self.keep += [im, ist]
        self.c.imu_mean, self.c.imu_step, self.c.imu_rows = im.ctypes.data, ist.ctypes.data, im.shape[0]
        self.c.sigma_gyro, self.c.sigma_accel, self.c.dt = float(sigma_gyro), float(sigma_accel), float(dt)
        self.sarr = (capi.SynthStream * max(1, len(streams)))()
        self.shapes = []
        for k, st in enumerate(streams):
            mean = f8(st["mean"])
            rows, m = mean.shape
            step = i8(st["step"]).reshape(-1)
            assert step.shape[0] == rows
            d = self.sarr[k]
            d.m, d.channel, d.rows = m, int(st["channel"]), rows
            d.mean, d.step = mean.ctypes.data, step.ctypes.data
            sig = np.broadcast_to(np.asarray(st["sigma"], dtype=np.float64), (m,))
            for a in range(m):
                d.sigma[a] = float(sig[a])
            self.keep += [mean, step]
            mq = st.get("mean_quat")
            d.has_orientation = int(mq is not None)
            if mq is not None:
                mq = f8(mq).reshape(rows, 4)
                d.mean_quat, d.channel_rot = mq.ctypes.data, int(st["channel_rot"])
                sr = np.broadcast_to(np.asarray(st["sigma_rot"], dtype=np.float64), (3,))
                for a in range(3):
                    d.sigma_rot[a] = float(sr[a])
                self.keep.append(mq)
            self.shapes.append((rows, m, mq is not None))
        self.c.n_streams = len(streams)
        self.c.streams = self.sarr


def _shared_or_row_R(R, m, rows, s):
    """(r_mode, column-major host copy) of a stream's R given as m x m (shared) or [rows][m][m] (per row)."""
    R = np.asarray(R, dtype=np.float64)
    if R.ndim == 3:
        if R.shape != (rows, m, m):
            raise ValueError(f"stream {s}: a per-row R must be [rows][{m}][{m}] = {(rows, m, m)}, got {R.shape}")
        return capi.R_PER_ROW_FULL, np.ascontiguousarray(R.transpose(0, 2, 1))
    return capi.R_SHARED_FULL, np.ascontiguousarray(R.reshape(m, m).T)


_QUAT_NAMES = ("quat_w", "quat_x", "quat_y", "quat_z")


def record_fields(vec=(), quat=False, loglik=False, cov_diag=()):
    """rbis_record_t::fields of a record set: state vector entries `vec` (indices 0..20), the quaternion (w, x, y, z), the
    log-likelihood and the covariance diagonal entries P(i, i) for i in `cov_diag`."""
    mask = 0
    for i in list(vec) + list(cov_diag):
        if not 0 <= int(i) < capi.NUM_STATES:
            raise ValueError(f"state index {i} outside [0, {capi.NUM_STATES})")
    for i in vec:
        mask |= 1 << int(i)
    if quat:
        mask |= 0xF << 21
    if loglik:
        mask |= 1 << 25
    for i in cov_diag:
        mask |= 1 << (26 + int(i))
    return mask


def record_cov_blocks(blocks=()):
    """rbis_record_t::cov_blocks of covariance block numbers 0..6 (state indices 3b..3b+2: omega, v, chi, p, a, gyro bias,
    accel bias)."""
    cb = 0
    for b in blocks:
        if not 0 <= int(b) < capi.REC_BLOCKS:
            raise ValueError(f"covariance block {b} outside [0, {capi.REC_BLOCKS})")
        cb |= 1 << int(b)
    return cb


def record_layout(mask, cov_blocks=()):
    """Names of the fields of a record row in output order: 'vec<i>', 'quat_w' .. 'quat_z', 'loglik', 'cov_diag<i>', then
    'cov<i>_<j>' for P(i, j), i <= j, of the covariance blocks `cov_blocks` (block numbers 0..6), packed column by column."""
    mask = int(mask)
    cb = record_cov_blocks(cov_blocks)
    if mask < 0 or mask >> capi.REC_FIELDS or (mask == 0 and cb == 0):
        raise ValueError(f"record fields {mask:#x}: need a non-empty set of bits 0..{capi.REC_FIELDS - 1} or covariance blocks")
    names = []
    for f in range(capi.REC_FIELDS):
        if mask >> f & 1:
            names.append(f"vec{f}" if f < 21 else _QUAT_NAMES[f - 21] if f < 25 else "loglik" if f == 25 else f"cov_diag{f - 26}")
    idx = [3 * b + c for b in range(capi.REC_BLOCKS) if cb >> b & 1 for c in range(3)]
    for jj, j in enumerate(idx):
        names.extend(f"cov{i}_{j}" for i in idx[:jj + 1])
    return names


def innovation_layout(m, fields):
    """Names of the entries of an innovation row in output order: 'nis', then 'y<a>' and 's<a>' (S(a,a)) for a < m, then
    'applied', as the RBIS_INNOV_* bits of `fields` select them (INNOV_APPLIED only beside one of the others)."""
    m, fields = int(m), int(fields)
    if not 1 <= m <= capi.MAX_MEAS:
        raise ValueError(f"innovation m = {m} outside 1..{capi.MAX_MEAS}")
    values = capi.INNOV_NIS | capi.INNOV_Y | capi.INNOV_S_DIAG
    if fields <= 0 or not fields & values or fields & ~(values | capi.INNOV_APPLIED):
        raise ValueError(f"innovation fields {fields:#x}: need a non-empty set of INNOV_NIS / INNOV_Y / INNOV_S_DIAG, optionally "
                         "with INNOV_APPLIED")
    names = ["nis"] if fields & capi.INNOV_NIS else []
    if fields & capi.INNOV_Y:
        names += [f"y{a}" for a in range(m)]
    if fields & capi.INNOV_S_DIAG:
        names += [f"s{a}" for a in range(m)]
    if fields & capi.INNOV_APPLIED:
        names.append("applied")
    return names


def make_ops(entries):
    """entries: iterable of (kind, stream, row, utime, dt) -> structured numpy op array."""
    entries = list(entries)
    ops = np.zeros(len(entries), dtype=OP_DTYPE)
    for i, (kind, stream, row, utime, dt) in enumerate(entries):
        ops[i] = (kind, stream, row, utime, dt)
    return ops


class RBISBatch:
    """An ensemble of N RBIS filters on one GPU (rbis_batch_t)."""

    def __init__(self, n_filters, device=0, g_val=9.8, chi_tol=1e-6, ctor_folds_chi=True, renormalize_quat=False,
                 snapshot_slots=0, launch_groups=0, dense_only=False, mapping=0, lane_filters_per_cta=0, piece_ops=0,
                 synth_materialize=False):
        self.lib = capi.load()
        cfg = capi.Config()
        self.lib.rbis_default_config(C.byref(cfg))
        cfg.g_val, cfg.chi_tol = float(g_val), float(chi_tol)
        cfg.ctor_folds_chi, cfg.renormalize_quat = int(bool(ctor_folds_chi)), int(bool(renormalize_quat))
        cfg.snapshot_slots, cfg.device = int(snapshot_slots), int(device)
        cfg.launch_groups = int(launch_groups)
        cfg.dense_only = int(bool(dense_only))
        cfg.lane_filters_per_cta = int(lane_filters_per_cta)
        cfg.piece_ops = int(piece_ops)
        cfg.synth_materialize = int(bool(synth_materialize))
        cfg.mapping = int(mapping)  # lanes per filter: 0 automatic, 1 lane-per-filter kernels, 2/4/8/16 warp-group kernels
        self.h = C.c_void_p()
        capi.check(self.lib.rbis_batch_create(C.byref(self.h), int(n_filters), C.byref(cfg)))
        self.N = int(n_filters)
        self.device = int(device)
        self._keep = []  # arrays that must outlive asynchronous calls

    def close(self):
        if getattr(self, "h", None) is not None and self.h.value:
            self.lib.rbis_batch_destroy(self.h)
            self.h = C.c_void_p()
        self._keep = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- state ----
    def set_state(self, vec, quat, cov=None, loglik=None, utime=0):
        N = self.N
        pv, m1 = _ptr(vec, (21, N), "vec")
        pq, m2 = _ptr(quat, (4, N), "quat")
        pc, m3 = _ptr(cov, (441, N), "cov")
        pl, m4 = _ptr(loglik, (N,), "loglik")
        mem = _common_mem([m1, m2, m3, m4], "set_state")
        capi.check(self.lib.rbis_batch_set_state(self.h, pv, pq, pc, pl, int(utime), mem))

    def get_state(self, cov=True):
        """-> (vec [21][N], quat [4][N], cov [441][N] or None, loglik [N], utime) as numpy."""
        N = self.N
        vec = np.empty((21, N)); quat = np.empty((4, N)); ll = np.empty(N)
        P = np.empty((441, N)) if cov else None
        ut = C.c_int64(0)
        capi.check(self.lib.rbis_batch_get_state(self.h, vec.ctypes.data, quat.ctypes.data,
                                                 P.ctypes.data if cov else None, ll.ctypes.data, C.byref(ut),
                                                 capi.MEM_HOST))
        return vec, quat, P, ll, ut.value

    def get_state_into(self, vec=None, quat=None, cov=None, loglik=None):
        """Device or host destination arrays (torch CUDA tensors or numpy); any may be None."""
        N = self.N
        pv, m1 = _ptr(vec, (21, N), "vec")
        pq, m2 = _ptr(quat, (4, N), "quat")
        pc, m3 = _ptr(cov, (441, N), "cov")
        pl, m4 = _ptr(loglik, (N,), "loglik")
        mem = _common_mem([m1, m2, m3, m4], "get_state_into")
        ut = C.c_int64(0)
        capi.check(self.lib.rbis_batch_get_state(self.h, pv, pq, pc, pl, C.byref(ut), mem))
        return ut.value

    def get_snapshot(self, slot, cov=True):
        """Ring slot -> (vec [21][N], quat [4][N], cov [441][N] or None, loglik [N]) as numpy."""
        N = self.N
        vec = np.empty((21, N)); quat = np.empty((4, N)); ll = np.empty(N)
        P = np.empty((441, N)) if cov else None
        capi.check(self.lib.rbis_batch_get_snapshot(self.h, int(slot), vec.ctypes.data, quat.ctypes.data,
                                                    P.ctypes.data if cov else None, ll.ctypes.data, capi.MEM_HOST))
        return vec, quat, P, ll

    def smooth_backward(self, next_pred_slot, next_slot, steps, dt):
        """rbis_batch_smooth_backward; steps: structured array of smoother.STEP_DTYPE in execution order."""
        steps = np.ascontiguousarray(steps)
        assert steps.dtype.itemsize == 16
        capi.check(self.lib.rbis_batch_smooth_backward(self.h, int(next_pred_slot), int(next_slot), len(steps),
                                                       steps.ctypes.data, float(dt)))

    def notch_configure(self, notch_freq, fs=1000.0, n_stages=3, cols=None):
        """Accelerometer notch cascade of InsHandler::doFilter (MSE/sensor_handlers.cpp:29-41,155-162)."""
        self._notch_cols = int(self.N if cols is None else cols)
        capi.check(self.lib.rbis_batch_notch_configure(self.h, float(notch_freq), float(fs), int(n_stages), self._notch_cols))

    def notch_filter(self, imu):
        """Filters the accelerometer rows of imu [rows][6][cols] in place (numpy host array or torch CUDA tensor)."""
        rows = int(imu.shape[0])
        ptr, mem = _ptr(imu, (rows, 6, self._notch_cols), "imu")
        capi.check(self.lib.rbis_batch_notch_filter(self.h, ptr, rows, mem))

    def set_filter(self, n, vec, quat, cov, loglik=0.0):
        vec = np.ascontiguousarray(vec, dtype=np.float64); quat = np.ascontiguousarray(quat, dtype=np.float64)
        cov = np.ascontiguousarray(cov, dtype=np.float64)
        assert vec.size == 21 and quat.size == 4 and cov.size == 441
        capi.check(self.lib.rbis_batch_set_filter(self.h, int(n), vec.ctypes.data, quat.ctypes.data, cov.ctypes.data,
                                                  float(loglik)))

    def get_filter(self, n):
        vec = np.empty(21); quat = np.empty(4); cov = np.empty(441); ll = C.c_double(0)
        capi.check(self.lib.rbis_batch_get_filter(self.h, int(n), vec.ctypes.data, quat.ctypes.data, cov.ctypes.data,
                                                  C.byref(ll)))
        return vec, quat, cov, ll.value

    def set_process_noise(self, q_gyro, q_accel, q_gyro_bias, q_accel_bias):
        args = [q_gyro, q_accel, q_gyro_bias, q_accel_bias]
        if all(np.isscalar(a) for a in args):
            capi.check(self.lib.rbis_batch_set_process_noise(self.h, *[float(a) for a in args]))
            return
        ptrs, mems = [], []
        for a in args:
            if np.isscalar(a):
                a = np.full(self.N, float(a))
            p, m = _ptr(a, (self.N,), "q")
            ptrs.append(p); mems.append(m)
        capi.check(self.lib.rbis_batch_set_process_noise_per_filter(self.h, *ptrs, _common_mem(mems, "process noise")))

    # ---- single updates ----
    def ins_step(self, gyro, accel, dt, utime=0):
        pg, m1 = _ptr(gyro, (3, self.N), "gyro")
        pa, m2 = _ptr(accel, (3, self.N), "accel")
        capi.check(self.lib.rbis_batch_ins_step(self.h, pg, pa, float(dt), int(utime), _common_mem([m1, m2], "ins_step")))

    def indexed_update(self, idx, z, R, utime=0, quat=None, per_filter_diag=False):
        m = len(idx)
        idx_a = (C.c_int32 * m)(*[int(i) for i in idx])
        pz, m1 = _ptr(z, (m, self.N), "z")
        if per_filter_diag:
            pr, m2 = _ptr(R, (m, self.N), "R")
        else:
            R = np.ascontiguousarray(np.asarray(R, dtype=np.float64).reshape(m, m).T)  # column-major m x m
            pr, m2 = R.ctypes.data, None
        r_mode = capi.R_PER_FILTER_DIAG if per_filter_diag else capi.R_SHARED_FULL
        if quat is None:
            mem = _common_mem([m1, m2], "indexed_update")
            capi.check(self.lib.rbis_batch_indexed_update(self.h, m, idx_a, pz, pr, r_mode, int(utime), mem))
        else:
            pq, m3 = _ptr(quat, (4, self.N), "quat")
            mem = _common_mem([m1, m2, m3], "indexed_orient_update")
            capi.check(self.lib.rbis_batch_indexed_orient_update(self.h, m, idx_a, pz, pq, pr, r_mode, int(utime), mem))

    # ---- shared input columns ----
    def set_column_map(self, which, col_map=None, cols=0):
        """Filter n reads column col_map[n] of the IMU array (which = -1) or of measurement stream `which`;
        those arrays then have `cols` columns instead of N.  col_map=None restores the identity."""
        k = int(which) + 1
        if not hasattr(self, "_cols"):
            self._cols = {}
        if col_map is None:
            capi.check(self.lib.rbis_batch_set_column_map(self.h, int(which), None, 0))
            self._cols.pop(k, None)
            return
        m = np.ascontiguousarray(col_map, dtype=np.int32)
        if m.shape != (self.N,):
            raise ValueError("col_map must be int32[N]")
        capi.check(self.lib.rbis_batch_set_column_map(self.h, int(which), m.ctypes.data, int(cols)))
        self._cols[k] = int(cols)

    def _ncols(self, which):
        return getattr(self, "_cols", {}).get(int(which) + 1, self.N)

    # ---- fused program ----
    def prepare_fused(self, ops, imu=None, streams=()):
        """Marshal one rbis_batch_run_fused call once (ctypes structures, pointer checks); run_prepared() then costs one foreign
        call.  The arrays are referenced by the returned object and must keep their contents until the launch has run."""
        if not (isinstance(ops, np.ndarray) and ops.dtype == OP_DTYPE):
            ops = make_ops(ops)
        ops = np.ascontiguousarray(ops)
        mems, f32s = [], []
        p_imu, imu_rows = None, 0
        if imu is not None:
            if imu.ndim != 3 or tuple(imu.shape[1:]) != (6, self._ncols(-1)):
                raise ValueError("imu must be [rows][6][N] ([rows][6][cols] under a column map)")
            p_imu, mm, f = _ptr_rows(imu, "imu")
            imu_rows = int(imu.shape[0]); mems.append(mm); f32s.append(f)
        sarr = (capi.Stream * max(1, len(streams)))()
        keep = [ops, imu]
        for s, st in enumerate(streams):
            m = len(st.idx)
            d = sarr[s]
            d.m, d.has_orientation, d.sensor_id = m, int(st.quat is not None), st.sensor_id
            d.flags = capi.STREAM_SKIP_NAN_ROWS if st.skip_nan_rows else 0
            d.r_mode = capi.R_PER_FILTER_DIAG if st.per_filter_diag else capi.R_SHARED_FULL
            for a, i in enumerate(st.idx):
                d.idx[a] = i
            if st.z.ndim != 3 or tuple(st.z.shape[1:]) != (m, self._ncols(s)):
                raise ValueError(f"stream {s}: z must be [rows][{m}][N] (cols under a column map)")
            d.rows = int(st.z.shape[0])
            d.z, mm, f = _ptr_rows(st.z, "z"); mems.append(mm); f32s.append(f)
            if st.quat is not None:
                if tuple(st.quat.shape) != (d.rows, 4, self._ncols(s)):
                    raise ValueError(f"stream {s}: quat must be [rows][4][N] (cols under a column map)")
                d.quat, mm, f = _ptr_rows(st.quat, "quat"); mems.append(mm); f32s.append(f)
            if st.per_filter_diag:
                d.R, mm = _ptr(st.R, (m, self.N), "R"); mems.append(mm)
            else:
                d.r_mode, R = _shared_or_row_R(st.R, m, d.rows, s)
                keep.append(R)
                d.R = R.ctypes.data
            keep.append(st)
        mem = _common_mem(mems, "run_fused")
        if f32s and any(f32s):
            if not all(f32s):
                raise ValueError("run_fused: the sensor rows (imu, z, quat) of one call must all be float64 or all float32")
            mem |= capi.MEM_F32_ROWS   # float rows: widened exactly on the device (rbis_mem_t)
        return (len(ops), ops.ctypes.data_as(C.POINTER(capi.Op)), p_imu, imu_rows, len(streams), sarr, mem, keep)

    # ---- records ----
    def set_record(self, out, fields, cov_blocks=()):
        """Record set of the RBIS_OP_RECORD ops of later fused calls (rbis_batch_set_record).  out: float64 [rows][k][N], k the number
        of entries of record_layout(fields, cov_blocks), a CUDA tensor (written in place) or a PINNED CPU tensor or array (filled by an
        asynchronous copy); its rows are valid after wait(record()) or synchronize().  cov_blocks: covariance block numbers 0..6
        recorded after the fields.  Does not synchronise."""
        fields = int(fields)
        cb = record_cov_blocks(cov_blocks)
        if 0 <= fields < 1 << capi.REC_FIELDS and (fields or cb):
            k = len(record_layout(fields, cov_blocks))
            if out.ndim != 3 or tuple(out.shape[1:]) != (k, self.N):
                raise ValueError(f"record output must be [rows][{k}][{self.N}], got {tuple(out.shape)}")
        p, mem = _ptr(out, None, "out")
        rec = capi.Record()
        rec.fields, rec.out, rec.rows, rec.mem, rec.cov_blocks = fields, p, int(out.shape[0]), mem, cb
        capi.check(self.lib.rbis_batch_set_record(self.h, C.byref(rec)))
        # the previous buffer may still be written by enqueued calls: held until the next synchronize()
        self._pending_keep = getattr(self, "_pending_keep", [])
        self._pending_keep.append(getattr(self, "_record_out", None))
        self._record_out = out

    def clear_record(self):
        capi.check(self.lib.rbis_batch_set_record(self.h, None))

    # ---- innovation sets ----
    def set_innovations(self, stream, out, m, fields=capi.INNOV_NIS | capi.INNOV_Y | capi.INNOV_S_DIAG):
        """Innovation set of stream slot `stream` (rbis_batch_set_innovations): every MEAS op on that stream of later fused calls
        writes row op.row of out, a CUDA float64 tensor [rows][k][N] with the entries of innovation_layout(m, fields).  Valid after
        wait(record()) or synchronize().  Does not synchronise."""
        try:
            k = len(innovation_layout(m, fields))
        except ValueError:
            k = None  # the library refuses it with its own message
        if k is not None and (out.ndim != 3 or tuple(out.shape[1:]) != (k, self.N)):
            raise ValueError(f"innovation output must be [rows][{k}][{self.N}], got {tuple(out.shape)}")
        p, _ = _ptr(out, None, "out")
        spec = capi.Innovation()
        spec.fields, spec.m, spec.out, spec.rows = int(fields), int(m), p, int(out.shape[0])
        capi.check(self.lib.rbis_batch_set_innovations(self.h, int(stream), C.byref(spec)))
        self._pending_keep = getattr(self, "_pending_keep", [])
        self._innov_out = getattr(self, "_innov_out", {})
        self._pending_keep.append(self._innov_out.get(int(stream)))
        self._innov_out[int(stream)] = out

    def clear_innovations(self, stream):
        capi.check(self.lib.rbis_batch_set_innovations(self.h, int(stream), None))

    # ---- NIS gates ----
    def set_nis_gate(self, stream, nis_max=float("inf"), per_filter=None):
        """NIS gate of stream slot `stream` (rbis_batch_set_nis_gate): in later fused calls every filter rejects a row of that
        stream whose prior NIS exceeds its threshold, and then keeps its values as for a missing row.  per_filter: a CUDA float64
        tensor [N] of thresholds (filter n uses per_filter[n]) or None for nis_max everywhere.  Does not synchronise."""
        gate = capi.NisGate()
        gate.nis_max = float(nis_max)
        gate.nis_max_per_filter = None
        if per_filter is not None:
            if tuple(per_filter.shape) != (self.N,):
                raise ValueError(f"per-filter NIS thresholds must be [{self.N}], got {tuple(per_filter.shape)}")
            gate.nis_max_per_filter, _ = _ptr(per_filter, None, "per_filter")
        capi.check(self.lib.rbis_batch_set_nis_gate(self.h, int(stream), C.byref(gate)))
        # the previous array may still be read by enqueued calls: held until the next synchronize()
        self._pending_keep = getattr(self, "_pending_keep", [])
        self._gate_thr = getattr(self, "_gate_thr", {})
        self._pending_keep.append(self._gate_thr.get(int(stream)))
        self._gate_thr[int(stream)] = per_filter

    def clear_nis_gate(self, stream):
        capi.check(self.lib.rbis_batch_set_nis_gate(self.h, int(stream), None))

    def stats_innovations_enqueue(self, stream, first_row, out_chunks, out_totals=None, chunk=1024):
        """Statistics of innovation rows first_row .. first_row + n_rows - 1 of stream slot `stream`'s innovation set on the
        statistics side stream (rbis_batch_stats_innovations_enqueue): out_chunks a PINNED host array [n_rows][n_chunks][96] (n_rows
        is its first dimension), out_totals a PINNED host array [n_rows][96] or None.  Returns the ticket to wait() for."""
        n_rows = int(out_chunks.shape[0])
        n_chunks = (self.N + chunk - 1) // chunk
        po, _ = _ptr(out_chunks, (n_rows, n_chunks, capi.NUM_STATS), "out_chunks")
        pt, _ = _ptr(out_totals, (n_rows, capi.NUM_STATS), "out_totals")
        nch, t = C.c_int64(0), C.c_int32(0)
        capi.check(self.lib.rbis_batch_stats_innovations_enqueue(self.h, int(stream), int(first_row), n_rows, int(chunk), po, pt,
                                                                 C.byref(nch), C.byref(t)))
        return t.value

    def run_prepared(self, prep):
        capi.check(self.lib.rbis_batch_run_fused(self.h, *prep[:7]))

    def run_fused(self, ops, imu=None, streams=()):
        """ops: structured array (OP_DTYPE) or iterable of (kind, stream, row, utime, dt)."""
        prep = self.prepare_fused(ops, imu, streams)
        # host inputs must outlive their asynchronous copies (rbis_batch.h, "lifetime of host inputs"): every call's arrays are
        # held until a later synchronize() / wait() has shown that the copies ran
        self._pending_keep = getattr(self, "_pending_keep", [])
        self._pending_keep.append(prep)
        if len(self._pending_keep) > 64:   # bounded: beyond this many un-synchronised calls, drain
            self.synchronize()
        self.run_prepared(prep)

    def run_fused_synth(self, ops, streams, spec):
        """rbis_batch_run_fused_synth: `streams` carry idx / R (z, quat ignored: MeasStream(idx, None, R, quat=True/None)),
        `spec` (SynthSpec) the noise-free rows; per-filter input rows are generated on the device."""
        if not (isinstance(ops, np.ndarray) and ops.dtype == OP_DTYPE):
            ops = make_ops(ops)
        ops = np.ascontiguousarray(ops)
        sarr = (capi.Stream * max(1, len(streams)))()
        keep = [ops, spec]
        for s, st in enumerate(streams):
            m = len(st.idx)
            d = sarr[s]
            d.m, d.has_orientation, d.sensor_id = m, int(st.quat is not None), st.sensor_id
            d.flags = capi.STREAM_SKIP_NAN_ROWS if st.skip_nan_rows else 0   # rejected by the library: rows are drawn, not read
            d.r_mode = capi.R_PER_FILTER_DIAG if st.per_filter_diag else capi.R_SHARED_FULL
            for a, i in enumerate(st.idx):
                d.idx[a] = i
            if st.per_filter_diag:
                d.R, mm = _ptr(st.R, (m, self.N), "R")
                if mm != capi.MEM_DEVICE:
                    raise ValueError("run_fused_synth: a per-filter R must be a device tensor")
            else:
                d.r_mode, R = _shared_or_row_R(st.R, m, int(spec.sarr[s].rows) if s < spec.c.n_streams else 0, s)
                keep.append(R)
                d.R = R.ctypes.data
            keep.append(st)
        self._pending_keep = getattr(self, "_pending_keep", [])
        self._pending_keep.append(keep)
        capi.check(self.lib.rbis_batch_run_fused_synth(self.h, len(ops), ops.ctypes.data_as(C.POINTER(capi.Op)), len(streams), sarr,
                                                       C.byref(spec.c)))

    def synthesize(self, spec):
        """rbis_batch_synthesize -> dict(imu [rows][6][N], z [list], quat [list]) as torch CUDA tensors (what the device draws)."""
        import torch

        dev = torch.device("cuda", self.device)
        imu = torch.empty((int(spec.c.imu_rows), 6, self.N), dtype=torch.float64, device=dev)
        zs, qs = [], []
        zp = (C.c_void_p * max(1, len(spec.shapes)))()
        qp = (C.c_void_p * max(1, len(spec.shapes)))()
        for k, (rows, m, orient) in enumerate(spec.shapes):
            zs.append(torch.empty((rows, m, self.N), dtype=torch.float64, device=dev))
            qs.append(torch.empty((rows, 4, self.N), dtype=torch.float64, device=dev) if orient else None)
            zp[k] = zs[k].data_ptr()
            qp[k] = qs[k].data_ptr() if orient else None
        capi.check(self.lib.rbis_batch_synthesize(self.h, C.byref(spec.c), imu.data_ptr(), zp, qp))
        self.synchronize()
        return dict(imu=imu, z=zs, quat=qs)

    def synchronize(self):
        capi.check(self.lib.rbis_batch_synchronize(self.h))
        self._pending_keep = []   # every copy enqueued so far has run

    @property
    def launch_count(self):
        return int(self.lib.rbis_batch_launch_count(self.h))

    @property
    def last_kernel_variant(self):
        """0 dense, 2 decoupled (rbis_batch_config_t::dense_only), +1 with correlated-row chunks, +4 input rows drawn in the
        kernel, +8 a program with RBIS_OP_RECORD ops, +16 * lanes per filter for the warp-group kernels, +512 a stream that skips
        NaN rows (MeasStream skip_nan_rows), +2048 (with +512) a NIS gate or INNOV_APPLIED (set_nis_gate); -1 before any launch."""
        return int(self.lib.rbis_batch_last_kernel_variant(self.h))

    @property
    def cuda_stream(self):
        return int(self.lib.rbis_batch_stream(self.h) or 0)

    # ---- statistics ----
    def stats(self, truth_vec, truth_quat, chunk=1024, per_filter_truth=False, want_per_filter=False):
        """-> (chunks [n_chunks][96], per_filter [23][N] or None).  See rbis_batch_stats."""
        N = self.N
        n_chunks = (N + chunk - 1) // chunk
        out = np.zeros((n_chunks, capi.NUM_STATS))
        pf = np.empty((23, N)) if want_per_filter else None
        if per_filter_truth:
            pv, m1 = _ptr(truth_vec, (21, N), "truth_vec"); pq, m2 = _ptr(truth_quat, (4, N), "truth_quat")
            mem = _common_mem([m1, m2], "stats")
            if mem != capi.MEM_HOST:
                raise ValueError("stats: per-filter truth must be host arrays in this wrapper")
        else:
            tv = np.ascontiguousarray(truth_vec, dtype=np.float64); tq = np.ascontiguousarray(truth_quat, dtype=np.float64)
            assert tv.size == 21 and tq.size == 4
            pv, pq, mem = tv.ctypes.data, tq.ctypes.data, capi.MEM_HOST
        nch = C.c_int64(0)
        capi.check(self.lib.rbis_batch_stats(self.h, pv, pq, int(per_filter_truth), int(chunk), out.ctypes.data,
                                             C.byref(nch), pf.ctypes.data if want_per_filter else None, mem))
        assert nch.value == n_chunks
        return out, pf


    def stats_allreduce(self, comm, truth_vec, truth_quat, first_chunk, total_chunks, chunk=1024, want_table=False):
        """rbis_batch_stats_allreduce: statistics of a sharded ensemble through a raw NCCL communicator (pronto_b200.nccl.
        Communicator, or None for a single process) -> (totals [96], table [total_chunks][96] or None)."""
        tv = np.ascontiguousarray(truth_vec, dtype=np.float64); tq = np.ascontiguousarray(truth_quat, dtype=np.float64)
        assert tv.size == 21 and tq.size == 4
        totals = np.zeros(capi.NUM_STATS)
        table = np.zeros((int(total_chunks), capi.NUM_STATS)) if want_table else None
        capi.check(self.lib.rbis_batch_stats_allreduce(self.h, comm.handle if comm is not None else None, tv.ctypes.data, tq.ctypes.data,
                                                       int(chunk), int(first_chunk), int(total_chunks), totals.ctypes.data,
                                                       table.ctypes.data if want_table else None))
        return totals, table

    def stats_enqueue(self, truth_vec, truth_quat, out_chunks, chunk=1024):
        """Asynchronous statistics into a PINNED host array [n_chunks][96]; valid after wait(record())."""
        tv = np.ascontiguousarray(truth_vec, dtype=np.float64); tq = np.ascontiguousarray(truth_quat, dtype=np.float64)
        assert tv.size == 21 and tq.size == 4
        n_chunks = (self.N + chunk - 1) // chunk
        po, _ = _ptr(out_chunks, (n_chunks, capi.NUM_STATS), "out_chunks")
        nch = C.c_int64(0)
        capi.check(self.lib.rbis_batch_stats_enqueue(self.h, tv.ctypes.data, tq.ctypes.data, int(chunk), po, C.byref(nch)))

    def stats_snapshot_enqueue(self, slot, truth_vec, truth_quat, out_chunks, chunk=1024):
        """Statistics over snapshot slot `slot` on a side stream (rbis_batch_stats_snapshot_enqueue) into a PINNED host array
        [n_chunks][96]; returns the ticket to wait() for.  The fused launches that follow do not wait for it."""
        tv = np.ascontiguousarray(truth_vec, dtype=np.float64); tq = np.ascontiguousarray(truth_quat, dtype=np.float64)
        assert tv.size == 21 and tq.size == 4
        n_chunks = (self.N + chunk - 1) // chunk
        po, _ = _ptr(out_chunks, (n_chunks, capi.NUM_STATS), "out_chunks")
        nch, t = C.c_int64(0), C.c_int32(0)
        capi.check(self.lib.rbis_batch_stats_snapshot_enqueue(self.h, int(slot), tv.ctypes.data, tq.ctypes.data, int(chunk), po, C.byref(nch),
                                                              C.byref(t)))
        return t.value

    def stats_records_enqueue(self, first_row, truth_vec, truth_quat, out_chunks, out_totals=None, chunk=1024):
        """Statistics of record rows first_row .. first_row + n_rows - 1 of the current (device) record set on the statistics side
        stream (rbis_batch_stats_records_enqueue): truth_vec [n_rows][21], truth_quat [n_rows][4]; out_chunks a PINNED host array
        [n_rows][n_chunks][96], out_totals a PINNED host array [n_rows][96] or None.  Returns the ticket to wait() for."""
        tv = np.ascontiguousarray(truth_vec, dtype=np.float64).reshape(-1, 21)
        tq = np.ascontiguousarray(truth_quat, dtype=np.float64).reshape(-1, 4)
        n_rows = tv.shape[0]
        if tq.shape[0] != n_rows:
            raise ValueError(f"truth_vec has {n_rows} rows, truth_quat {tq.shape[0]}")
        n_chunks = (self.N + chunk - 1) // chunk
        po, _ = _ptr(out_chunks, (n_rows, n_chunks, capi.NUM_STATS), "out_chunks")
        pt, _ = _ptr(out_totals, (n_rows, capi.NUM_STATS), "out_totals")
        nch, t = C.c_int64(0), C.c_int32(0)
        capi.check(self.lib.rbis_batch_stats_records_enqueue(self.h, int(first_row), n_rows, tv.ctypes.data, tq.ctypes.data, int(chunk),
                                                             po, pt, C.byref(nch), C.byref(t)))
        return t.value

    def record(self):
        t = C.c_int32(0)
        capi.check(self.lib.rbis_batch_record(self.h, C.byref(t)))
        return t.value

    def wait(self, ticket):
        capi.check(self.lib.rbis_batch_wait(self.h, int(ticket)))


def filter_states_from_record(row, fields, cov_blocks=range(7), utime=0, first=0, count=None):
    """filter_state_t messages (capi.FilterState array) of filters first .. first+count-1 of one record row already on the host
    (rbis_record_filter_states): row [k][N] with fields 0..24 and all seven covariance blocks; the messages are those
    rbis_batch_get_filter_states writes for the same state."""
    row = np.ascontiguousarray(row, dtype=np.float64)
    if row.ndim != 2:
        raise ValueError(f"record row must be [k][N], got {row.shape}")
    n = row.shape[1]
    count = n - int(first) if count is None else int(count)
    out = (capi.FilterState * max(1, count))()
    capi.check(capi.load().rbis_record_filter_states(int(fields), record_cov_blocks(cov_blocks), row.ctypes.data, n, int(utime), int(first),
                                                     count, out))
    return out


def reduce_chunks(chunks):
    """Fixed ascending-order sum of chunk partials -> [96] (rbis_stats_reduce_chunks)."""
    chunks = np.ascontiguousarray(chunks, dtype=np.float64)
    out = np.zeros(capi.NUM_STATS)
    capi.check(capi.load().rbis_stats_reduce_chunks(chunks.ctypes.data, chunks.shape[0], out.ctypes.data))
    return out


def measure_fp64_peak(device=0, iters=2000):
    """-> (dfma_tflops, dmma_tflops) measured on `device`."""
    a, b = C.c_double(0), C.c_double(0)
    capi.check(capi.load().rbis_measure_fp64_peak(int(device), int(iters), C.byref(a), C.byref(b)))
    return a.value, b.value
