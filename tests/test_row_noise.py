"""Measurement streams whose noise covariance changes from row to row (RBIS_R_PER_ROW_FULL, include/rbis_batch.h).

Every RBISIndexed[PlusOrientation]Measurement of the reference carries its own measurement_cov
(MSE/rbis_update_interface.hpp:90-96,111-117): leg odometry switches between a certain and an uncertain R
(LegOdoCommon), indexed_measurement_t carries R_effective per message.  A per-row stream must compute what the
oracle computes with each event's own R, and -- where the same program can be written with shared-R streams --
the same bits as that program."""
import ctypes as C
import os
import struct
import subprocess

import numpy as np
import pytest

from pronto_b200 import MeasStream, RBISBatch, SynthSpec, capi, synth
from pronto_b200.parity import max_errors

from common import nominal_q, scenario

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NTHREADS = min(16, os.cpu_count() or 1)
STEP_TOL = 1e-9
TRAJ_TOL = 1e-6
QL_IDX = [8, 9, 10, 11]      # quick-lock: yaw + position (quick_lock.cpp:132)
YAW_IDX = [17, 8]            # a yaw lock with the measured orientation
MIX_IDX = [3, 4, 5, 9, 10, 11]
R_CERTAIN = synth.NOMINAL["r_vxyz"] ** 2
R_UNCERTAIN = (5 * synth.NOMINAL["r_vxyz"]) ** 2


def legodo_R(rows, seed=3, frac=0.1, uncertain=R_UNCERTAIN):
    """[rows][3][3] leg-odometry R switching between certain and uncertain on a seeded pattern; and the pattern."""
    unc = np.random.default_rng(seed).random(rows) < frac
    R = np.empty((rows, 3, 3))
    R[:] = np.eye(3) * R_CERTAIN
    R[unc] = np.eye(3) * uncertain
    return R, unc


def spd(rng, m, scale):
    A = rng.normal(size=(m, m))
    return (A @ A.T / m + np.eye(m)) * scale


def _rel_ll(a, b):
    return float(np.max(np.abs(a - b) / np.maximum(1.0, np.abs(b))))


def _equal(a, b):
    for x, y in zip(a[:4], b[:4]):
        assert np.array_equal(x, y)


def extra_streams(sc, k_ql=(), k_yaw=(), k_mix=(), seed=7):
    """Quick-lock (full 4x4 R per row), yaw-lock (orientation) and mixed diagonal / correlated streams at the given steps of
    the scenario, as streams 2, 3, 4 after leg odometry (0) and pose (1); returns (streams as dicts, arrival-ordered events)."""
    rng = np.random.default_rng(seed)
    truth, st = sc["truth"], sc["st"]
    N = sc["vec"].shape[1]
    noise = lambda *s: rng.normal(size=s)
    out = []
    k = np.asarray(k_ql, dtype=int)
    z = np.zeros((len(k), 4, N))
    z[:, 0] = 0.02 * noise(len(k), N)
    z[:, 1:] = truth["p"][k][:, :, None] + 0.05 * noise(len(k), 3, N)
    out.append(dict(idx=QL_IDX, z=z, R=np.stack([spd(rng, 4, 0.05 ** 2) for _ in k]) if len(k) else np.zeros((0, 4, 4))))
    k = np.asarray(k_yaw, dtype=int)
    z = np.zeros((len(k), 2, N))
    z[:, 0] = synth.NOMINAL["bg"][2] + 1e-4 * noise(len(k), N)
    q = np.ascontiguousarray(np.repeat(truth["quat"][k][:, :, None], N, axis=2))
    out.append(dict(idx=YAW_IDX, z=z, quat=q, R=np.stack([spd(rng, 2, (0.001 + 0.002 * (i % 3)) ** 2) for i in range(len(k))])
                    if len(k) else np.zeros((0, 2, 2))))
    k = np.asarray(k_mix, dtype=int)
    z = np.zeros((len(k), 6, N))
    z[:, 0:3] = truth["v"][k][:, :, None] + 0.1 * noise(len(k), 3, N)
    z[:, 3:6] = truth["p"][k][:, :, None] + 0.05 * noise(len(k), 3, N)
    Rm = []
    for i in range(len(k)):   # every other row couples v_y with p_x: the union plan cuts [3] [4 5 9 10] [11]
        R = np.diag([0.1 ** 2] * 3 + [0.05 ** 2] * 3) * (1 + i % 4)
        if i % 2:
            R[1, 4] = R[4, 1] = 0.5 * np.sqrt(R[1, 1] * R[4, 4])
        Rm.append(R)
    out.append(dict(idx=MIX_IDX, z=z, R=np.stack(Rm) if Rm else np.zeros((0, 6, 6))))
    at = {}
    for s, ks in ((2, k_ql), (3, k_yaw), (4, k_mix)):
        for r, kk in enumerate(ks):
            at.setdefault(int(kk), []).append((s, r))
    ev = []
    for e in st["events"]:
        ev.append(e)
        if e[0] == capi.OP_IMU:
            kk = int(st["steps"][e[2]])
            for s, r in at.get(kk, []):
                ev.append((capi.OP_MEAS, s, r, e[3], 0.0))
    return out, ev


def base_streams(st, R_lego=None, R_pose=None):
    return [dict(idx=synth.LEGODO_IDX, z=st["legodo"], R=st["R_legodo"] if R_lego is None else R_lego),
            dict(idx=synth.POSE_IDX, z=st["pose_z"], R=st["R_pose"] if R_pose is None else R_pose, quat=st["pose_q"])]


def run_oracle(run_ensemble, vec, quat, cov, loglik, utime0, imu, streams, events, **kw):
    """The CPU oracle's ensemble runner with per-row R: every row of a [rows][m][m] stream becomes a stream of its own whose
    shared R is that row's, so the event on row r builds its update object with R row r, as the reference does."""
    split, where = [], {}
    for s, d in enumerate(streams):
        R = np.asarray(d["R"])
        if R.ndim != 3:
            where[s] = len(split)
            split.append(d)
            continue
        for r in range(d["z"].shape[0]):
            where[(s, r)] = len(split)
            one = dict(idx=d["idx"], z=d["z"][r:r + 1], R=R[r])
            if d.get("quat") is not None:
                one["quat"] = d["quat"][r:r + 1]
            split.append(one)
    ev = []
    for e in events:
        if e[0] == capi.OP_MEAS:
            e = (e[0], where[e[1]], e[2]) + tuple(e[3:]) if e[1] in where else (e[0], where[(e[1], e[2])], 0) + tuple(e[3:])
        ev.append(e)
    return run_ensemble(vec, quat, cov, loglik, utime0, nominal_q(), imu, split, ev, **kw)


def gpu(streams):
    return [MeasStream(d["idx"], d["z"], d["R"], quat=d.get("quat")) for d in streams]


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
def _message(idx, R, z=None):
    msg = capi.IndexedMeasurement()
    m = len(idx)
    msg.measured_dim, msg.measured_cov_dim = m, m * m
    for a in range(m):
        msg.z_indices[a] = idx[a]
        msg.z_effective[a] = 0.0 if z is None else z[a]
    for e, v in enumerate(np.asarray(R).T.reshape(-1)):   # Map<MatrixXd>(R_effective, m, m): column-major
        msg.R_effective[e] = v
    return msg


def test_sequence_of_messages_becomes_one_stream(rbis_lib):
    lib = rbis_lib
    rng = np.random.default_rng(2)
    K = 5
    Rs = [spd(rng, 4, 0.01) for _ in range(K)]
    msgs = (capi.IndexedMeasurement * K)(*[_message(QL_IDX, Rs[0]) for _ in range(K)])
    st, Rout = capi.Stream(), np.full(K * 16, np.nan)
    capi.check(lib.rbis_stream_from_indexed_measurements(msgs, K, C.byref(st), Rout.ctypes.data))
    assert (st.m, st.has_orientation, st.r_mode, st.sensor_id, st.rows) == (4, 0, capi.R_SHARED_FULL, 5, K)
    assert list(st.idx)[:4] == QL_IDX and st.R == Rout.ctypes.data
    assert np.array_equal(Rout.reshape(K, 4, 4).transpose(0, 2, 1), np.stack([Rs[0]] * K))
    msgs = (capi.IndexedMeasurement * K)(*[_message(QL_IDX, R) for R in Rs])
    capi.check(lib.rbis_stream_from_indexed_measurements(msgs, K, C.byref(st), Rout.ctypes.data))
    assert (st.m, st.r_mode, st.rows) == (4, capi.R_PER_ROW_FULL, K) and st.R == Rout.ctypes.data
    assert np.array_equal(Rout.reshape(K, 4, 4).transpose(0, 2, 1), np.stack(Rs))   # [rows][m][m], each column-major
    # one message is a one-row shared stream; mismatches are rejected
    capi.check(lib.rbis_stream_from_indexed_measurements(msgs, 1, C.byref(st), Rout.ctypes.data))
    assert (st.r_mode, st.rows) == (capi.R_SHARED_FULL, 1)
    for bad in ("idx", "dim", "cov_dim"):
        msgs = (capi.IndexedMeasurement * K)(*[_message(QL_IDX, R) for R in Rs])
        if bad == "idx":
            msgs[3].z_indices[2] = 17
        elif bad == "dim":
            msgs[2] = _message([8, 9, 10], Rs[2][:3, :3])
        else:
            msgs[4].measured_cov_dim = 15
        assert lib.rbis_stream_from_indexed_measurements(msgs, K, C.byref(st), Rout.ctypes.data) == -1, bad
    assert lib.rbis_stream_from_indexed_measurements(msgs, 0, C.byref(st), Rout.ctypes.data) == -1


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mapping", [1, 4])
@pytest.mark.parametrize("dense_only", [False, True])
def test_equal_rows_run_as_the_shared_stream(mapping, dense_only):
    """A per-row stream whose rows all equal one R: same chunk plan, kernel variant and bits as that R shared."""
    N, T = 300, 220
    sc = scenario(N, T)
    st = sc["st"]
    extra, ev = extra_streams(sc, k_ql=range(7, T, 13))
    ql_R = extra[0]["R"][0]
    shared = base_streams(st) + [dict(extra[0], R=ql_R)]
    rows = lambda d: np.ascontiguousarray(np.broadcast_to(d["R"], (d["z"].shape[0],) + np.shape(d["R"])))
    per_row = [dict(d, R=rows(d)) for d in shared]
    outs = []
    for streams in (shared, per_row):
        with RBISBatch(N, mapping=mapping, dense_only=dense_only) as b:
            b.set_process_noise(*nominal_q())
            b.set_state(sc["vec"], sc["quat"], sc["cov"])
            b.run_fused(ev, imu=st["imu"], streams=gpu(streams))
            outs.append((b.get_state(), b.last_kernel_variant))
    _equal(outs[0][0], outs[1][0])
    assert outs[0][1] == outs[1][1] and (outs[0][1] & 1) == 1 and bool(outs[0][1] & 2) == (not dense_only)
    assert outs[0][1] >> 4 == (mapping if mapping > 1 else 0)


def _split_by_R(st, unc):
    """The program MavStateEstimator built before per-row streams: one shared-R stream per distinct leg-odometry R."""
    lego = st["legodo"]
    rows = {False: np.flatnonzero(~unc), True: np.flatnonzero(unc)}
    pos = {int(r): (1 if unc[r] else 0, int(np.searchsorted(rows[bool(unc[r])], r))) for r in range(len(unc))}
    streams = [dict(idx=synth.LEGODO_IDX, z=np.ascontiguousarray(lego[rows[False]]), R=np.eye(3) * R_CERTAIN),
               dict(idx=synth.LEGODO_IDX, z=np.ascontiguousarray(lego[rows[True]]), R=np.eye(3) * R_UNCERTAIN),
               dict(idx=synth.POSE_IDX, z=st["pose_z"], R=st["R_pose"], quat=st["pose_q"])]
    ev = []
    for e in st["events"]:
        if e[0] == capi.OP_MEAS:
            e = (e[0],) + (pos[e[2]] if e[1] == 0 else (2, e[2])) + tuple(e[3:])
        ev.append(e)
    return streams, ev


@pytest.mark.gpu
@pytest.mark.parametrize("mapping", [1, 4])
def test_switching_legodo_R_equals_one_stream_per_distinct_R(mapping):
    N, T = 500, 400
    sc = scenario(N, T)
    st = sc["st"]
    R_lego, unc = legodo_R(st["legodo"].shape[0], frac=0.3)
    assert 0 < unc.sum() < len(unc)
    two, ev2 = _split_by_R(st, unc)
    outs = []
    for streams, ev in ((base_streams(st, R_lego), st["events"]), (two, ev2)):
        with RBISBatch(N, mapping=mapping) as b:
            b.set_process_noise(*nominal_q())
            b.set_state(sc["vec"], sc["quat"], sc["cov"])
            b.run_fused(ev, imu=st["imu"], streams=gpu(streams))
            outs.append((b.get_state(), b.last_kernel_variant))
    _equal(outs[0][0], outs[1][0])
    assert outs[0][1] == outs[1][1]


@pytest.mark.gpu
@pytest.mark.parametrize("mapping", [1, 4])
def test_correlated_row_varying_R_matches_oracle_event_by_event(oracle, mapping):
    """Quick-lock with a different full 4x4 R per row, a yaw lock [17, 8] with orientation and a stream whose rows mix
    diagonal and correlated R (one union chunk plan), each event its own launch, against the oracle's head after it."""
    N, T = 48, 160
    sc = scenario(N, T)
    st = sc["st"]
    extra, ev = extra_streams(sc, k_ql=range(4, T, 9), k_yaw=range(6, T, 14), k_mix=range(2, T, 7))
    R_lego, _ = legodo_R(st["legodo"].shape[0], frac=0.3)
    streams = base_streams(st, R_lego) + extra
    ref = run_oracle(oracle.run_ensemble, sc["vec"], sc["quat"], sc["cov"], None, 0, st["imu"], streams, ev, n_threads=NTHREADS, trace=True)
    worst = dict(vec=0.0, quat=0.0, cov=0.0, ll=0.0)
    g = gpu(streams)
    with RBISBatch(N, mapping=mapping) as b:
        b.set_process_noise(*nominal_q())
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        for e, event in enumerate(ev):
            b.run_fused([event], imu=st["imu"], streams=g)
            gv, gq, gP, gll, _ = b.get_state()
            err = max_errors(gv, gq, gP, ref["trace_vec"][e], ref["trace_quat"][e], ref["trace_cov"][e])
            err["ll"] = _rel_ll(gll, ref["trace_loglik"][e])
            for k in worst:
                worst[k] = max(worst[k], err[k])
        assert b.last_kernel_variant & 1
        step_by_step = b.get_state()
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        b.run_fused(ev, imu=st["imu"], streams=g)
        _equal(step_by_step, b.get_state())
    assert max(worst.values()) <= STEP_TOL, worst


@pytest.mark.gpu
def test_long_trajectory_with_switching_legodo_R_matches_oracle(oracle):
    """Config-3 shape (1 kHz IMU, 500 Hz leg odometry, 10 Hz pose) for 30 s in chunks of 2,000 steps, leg-odometry R
    switching per row: <= 1e-6 at the end."""
    N, T, CH = 16, 30_000, 2_000
    truth = synth.truth_trajectory(T)
    sc0 = scenario(N, 1, truth=truth)
    rv, rq, rP, rll = sc0["vec"].copy(), sc0["quat"].copy(), sc0["cov"].copy(), np.zeros(N)
    with RBISBatch(N) as b:
        b.set_process_noise(*nominal_q())
        b.set_state(sc0["vec"], sc0["quat"], sc0["cov"])
        for k0 in range(0, T, CH):
            st = synth.make_streams(truth, N, k0, CH)
            R_lego, _ = legodo_R(st["legodo"].shape[0], seed=k0)
            streams = base_streams(st, R_lego)
            b.run_fused(st["events"], imu=st["imu"], streams=gpu(streams))
            ref = run_oracle(oracle.run_ensemble, rv, rq, rP, rll, k0 * 1000, st["imu"], streams, st["events"], n_threads=NTHREADS)
            rv, rq, rP, rll = ref["vec"], ref["quat"], ref["cov"], ref["loglik"]
            b.synchronize()
        gv, gq, gP, gll, _ = b.get_state()
    e = max_errors(gv, gq, gP, rv, rq, rP)
    assert max(e.values()) <= TRAJ_TOL and _rel_ll(gll, rll) <= TRAJ_TOL, e


@pytest.mark.gpu
def test_delayed_pose_fixes_replay_each_row_with_its_own_R(oracle):
    from pronto_b200.schedule import program_from_arrivals

    N, T, LAT = 96, 400, 50
    sc = scenario(N, T)
    st = sc["st"]
    R_lego, _ = legodo_R(st["legodo"].shape[0], frac=0.3)
    n_pose = st["pose_z"].shape[0]
    R_pose = np.stack([st["R_pose"] * (1.0 + 3.0 * (r % 2)) for r in range(n_pose)])
    streams = base_streams(st, R_lego, R_pose)
    ev = st["events"]
    pose = [e for e in ev if e[0] == 1 and e[1] == 1]
    arrivals, pending = [], list(pose)
    for e in ev:
        if e[0] == 1 and e[1] == 1:
            continue
        arrivals.append(e)
        while pending and e[0] == 0 and e[3] >= pending[0][3] + LAT * 1000:
            arrivals.append(pending.pop(0))
    arrivals += pending
    ref = run_oracle(oracle.run_ensemble, sc["vec"], sc["quat"], sc["cov"], None, 0, st["imu"], streams, arrivals, n_threads=NTHREADS)
    ops, cnt = program_from_arrivals(arrivals, snapshot_slots=3, snapshot_period_us=100_000, snapshot_phase_us=1000)
    assert cnt["rewinds"] == len(pose) and cnt["discarded"] == 0
    with RBISBatch(N, snapshot_slots=3) as b:
        b.set_process_noise(*nominal_q())
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        b.run_fused(ops, imu=st["imu"], streams=gpu(streams))
        gv, gq, gP, gll, _ = b.get_state()
    e = max_errors(gv, gq, gP, ref["vec"], ref["quat"], ref["cov"])
    assert max(e.values()) <= STEP_TOL and _rel_ll(gll, ref["loglik"]) <= STEP_TOL, e


@pytest.mark.gpu
@pytest.mark.parametrize("mapping,materialize", [(1, False), (1, True), (4, False)])
def test_synthesised_inputs_with_per_row_R(mapping, materialize):
    """rbis_batch_run_fused_synth with a per-row leg-odometry stream, rows drawn in the kernel or materialised first, equals
    rbis_batch_synthesize + rbis_batch_run_fused to the bit."""
    N, T = 300, 220
    sc = scenario(N, T, tumbling=True)
    st = sc["st"]
    d = synth.synth_spec_inputs(sc["truth"], 0, T)
    R_lego, _ = legodo_R(len(d["streams"][0]["step"]), frac=0.3)
    with RBISBatch(N, mapping=mapping, synth_materialize=materialize) as b:
        b.set_process_noise(*nominal_q())
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        spec = SynthSpec(synth.SEED, d["imu_mean"], d["imu_step"], d["streams"], mode=1)
        b.run_fused_synth(st["events"], [MeasStream(synth.LEGODO_IDX, None, R_lego), MeasStream(synth.POSE_IDX, None, st["R_pose"], quat=True)],
                          spec)
        assert bool(b.last_kernel_variant & 4) == (not materialize)
        a = b.get_state()
        rows = b.synthesize(spec)
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        b.run_fused(st["events"], imu=rows["imu"], streams=[MeasStream(synth.LEGODO_IDX, rows["z"][0], R_lego),
                                                            MeasStream(synth.POSE_IDX, rows["z"][1], st["R_pose"], quat=rows["quat"][1])])
        _equal(a, b.get_state())


@pytest.mark.gpu
def test_tables_outlive_grouped_pieced_unsynchronised_calls():
    """Launch groups, programs cut into pieces and many consecutive calls without a synchronise, every call with tables of its
    own: same bits as one group with a synchronise after every call (a launch that read a later call's table would differ)."""
    N, T, CH = 4000, 240, 20
    sc = scenario(N, T)
    outs = []
    for groups, piece, sync in ((1, 0, True), (4, 8, False), (6, 0, False)):
        with RBISBatch(N, launch_groups=groups, mapping=1, piece_ops=piece) as b:
            b.set_process_noise(*nominal_q())
            b.set_state(sc["vec"], sc["quat"], sc["cov"])
            for k0 in range(0, T, CH):
                st = synth.make_streams(sc["truth"], N, k0, CH)
                R_lego, _ = legodo_R(st["legodo"].shape[0], seed=k0, frac=0.5, uncertain=(1 + k0 / 40) * R_UNCERTAIN)
                extra, ev = extra_streams(dict(sc, st=st), k_ql=range(k0 + 1, k0 + CH, 3), seed=k0)
                b.run_fused(ev, imu=st["imu"], streams=gpu(base_streams(st, R_lego) + extra[:1]))
                if sync:
                    b.synchronize()
            outs.append(b.get_state())
    _equal(outs[0], outs[1])
    _equal(outs[0], outs[2])


@pytest.mark.gpu
def test_column_maps_and_float_rows_with_per_row_R():
    from pronto_b200.batch import make_ops

    C_, G_, T = 16, 8, 120
    N = C_ * G_
    sc = scenario(C_, T)
    st = sc["st"]
    cmap = (np.arange(N) % C_).astype(np.int32)
    ex = lambda a: np.ascontiguousarray(a[..., cmap])
    R_lego, _ = legodo_R(st["legodo"].shape[0], frac=0.3)
    extra, ev = extra_streams(sc, k_ql=range(3, T, 8))
    ops = make_ops(ev)
    outs = []
    for mapped in (True, False):
        with RBISBatch(N) as b:
            b.set_process_noise(*nominal_q())
            b.set_state(ex(sc["vec"]), ex(sc["quat"]), ex(sc["cov"]))
            if mapped:
                for w in (-1, 0, 1, 2):
                    b.set_column_map(w, cmap, C_)
            f = (lambda a: a) if mapped else ex
            b.run_fused(ops, imu=f(st["imu"]), streams=[MeasStream(synth.LEGODO_IDX, f(st["legodo"]), R_lego),
                                                        MeasStream(synth.POSE_IDX, f(st["pose_z"]), st["R_pose"], quat=f(st["pose_q"])),
                                                        MeasStream(QL_IDX, f(extra[0]["z"]), extra[0]["R"])])
            outs.append(b.get_state())
    _equal(outs[0], outs[1])
    # float rows: widened exactly on the device
    f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)
    w = lambda a: f32(a).astype(np.float64)
    outs = []
    for conv in (f32, w):
        with RBISBatch(C_) as b:
            b.set_process_noise(*nominal_q())
            b.set_state(sc["vec"], sc["quat"], sc["cov"])
            b.run_fused(ops, imu=conv(st["imu"]), streams=[MeasStream(synth.LEGODO_IDX, conv(st["legodo"]), R_lego),
                                                           MeasStream(synth.POSE_IDX, conv(st["pose_z"]), st["R_pose"], quat=conv(st["pose_q"])),
                                                           MeasStream(QL_IDX, conv(extra[0]["z"]), extra[0]["R"])])
            outs.append(b.get_state())
    _equal(outs[0], outs[1])


@pytest.mark.gpu
def test_errors_leave_the_ensemble_unchanged():
    N, T = 64, 40
    sc = scenario(N, T)
    st = sc["st"]
    extra, ev = extra_streams(sc, k_ql=range(1, T, 4))
    bad = np.array(extra[0]["R"])
    k = 3
    bad[k, 0, 1] = bad[k, 1, 0] = 2.0 * np.sqrt(bad[k, 0, 0] * bad[k, 1, 1])   # indefinite 2x2 minor in row k
    with RBISBatch(N) as b:
        b.set_process_noise(*nominal_q())
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        b.run_fused(ev[:10], imu=st["imu"], streams=gpu(base_streams(st) + [extra[0]]))
        before = b.get_state()
        with pytest.raises(capi.RBISError, match=f"stream 2, stream row {k}:.*not positive definite"):
            b.run_fused(ev[10:], imu=st["imu"], streams=gpu(base_streams(st) + [dict(extra[0], R=bad)]))
        _equal(before, b.get_state())
        assert b.get_state()[4] == before[4]
        # R == NULL with rows > 0
        prep = b.prepare_fused(ev[10:], imu=st["imu"], streams=gpu(base_streams(st) + [extra[0]]))
        prep[5][2].R = None
        with pytest.raises(capi.RBISError, match="z and R are required"):
            b.run_prepared(prep)
        # a single update has one R
        idx = (C.c_int32 * 3)(*synth.LEGODO_IDX)
        z = np.ascontiguousarray(st["legodo"][0])
        R = np.ascontiguousarray(np.stack([np.eye(3) * R_CERTAIN] * 2))
        q = np.ascontiguousarray(st["pose_q"][0])
        assert b.lib.rbis_batch_indexed_update(b.h, 3, idx, z.ctypes.data, R.ctypes.data, capi.R_PER_ROW_FULL, 0, capi.MEM_HOST) == -1
        assert b"fused programs only" in b.lib.rbis_last_error()
        assert b.lib.rbis_batch_indexed_orient_update(b.h, 3, idx, z.ctypes.data, q.ctypes.data, R.ctypes.data, capi.R_PER_ROW_FULL, 0,
                                                      capi.MEM_HOST) == -1
        _equal(before, b.get_state())
        # the Python mirror checks the row count of a per-row R
        with pytest.raises(ValueError, match="per-row R"):
            b.run_fused(ev, imu=st["imu"], streams=[MeasStream(synth.LEGODO_IDX, st["legodo"], np.stack([np.eye(3)] * 2))])


# ------------------------------------------------------------------------------------------------
# C++ shim (include/rbis_batch.hpp)
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def shim_exe(rbis_lib):
    build = os.path.join(ROOT, "tests", "cpp", "_build")
    os.makedirs(build, exist_ok=True)
    exe = os.path.join(build, "shim_replay_row_noise")
    libdir = os.path.join(ROOT, "pronto_b200", "lib")
    subprocess.check_call(["g++", "-std=c++14", "-O2", "-Wall", "-Wextra", "-o", exe, os.path.join(ROOT, "tests", "cpp", "shim_replay.cpp"),
                           f"-L{libdir}", "-lrbis_b200", f"-Wl,-rpath,{libdir}"])
    return exe


@pytest.mark.gpu
def test_shim_switching_and_per_message_R_match_oracle_without_extra_flushes(shim_exe, tmp_path):
    """LegOdoCommon-style switching leg-odometry R plus 20 indexed measurements (quick-lock) with distinct correlated R, pose
    fixes 50 steps late: the shim's replays hold up to 13 distinct R, which used to cost a synchronised flush per 8; now
    every roll-forward is one launch, and the head matches the oracle's multimap history."""
    from oracle import oracle_api

    N, T, LAT = 40, 300, 50
    sc = scenario(N, T)
    st = sc["st"]
    extra, ev = extra_streams(sc, k_ql=range(150, 250, 5))
    assert extra[0]["z"].shape[0] == 20
    R_lego, unc = legodo_R(st["legodo"].shape[0], frac=0.3)
    streams = base_streams(st, R_lego) + extra[:1]
    pose = [e for e in ev if e[0] == 1 and e[1] == 1]
    arrivals, pending = [], list(pose)
    for e in ev:
        if e[0] == 1 and e[1] == 1:
            continue
        arrivals.append(e)
        while pending and e[0] == 0 and e[3] >= pending[0][3] + LAT * 1000:
            arrivals.append(pending.pop(0))
    arrivals += pending
    q = nominal_q()
    p_in, p_out = str(tmp_path / "in.bin"), str(tmp_path / "out.bin")
    with open(p_in, "wb") as f:
        f.write(struct.pack("<6q", N, 0, 10_000_000, 3, 100_000, len(arrivals)))
        for a in (sc["vec"], sc["quat"], sc["cov"]):
            f.write(np.ascontiguousarray(a, dtype=np.float64).tobytes())
        for kind, s, row, utime, dt in arrivals:
            if kind == 0:
                f.write(struct.pack("<2q", 0, utime))
                f.write(struct.pack("<5d", dt, *q))
                f.write(np.ascontiguousarray(st["imu"][row]).tobytes())
                continue
            d = streams[s]
            R = np.asarray(d["R"])
            R = R[row] if R.ndim == 3 else R
            f.write(struct.pack("<2q", 2 if d.get("quat") is not None else 1, utime))
            f.write(struct.pack(f"<{1 + len(d['idx'])}q", len(d["idx"]), *d["idx"]))
            f.write(np.ascontiguousarray(R.T).tobytes())
            f.write(np.ascontiguousarray(d["z"][row]).tobytes())
            if d.get("quat") is not None:
                f.write(np.ascontiguousarray(d["quat"][row]).tobytes())
    r = subprocess.run([shim_exe, p_in, p_out], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    raw = np.fromfile(p_out, dtype=np.float64)
    n0 = 21 * N + 4 * N + 441 * N + N
    gv, gq, gP, gll = np.split(raw[:n0], [21 * N, 25 * N, 466 * N])
    launches, dropped = np.frombuffer(raw[n0:n0 + 2].tobytes(), dtype=np.int64)
    ref = run_oracle(oracle_api.run_ensemble, sc["vec"], sc["quat"], sc["cov"], None, 0, st["imu"], streams, arrivals, n_threads=NTHREADS)
    e = max_errors(gv.reshape(21, N), gq.reshape(4, N), gP.reshape(441, N), ref["vec"], ref["quat"], ref["cov"])
    assert max(e.values()) < STEP_TOL, e
    assert _rel_ll(gll, ref["loglik"]) < STEP_TOL
    assert dropped == 0 and launches == len(arrivals)   # one launch per roll-forward, no flush for a new R
