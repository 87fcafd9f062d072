"""Records (RBIS_OP_RECORD, rbis_batch_set_record in include/rbis_batch.h): chosen per-filter fields written from inside a fused
program, so that a replay's trajectory (the head poses MSE/lcm_front_end.cpp:144-166 publishes, or the error and 1-sigma
envelopes of a Monte-Carlo study) comes out of ONE launch.  A record row must hold, bit for bit, what a snapshot at the same
program position holds in those fields, and recording must not change what the program computes."""
import ctypes as C
import os

import numpy as np
import pytest

from pronto_b200 import MeasStream, RBISBatch, SynthSpec, capi, record_fields, record_layout, synth
from pronto_b200.parity import max_errors

from common import gpu_streams, nominal_q, oracle_streams, random_ensemble, scenario

NTHREADS = min(16, os.cpu_count() or 1)
STEP_TOL = 1e-9
ALL = (1 << capi.REC_FIELDS) - 1
POSE = record_fields(vec=(9, 10, 11), quat=True)
# every output position != its field index, so the lanes of a warp group share the stores differently than with ALL; covariance
# diagonals on chip and of omega / a
SPARSE = record_fields(vec=(4, 9, 10, 11), quat=True, loglik=True, cov_diag=(1, 8, 13, 19))
DIAG = [i + 21 * i for i in range(21)]


def fields_of(vec, quat, cov, ll, *_):
    """[47][N]: the record fields of a state as get_state / get_snapshot return it (full covariance [441][N])."""
    return np.concatenate([vec, quat, ll[None], cov[DIAG]])


def select(full, mask):
    """Rows of a [.., 47, N] array that a record set with `mask` holds, in output order."""
    return full[..., [f for f in range(capi.REC_FIELDS) if mask >> f & 1], :]


def device_out(rows, mask, N):
    import torch

    return torch.full((rows, bin(mask).count("1"), N), float("nan"), dtype=torch.float64, device="cuda")


def pinned_out(rows, mask, N):
    import torch

    return torch.full((rows, bin(mask).count("1"), N), float("nan"), dtype=torch.float64).pin_memory()


def as_np(t):
    return t.cpu().numpy() if hasattr(t, "cpu") else np.asarray(t)


def rec_op(row):
    return (capi.OP_RECORD, 0, int(row), 0, 0.0)


def _equal(a, b):
    for x, y in zip(a[:4], b[:4]):
        assert np.array_equal(x, y)


def _setup(b, sc):
    b.set_process_noise(*nominal_q())
    b.set_state(sc["vec"], sc["quat"], sc["cov"])


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
def test_record_fields_and_layout_round_trip(rbis_lib):
    assert hasattr(rbis_lib, "rbis_batch_set_record")
    assert record_layout(POSE) == ["vec9", "vec10", "vec11", "quat_w", "quat_x", "quat_y", "quat_z"]
    assert record_fields(vec=range(21), quat=True, loglik=True, cov_diag=range(21)) == ALL
    assert record_layout(record_fields(loglik=True, cov_diag=[0, 20])) == ["loglik", "cov_diag0", "cov_diag20"]
    rng = np.random.default_rng(1)
    for _ in range(200):
        vec = sorted(set(rng.integers(0, 21, rng.integers(0, 6)).tolist()))
        diag = sorted(set(rng.integers(0, 21, rng.integers(0, 6)).tolist()))
        quat, ll = bool(rng.integers(2)), bool(rng.integers(2))
        if not (vec or diag or quat or ll):
            continue
        mask = record_fields(vec=vec, quat=quat, loglik=ll, cov_diag=diag)
        names = record_layout(mask)
        assert len(names) == bin(mask).count("1")
        back = record_fields(vec=[int(n[3:]) for n in names if n.startswith("vec")], quat="quat_w" in names, loglik="loglik" in names,
                             cov_diag=[int(n[8:]) for n in names if n.startswith("cov_diag")])
        assert back == mask
    for bad in (0, 1 << capi.REC_FIELDS, -1):
        with pytest.raises(ValueError):
            record_layout(bad)
    with pytest.raises(ValueError):
        record_fields(vec=[21])


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("tumbling", [False, True])
def test_every_event_recorded_in_one_launch(oracle, tumbling):
    """All 47 fields after every event of one program, in ONE launch: equal to get_state after running each event as its own
    launch, and within the per-step gate of the oracle's head after the same event."""
    N, T = 150, 220
    sc = scenario(N, T, tumbling=tumbling)
    st = sc["st"]
    ev = st["events"]
    ref = oracle.run_ensemble(sc["vec"], sc["quat"], sc["cov"], None, 0, nominal_q(), st["imu"], oracle_streams(st), ev,
                              n_threads=NTHREADS, trace=True)
    prog = []
    for e, event in enumerate(ev):
        prog += [event, rec_op(e)]
    out = device_out(len(ev), ALL, N)
    with RBISBatch(N) as b:
        _setup(b, sc)
        streams = gpu_streams(st)
        steps = []
        for event in ev:
            b.run_fused([event], imu=st["imu"], streams=streams)
            steps.append(fields_of(*b.get_state()))
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        b.set_record(out, ALL)
        b.run_fused(prog, imu=st["imu"], streams=streams)
        assert b.last_kernel_variant & 8
        b.synchronize()
        assert b.get_state()[4] == ev[-1][3]   # RECORD ops leave the ensemble's utime alone
    rec = as_np(out)
    assert np.array_equal(rec, np.stack(steps))
    worst = dict(vec=0.0, quat=0.0, diag=0.0, ll=0.0)
    for e in range(len(ev)):
        err = max_errors(rec[e, 0:21], rec[e, 21:25], None, ref["trace_vec"][e], ref["trace_quat"][e], None)
        d_ref = np.asarray(ref["trace_cov"][e])[DIAG]
        err["diag"] = float(np.max(np.abs(rec[e, 26:] - d_ref) / np.where(d_ref > 0, d_ref, 1.0)))
        ll_ref = np.asarray(ref["trace_loglik"][e])
        err["ll"] = float(np.max(np.abs(rec[e, 25] - ll_ref) / np.maximum(1.0, np.abs(ll_ref))))
        for k in worst:
            worst[k] = max(worst[k], err[k])
    assert max(worst.values()) <= STEP_TOL, worst


def _rewind_program(N=64, T=200):
    """Delayed pose fixes replayed through SNAPSHOT / RESTORE rewinds, per-row leg-odometry R, quick-lock [8..11] with a dense
    per-row R and a yaw lock [17, 8] with orientation (one-row and correlated chunks).  -> (scenario, gpu streams, ops, the op
    indices after which to record: the start, after every restore and every 7th op)."""
    from pronto_b200.schedule import program_from_arrivals
    from test_row_noise import base_streams, extra_streams, gpu, legodo_R

    sc = scenario(N, T)
    st = sc["st"]
    extra, ev = extra_streams(sc, k_ql=range(4, T, 9), k_yaw=range(6, T, 14))
    R_lego, _ = legodo_R(st["legodo"].shape[0], frac=0.3)
    streams = gpu(base_streams(st, R_lego) + extra[:2])
    pose = [e for e in ev if e[0] == capi.OP_MEAS and e[1] == 1]
    arrivals, pending = [], list(pose)
    for e in ev:
        if e[0] == capi.OP_MEAS and e[1] == 1:
            continue
        arrivals.append(e)
        while pending and e[0] == capi.OP_IMU and e[3] >= pending[0][3] + 30_000:
            arrivals.append(pending.pop(0))
    arrivals += pending
    ops, cnt = program_from_arrivals(arrivals, snapshot_slots=3, snapshot_period_us=50_000, snapshot_phase_us=1000)
    assert cnt["rewinds"] > 0
    ops = [tuple(o.tolist()) for o in ops]
    at = sorted({-1} | {i for i, o in enumerate(ops) if o[0] == capi.OP_RESTORE} | set(range(3, len(ops), 7)))
    return sc, streams, ops, at


def _insert(ops, at, extra):
    """ops with extra(j) (a list of ops) inserted after op at[j] (-1: before the first op)."""
    out = list(extra(0)) if at and at[0] == -1 else []
    j = 1 if out else 0
    for i, o in enumerate(ops):
        out.append(o)
        if j < len(at) and at[j] == i:
            out += extra(j)
            j += 1
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("mapping,dense_only", [(1, False), (1, True), (4, False), (4, True)])
def test_records_equal_snapshots_at_the_same_positions(mapping, dense_only):
    sc, streams, ops, at = _rewind_program()
    st, N = sc["st"], sc["vec"].shape[1]
    R = len(at)
    prog = _insert(ops, at, lambda j: [rec_op(j), (capi.OP_SNAPSHOT, 0, 3 + j, 0, 0.0)])
    out = device_out(R, ALL, N)
    with RBISBatch(N, snapshot_slots=3 + R, mapping=mapping, dense_only=dense_only) as b:
        _setup(b, sc)
        b.set_record(out, ALL)
        b.run_fused(prog, imu=st["imu"], streams=streams)
        assert b.last_kernel_variant & 9 == 9   # correlated chunks, records
        assert bool(b.last_kernel_variant & 2) == (not dense_only)
        snaps = np.stack([fields_of(*b.get_snapshot(3 + j)) for j in range(R)])
    assert np.array_equal(as_np(out), snaps)


@pytest.mark.gpu
@pytest.mark.parametrize("mapping", [1, 4])
def test_records_do_not_perturb_the_filter(mapping):
    sc, streams, ops, at = _rewind_program()
    st, N = sc["st"], sc["vec"].shape[1]
    out = device_out(len(at), ALL, N)
    with RBISBatch(N, snapshot_slots=3, mapping=mapping) as b:
        _setup(b, sc)
        b.run_fused(ops, imu=st["imu"], streams=streams)
        plain, v_plain = b.get_state(), b.last_kernel_variant
        _setup(b, sc)
        b.set_record(out, ALL)
        b.run_fused(_insert(ops, at, lambda j: [rec_op(j)]), imu=st["imu"], streams=streams)
        recorded, v_rec = b.get_state(), b.last_kernel_variant
        # a record set alone changes nothing: programs without RECORD ops run the kernels they ran before
        _setup(b, sc)
        b.run_fused(ops, imu=st["imu"], streams=streams)
        again, v_again = b.get_state(), b.last_kernel_variant
    _equal(plain, recorded)
    _equal(plain, again)
    assert plain[4] == recorded[4]
    assert not v_plain & 8 and v_again == v_plain and v_rec == v_plain | 8
    assert not np.isnan(as_np(out)).any()


@pytest.mark.gpu
def test_record_bits_do_not_depend_on_mapping_or_kernel_variant():
    sc, streams, ops, at = _rewind_program(N=300, T=120)
    st, N = sc["st"], sc["vec"].shape[1]
    prog = _insert(ops, at, lambda j: [rec_op(j)])
    cfgs = [dict(mapping=1, lane_filters_per_cta=t) for t in (384, 256, 128)] + [dict(mapping=1, dense_only=True)] + \
        [dict(mapping=g) for g in (2, 4, 8, 16)] + [dict(mapping=g, dense_only=True) for g in (2, 16)]
    recs = []
    for cfg in cfgs:
        with RBISBatch(N, snapshot_slots=3, **cfg) as b:
            got = []
            for mask in (ALL, SPARSE):   # the sparse set: how the lanes of a group share the stores
                out = device_out(len(at), mask, N)
                _setup(b, sc)
                b.set_record(out, mask)
                b.run_fused(prog, imu=st["imu"], streams=streams)
                b.synchronize()
                assert b.last_kernel_variant & 8
                got.append(as_np(out))
        assert np.array_equal(got[1], select(got[0], SPARSE)), cfg
        recs.append(got[0])
    for cfg, r in zip(cfgs[1:], recs[1:]):
        assert np.array_equal(r, recs[0]), cfg
    # a coupled ensemble (dense covariances) runs the dense kernels of every mapping
    vec, quat, cov = random_ensemble(N, seed=5)
    ev = scenario(N, 60)["st"]
    prog = []
    for e, event in enumerate(ev["events"]):
        prog += [event] + ([rec_op(e // 5)] if e % 5 == 4 else [])
    rows = len(ev["events"]) // 5
    recs = []
    for mapping in (1, 2, 4, 8, 16):
        out = device_out(rows, ALL, N)
        with RBISBatch(N, mapping=mapping) as b:
            b.set_process_noise(*nominal_q())
            b.set_state(vec, quat, cov)
            b.set_record(out, ALL)
            b.run_fused(prog, imu=ev["imu"], streams=gpu_streams(ev))
            b.synchronize()
            assert not b.last_kernel_variant & 2 and b.last_kernel_variant & 8
        recs.append(as_np(out))
    for r in recs[1:]:
        assert np.array_equal(r, recs[0])


@pytest.mark.gpu
def test_records_across_launch_groups_and_pieces_and_to_pinned_host_memory():
    """A program of several 64-op pieces with records on both sides of every piece boundary, on an ensemble large enough for the
    automatic launch groups (40,000 filters: 157 dense CTAs on 148 SMs): automatic groups and launch_groups = 1 give the same
    bits, and a pinned host output receives exactly the device output."""
    N, T = 40_000, 80
    sc = scenario(N, T)
    st = sc["st"]
    ev = st["events"]
    prog, rows = [], 0
    for e, event in enumerate(ev):
        prog.append(event)
        if e % 5 == 0:
            prog.append(rec_op(rows))
            rows += 1
    assert len(prog) >= 2 * 64
    outs = []
    for groups, where in ((1, device_out), (0, device_out), (0, pinned_out)):
        out = where(rows, ALL, N)
        with RBISBatch(N, mapping=1, launch_groups=groups, piece_ops=64) as b:
            _setup(b, sc)
            b.set_record(out, ALL)
            before = b.launch_count
            b.run_fused(prog, imu=st["imu"], streams=gpu_streams(st))
            launches = b.launch_count - before
            b.wait(b.record())
            outs.append((as_np(out).copy(), b.get_state()))
            del out
        # automatic: several groups, each launching every piece
        assert (launches >= 2 * 2) if groups == 0 else (launches <= 2)
    for rec, state in outs[1:]:
        assert np.array_equal(rec, outs[0][0])
        _equal(state, outs[0][1])
    assert not np.isnan(outs[0][0]).any()


@pytest.mark.gpu
@pytest.mark.parametrize("mapping", [1, 4])
def test_pinned_host_records_leave_unrecorded_rows_untouched(mapping):
    """Calls whose record rows have holes, come in any order or repeat a row: a pinned host output equals the device output of
    the same calls, row for row, and the rows a call does not record keep what was there (NaN, or an earlier call's records)."""
    N, T, ROWS = 300, 60, 12
    sc = scenario(N, T)
    st = sc["st"]
    ev = st["events"]
    third = len(ev) // 3
    calls = [(ev[:third], [1]),                    # A: row 1
             (ev[third:2 * third], [0, 2, 5, 6]),  # B: around A's row, with a hole at 3, 4
             (ev[2 * third:], [9, 4, 9])]          # C: out of order, row 9 twice (the later record wins)
    res = []
    for where in (device_out, pinned_out):
        out = where(ROWS, POSE, N)
        with RBISBatch(N, mapping=mapping, launch_groups=1) as b:
            _setup(b, sc)
            b.set_record(out, POSE)
            for part, rows in calls:
                step = max(1, len(part) // len(rows))
                prog = []
                for e, event in enumerate(part):
                    prog.append(event)
                    if e % step == step - 1 and e // step < len(rows):
                        prog.append(rec_op(rows[e // step]))
                assert sum(1 for o in prog if o[0] == capi.OP_RECORD) == len(rows)
                b.run_fused(prog, imu=st["imu"], streams=gpu_streams(st))   # no synchronise between the calls
            b.wait(b.record())
        res.append(as_np(out).copy())
    dev, host = res
    recorded = [0, 1, 2, 4, 5, 6, 9]
    assert not np.isnan(dev[recorded]).any()
    assert np.isnan(dev[[3, 7, 8, 10, 11]]).all()
    assert np.array_equal(host, dev, equal_nan=True)


@pytest.mark.gpu
def test_pinned_host_records_of_unsynchronised_calls():
    """Consecutive calls without a synchronise record into different row ranges of pinned buffers pre-filled with NaN, switching
    between two record sets: after ONE wait every recorded row equals the device records of the same calls run one at a time,
    and every other row is still NaN."""
    N, T, CH, ROWS = 4000, 160, 20, 120
    sc = scenario(N, T)
    calls = []
    for c, k0 in enumerate(range(0, T, CH)):
        st = synth.make_streams(sc["truth"], N, k0, CH)
        base = 15 * c + (c % 3)   # gaps between the calls' row ranges
        prog, r = [], base
        for e in st["events"]:
            prog.append(e)
            if e[0] == capi.OP_IMU and e[2] % 4 == 1:
                prog.append(rec_op(r))
                r += 1
        calls.append((st, prog, c % 2))
    masks = (ALL, POSE)
    results = []
    for groups, where, sync in ((1, device_out, True), (6, pinned_out, False)):
        outs = [where(ROWS, m, N) for m in masks]
        with RBISBatch(N, mapping=1, launch_groups=groups, piece_ops=64) as b:
            _setup(b, sc)
            for st, prog, k in calls:
                b.set_record(outs[k], masks[k])
                b.run_fused(prog, imu=st["imu"], streams=gpu_streams(st))
                if sync:
                    b.synchronize()
            b.wait(b.record())
            results.append([as_np(o).copy() for o in outs])
    for k in range(2):
        ref, got = results[0][k], results[1][k]
        written = ~np.isnan(ref).all(axis=(1, 2))
        assert written.sum() == 20   # four calls of five records each
        assert np.array_equal(got[written], ref[written])
        assert np.isnan(got[~written]).all()
        assert not np.isnan(ref[written]).any()


@pytest.mark.gpu
@pytest.mark.parametrize("mapping", [1, 4])
def test_records_in_fused_synthesis_float_rows_and_column_maps(mapping):
    import torch

    N, T = 300, 220
    sc = scenario(N, T, tumbling=True)
    st = sc["st"]
    ev = st["events"]
    prog = []
    for e, event in enumerate(ev):
        prog += [event] + ([rec_op(e // 4)] if e % 4 == 0 else [])
    rows = (len(ev) + 3) // 4
    d = synth.synth_spec_inputs(sc["truth"], 0, T)
    outs = [device_out(rows, ALL, N) for _ in range(2)]
    with RBISBatch(N, mapping=mapping) as b:
        _setup(b, sc)
        spec = SynthSpec(synth.SEED, d["imu_mean"], d["imu_step"], d["streams"], mode=1)
        b.set_record(outs[0], ALL)
        b.run_fused_synth(prog, [MeasStream(synth.LEGODO_IDX, None, st["R_legodo"]), MeasStream(synth.POSE_IDX, None, st["R_pose"], quat=True)],
                          spec)
        assert b.last_kernel_variant & 12 == 12   # rows drawn in the kernel, records
        a = b.get_state()
        gen = b.synthesize(spec)
        _setup(b, sc)
        b.set_record(outs[1], ALL)
        b.run_fused(prog, imu=gen["imu"], streams=[MeasStream(synth.LEGODO_IDX, gen["z"][0], st["R_legodo"]),
                                                    MeasStream(synth.POSE_IDX, gen["z"][1], st["R_pose"], quat=gen["quat"][1])])
        b.synchronize()
        _equal(a, b.get_state())
    assert np.array_equal(as_np(outs[0]), as_np(outs[1]))
    torch.cuda.synchronize()
    # column maps: records stay per filter; float rows are widened exactly
    C_, G_ = 16, 8
    M = C_ * G_
    sc = scenario(C_, 120)
    st = sc["st"]
    cmap = (np.arange(M) % C_).astype(np.int32)
    ex = lambda a: np.ascontiguousarray(a[..., cmap])
    prog = []
    for e, event in enumerate(st["events"]):
        prog += [event] + ([rec_op(e // 3)] if e % 3 == 0 else [])
    rows = (len(st["events"]) + 2) // 3
    f32 = lambda a: np.ascontiguousarray(ex(a), dtype=np.float32)
    runs = (("mapped", lambda a: a), ("expanded", ex), ("float32", f32), ("widened", lambda a: f32(a).astype(np.float64)))
    recs = {}
    for what, f in runs:
        out = device_out(rows, ALL, M)
        with RBISBatch(M, mapping=mapping) as b:
            b.set_process_noise(*nominal_q())
            b.set_state(ex(sc["vec"]), ex(sc["quat"]), ex(sc["cov"]))
            if what == "mapped":
                for w in (-1, 0, 1):
                    b.set_column_map(w, cmap, C_)
            b.set_record(out, ALL)
            b.run_fused(prog, imu=f(st["imu"]), streams=[MeasStream(synth.LEGODO_IDX, f(st["legodo"]), st["R_legodo"]),
                                                         MeasStream(synth.POSE_IDX, f(st["pose_z"]), st["R_pose"], quat=f(st["pose_q"]))])
            b.synchronize()
        recs[what] = as_np(out)
    assert not np.isnan(recs["mapped"]).any()
    assert np.array_equal(recs["mapped"], recs["expanded"])
    assert np.array_equal(recs["float32"], recs["widened"])


@pytest.mark.gpu
def test_record_errors_leave_handle_and_ensemble_unchanged():
    import torch

    N, T = 64, 30
    sc = scenario(N, T)
    st = sc["st"]
    ev = st["events"]
    with RBISBatch(N) as b:
        _setup(b, sc)
        b.run_fused(ev[:10], imu=st["imu"], streams=gpu_streams(st))
        before = b.get_state()
        # a RECORD op without a record set
        with pytest.raises(capi.RBISError, match="rbis error -4: .*no record set"):
            b.run_fused(ev[10:] + [rec_op(0)], imu=st["imu"], streams=gpu_streams(st))
        _equal(before, b.get_state())
        out = device_out(4, POSE, N)
        b.set_record(out, POSE)
        for row in (-1, 4):
            with pytest.raises(capi.RBISError, match="rbis error -1: .*record row"):
                b.run_fused(ev[10:] + [rec_op(row)], imu=st["imu"], streams=gpu_streams(st))
        _equal(before, b.get_state())
        # invalid record sets are refused and leave the current one in place
        rec = capi.Record()
        rec.out, rec.rows, rec.mem = out.data_ptr(), 4, capi.MEM_DEVICE
        for fields in (0, 1 << capi.REC_FIELDS, 1 << 63):
            rec.fields = fields
            assert b.lib.rbis_batch_set_record(b.h, C.byref(rec)) == -1
        rec.fields, rec.out = POSE, None
        assert b.lib.rbis_batch_set_record(b.h, C.byref(rec)) == -1
        pageable = np.full((4, 7, N), np.nan)
        with pytest.raises(capi.RBISError, match="pinned"):
            b.set_record(pageable, POSE)
        host_as_device = pinned_out(4, POSE, N)
        rec.out, rec.mem = host_as_device.data_ptr(), capi.MEM_DEVICE
        assert b.lib.rbis_batch_set_record(b.h, C.byref(rec)) == -1
        _equal(before, b.get_state())
        b.run_fused([rec_op(2)], imu=st["imu"], streams=gpu_streams(st))   # the set made by set_record above
        b.synchronize()
        got = as_np(out)
        assert np.array_equal(got[2], select(fields_of(*before), POSE))
        assert np.isnan(got[[0, 1, 3]]).all()
        _equal(before, b.get_state())
        # cleared: RECORD fails again
        b.clear_record()
        with pytest.raises(capi.RBISError, match="no record set"):
            b.run_fused([rec_op(0)], imu=st["imu"], streams=gpu_streams(st))
    torch.cuda.synchronize()
