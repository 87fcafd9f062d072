"""Measurement rows that some filters did not receive (RBIS_STREAM_SKIP_NAN_ROWS, include/rbis_batch.h).

A Monte-Carlo outage study runs one schedule for the whole ensemble, but every realisation loses its own rows: a filter whose
row holds a NaN in a value the update reads skips that MEAS op.  The yardstick is deletion: filter n must end, bit for bit
(compared as bit patterns), where the same program ends with the MEAS ops of its missing rows deleted.  The tests group the
filters by dropout pattern and run one unflagged reference program per pattern at the same N."""
import ctypes as C
import os

import numpy as np
import pytest

from pronto_b200 import MeasStream, RBISBatch, SynthSpec, capi, synth
from pronto_b200.parity import max_errors

from common import nominal_q, scenario

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NTHREADS = min(16, os.cpu_count() or 1)
STEP_TOL = 1e-9
ALL = (1 << capi.REC_FIELDS) - 1
MASK_VARIANT = 512


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
def test_stream_struct_keeps_its_layout():
    """`reserved` became `flags`: same offset, type and size, so binaries built against the old header keep working."""
    assert C.sizeof(capi.Stream) == 4 * 4 + 4 * capi.MAX_MEAS + 4 + 3 * 8 + 8
    assert capi.Stream.flags.offset == 4 * 4 + 4 * capi.MAX_MEAS
    assert capi.Stream.flags.size == 4
    assert capi.Stream.z.offset == capi.Stream.flags.offset + 4
    assert capi.Stream().flags == 0   # ctypes zero-initialises: existing callers set no flag


def test_header_constant_matches_capi():
    with open(os.path.join(ROOT, "include", "rbis_batch.h")) as f:
        text = f.read()
    assert "#define RBIS_STREAM_SKIP_NAN_ROWS 1" in text
    assert capi.STREAM_SKIP_NAN_ROWS == 1
    assert "int32_t flags;" in text and "int32_t reserved;\n  const double* z;" not in text


# ------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------
def readable(d):
    """Columns of stream d's z that an update reads (not the chi entries of an orientation stream)."""
    orient = d.get("quat") is not None
    return [a for a, i in enumerate(d["idx"]) if not (orient and 6 <= i <= 8)]


def random_miss(streams, which, N, rng, frac=0.2, n_patterns=4, unique=(5, 77)):
    """{stream: bool [rows][N]}: a few shared dropout patterns (about `frac` of the rows of each stream in `which`) assigned
    to the filters at random, plus filters in `unique` with patterns of their own."""
    pid = rng.integers(0, n_patterns, N)
    miss = {}
    for s in which:
        rows = streams[s]["z"].shape[0]
        base = rng.random((n_patterns, rows)) < frac
        m = base[pid].T.copy()
        for n in unique:
            if n < N:
                m[:, n] = rng.random(rows) < frac
        miss[s] = m
    return miss


def with_nans(streams, miss, rng):
    """Copies of the streams whose z holds a NaN at one random readable column of every missing (row, filter); the chi
    entries of orientation streams are NaN everywhere (never read, so they must not count)."""
    out = []
    for s, d in enumerate(streams):
        d = dict(d)
        z = np.array(d["z"], dtype=np.float64, copy=True)
        if d.get("quat") is not None:
            for a, i in enumerate(d["idx"]):
                if 6 <= i <= 8:
                    z[:, a, :] = np.nan
        if s in miss:
            cols = readable(d)
            r, n = np.nonzero(miss[s])
            z[r, np.asarray(cols)[rng.integers(0, len(cols), len(r))], n] = np.nan
        d["z"] = z
        out.append(d)
    return out


def gpu(streams, flag):
    return [MeasStream(d["idx"], d["z"], d["R"], quat=d.get("quat"), per_filter_diag=d.get("per_filter_diag", False),
                       skip_nan_rows=flag) for d in streams]


def patterns(miss, N):
    """pattern key -> filter indices (filters that miss exactly the same rows)."""
    keys = {}
    if not miss:
        return {(): np.arange(N)}
    stacked = np.concatenate([miss[s] for s in sorted(miss)], axis=0)
    for n in range(N):
        keys.setdefault(stacked[:, n].tobytes(), []).append(n)
    return {k: np.asarray(v) for k, v in keys.items()}


def deleted(ops, miss, n):
    """The program with every MEAS op of a row that filter n misses deleted."""
    return [o for o in ops if not (o[0] == capi.OP_MEAS and o[1] in miss and miss[o[1]][o[2], n])]


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def assert_bits(got, want, cols=None):
    for x, y in zip(got[:4], want[:4]):
        x, y = np.asarray(x), np.asarray(y)
        if cols is not None:
            x, y = x[..., cols], y[..., cols]
        assert np.array_equal(bits(x), bits(y))


def run(sc, streams, ops, flag, rec=None, **cfg):
    """-> (vec, quat, cov, loglik, utime), kernel variant, records (or None)."""
    import torch

    N = sc["vec"].shape[1]
    with RBISBatch(N, **cfg) as b:
        b.set_process_noise(*nominal_q())
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        out = None
        if rec:
            out = torch.full((rec, capi.REC_FIELDS, N), float("nan"), dtype=torch.float64, device="cuda")
            b.set_record(out, ALL)
        b.run_fused(ops, imu=sc["st"]["imu"], streams=gpu(streams, flag))
        b.synchronize()
        return b.get_state(), b.last_kernel_variant, (out.cpu().numpy() if rec else None)


def references(sc, streams, ops, miss, rec=None, **cfg):
    """Per pattern: the unflagged program with that pattern's missing MEAS ops deleted, at the same N.  -> the state, and the
    records, every filter taken from the run of its own pattern."""
    N = sc["vec"].shape[1]
    groups = patterns(miss, N)
    state = [None] * 4
    recs = None
    for cols in groups.values():
        st, _, r = run(sc, streams, deleted(ops, miss, cols[0]), False, rec=rec, **cfg)
        for k in range(4):
            if state[k] is None:
                state[k] = np.empty_like(st[k])
            state[k][..., cols] = st[k][..., cols]
        if rec:
            recs = np.empty_like(r) if recs is None else recs
            recs[..., cols] = r[..., cols]
    return state, recs, groups


def with_records(ops, every=1):
    """ops with a RECORD op after every `every`-th op -> (program, record rows)."""
    prog, row = [], 0
    for i, o in enumerate(ops):
        prog.append(tuple(o))
        if i % every == every - 1:
            prog.append((capi.OP_RECORD, 0, row, 0, 0.0))
            row += 1
    return prog, row


def base(sc):
    st = sc["st"]
    return [dict(idx=synth.LEGODO_IDX, z=st["legodo"], R=st["R_legodo"]),
            dict(idx=synth.POSE_IDX, z=st["pose_z"], R=st["R_pose"], quat=st["pose_q"])]


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mapping,dense_only", [(1, False), (1, True), (4, False), (16, True)])
def test_flag_without_nans_changes_nothing(mapping, dense_only):
    """Config-3 program on a tumbling trajectory: with the flag set and no NaN anywhere, the MASK kernels give the bits of the
    ordinary kernels."""
    N, T = 300, 300
    sc = scenario(N, T, tumbling=True)
    ops = sc["st"]["events"]
    cfg = dict(mapping=mapping, dense_only=dense_only)
    a, va, _ = run(sc, base(sc), ops, False, **cfg)
    b, vb, _ = run(sc, base(sc), ops, True, **cfg)
    assert not va & MASK_VARIANT and vb == va | MASK_VARIANT
    assert_bits(b, a)


@pytest.mark.gpu
@pytest.mark.parametrize("mapping", [1, 4])
def test_random_dropouts_equal_deleted_ops_and_the_oracle(oracle, mapping):
    """About 20 % per-filter dropouts on leg odometry and pose fixes: every filter equals, bit for bit, the program without its
    missing ops, and after every event its records stay within the per-step gate of the oracle fed that pattern's events."""
    N, T = 256, 240
    rng = np.random.default_rng(11)
    sc = scenario(N, T, tumbling=True)
    streams = base(sc)
    miss = random_miss(streams, (0, 1), N, rng)
    ops = [tuple(e) for e in sc["st"]["events"]]
    prog, rows = with_records(ops)
    got, var, rec = run(sc, with_nans(streams, miss, rng), prog, True, rec=rows, mapping=mapping)
    assert var & MASK_VARIANT
    want, want_rec, groups = references(sc, streams, prog, miss, rec=rows, mapping=mapping)
    assert len(groups) >= 5
    assert_bits(got, want)
    assert np.array_equal(bits(rec), bits(want_rec))
    q = nominal_q()
    worst = 0.0
    for cols in groups.values():
        n0 = cols[0]
        keep = [e for e in range(len(ops)) if not (ops[e][0] == capi.OP_MEAS and ops[e][1] in miss and miss[ops[e][1]][ops[e][2], n0])]
        sub = lambda a: np.ascontiguousarray(np.asarray(a)[..., cols])
        ostreams = [dict(idx=d["idx"], z=sub(d["z"]), R=d["R"], **({"quat": sub(d["quat"])} if d.get("quat") is not None else {}))
                    for d in streams]
        ref = oracle.run_ensemble(sub(sc["vec"]), sub(sc["quat"]), sub(sc["cov"]), None, 0, q, sub(sc["st"]["imu"]), ostreams,
                                  [ops[e] for e in keep], n_threads=NTHREADS, trace=True)
        for j, e in enumerate(keep):
            r = rec[e][:, cols]
            err = max_errors(r[0:21], r[21:25], None, ref["trace_vec"][j], ref["trace_quat"][j], None)
            ll = np.asarray(ref["trace_loglik"][j])
            err["ll"] = float(np.max(np.abs(r[25] - ll) / np.maximum(1.0, np.abs(ll))))
            worst = max(worst, *err.values())
    assert worst <= STEP_TOL, worst


@pytest.mark.gpu
@pytest.mark.parametrize("mapping", [1, 8])
def test_patterns_at_the_edges(mapping):
    """A whole warp skips, a single lane skips, the first and the last filter skip, N is not a multiple of the CTA size (idle
    lanes shadow the last filter), and one row every filter skips (the same as deleting that op for everyone)."""
    N, T = 300, 200
    sc = scenario(N, T)
    streams = base(sc)
    rows = streams[0]["z"].shape[0]
    m = np.zeros((rows, N), dtype=bool)
    m[3, 0:32] = True          # a whole warp
    m[7, 40] = True            # one lane
    m[11, [0, N - 1]] = True   # first and last filter
    m[15, :] = True            # everyone
    m[rows - 1, N - 1] = True  # the last filter, last row
    miss = {0: m}
    ops = [tuple(e) for e in sc["st"]["events"]]
    got, var, _ = run(sc, with_nans(streams, miss, np.random.default_rng(2)), ops, True, mapping=mapping)
    assert var & MASK_VARIANT
    want, _, groups = references(sc, streams, ops, miss, mapping=mapping)
    assert len(groups) == 5
    assert_bits(got, want)
    everyone = [o for o in ops if not (o[0] == capi.OP_MEAS and o[1] == 0 and o[2] == 15)]
    rest = np.setdiff1d(np.arange(N), [0, 40, N - 1, *range(32)])
    alone, _, _ = run(sc, streams, everyone, False, mapping=mapping)
    assert_bits(got, alone, cols=rest)


def _chunk_program(N=200, T=200, per_filter=False):
    """Leg odometry (per-row R, or per-filter diagonal R), pose fixes, yaw lock [17, 8] with orientation (one-row chunks) and a
    quick-lock [8..11] block with correlated per-row R."""
    from test_row_noise import extra_streams, legodo_R

    sc = scenario(N, T, tumbling=True)
    st = sc["st"]
    extra, ev = extra_streams(sc, k_ql=range(4, T, 9), k_yaw=range(6, T, 11))
    streams = base(sc)
    if per_filter:
        streams[0]["R"] = np.ascontiguousarray(np.random.default_rng(4).uniform(0.5, 2.0, (3, N)) * synth.NOMINAL["r_vxyz"] ** 2)
        streams[0]["per_filter_diag"] = True
    else:
        streams[0]["R"] = legodo_R(st["legodo"].shape[0], frac=0.3)[0]
    streams += extra[:2]
    return sc, streams, [tuple(e) for e in ev]


@pytest.mark.gpu
@pytest.mark.parametrize("per_filter", [False, True])
def test_chunk_kinds_and_r_modes_in_every_mapping(per_filter):
    """One-row chunks (yaw lock with orientation), correlated blocks (quick lock), per-row and per-filter R: the deleted-op
    references, and the same bits from the dense and decoupled kernels and from every mapping."""
    sc, streams, ops = _chunk_program(per_filter=per_filter)
    N = sc["vec"].shape[1]
    rng = np.random.default_rng(5)
    miss = random_miss(streams, (0, 1, 2, 3), N, rng, frac=0.25)
    want, _, _ = references(sc, streams, ops, miss, mapping=1)
    flagged = with_nans(streams, miss, rng)
    for dense_only in (False, True):
        for mapping in (1, 2, 4, 8, 16):
            got, var, _ = run(sc, flagged, ops, True, mapping=mapping, dense_only=dense_only)
            assert var & MASK_VARIANT and bool(var & 2) == (not dense_only), (mapping, dense_only, var)
            assert_bits(got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("mapping,dense_only", [(1, False), (1, True), (2, False), (8, True)])
def test_records_inside_masked_programs(mapping, dense_only):
    """The MASK+REC kernels: records of a masked program equal the records of the per-pattern reference runs."""
    sc, streams, ops = _chunk_program(N=160)
    N = sc["vec"].shape[1]
    rng = np.random.default_rng(8)
    miss = random_miss(streams, (0, 1, 3), N, rng)
    prog, rows = with_records(ops, every=3)
    cfg = dict(mapping=mapping, dense_only=dense_only)
    got, var, rec = run(sc, with_nans(streams, miss, rng), prog, True, rec=rows, **cfg)
    assert var & (MASK_VARIANT | 8) == MASK_VARIANT | 8
    want, want_rec, _ = references(sc, streams, prog, miss, rec=rows, **cfg)
    assert_bits(got, want)
    assert np.array_equal(bits(rec), bits(want_rec))


@pytest.mark.gpu
@pytest.mark.parametrize("mapping", [1, 4])
def test_planner_rewinds_replay_missing_rows(oracle, mapping):
    """Late pose fixes planned into RESTORE + replay, with missing rows inside the replayed spans: the deleted-op references,
    and per pattern the oracle's own history (its multimap insert and replay) fed that pattern's arrivals."""
    from pronto_b200.schedule import program_from_arrivals

    N, T = 128, 240
    sc = scenario(N, T)
    streams = base(sc)
    ev = [tuple(e) for e in sc["st"]["events"]]
    arrivals, pending = [], [e for e in ev if e[0] == capi.OP_MEAS and e[1] == 1]
    for e in ev:
        if e[0] == capi.OP_MEAS and e[1] == 1:
            continue
        arrivals.append(e)
        while pending and e[0] == capi.OP_IMU and e[3] >= pending[0][3] + 30_000:
            arrivals.append(pending.pop(0))
    arrivals += pending
    ops, cnt = program_from_arrivals(arrivals, snapshot_slots=4, snapshot_period_us=50_000, snapshot_phase_us=1000)
    assert cnt["rewinds"] > 0
    ops = [tuple(o.tolist()) for o in ops]
    rng = np.random.default_rng(9)
    miss = random_miss(streams, (0, 1), N, rng)
    got, var, _ = run(sc, with_nans(streams, miss, rng), ops, True, snapshot_slots=4, mapping=mapping)
    assert var & MASK_VARIANT
    want, _, groups = references(sc, streams, ops, miss, snapshot_slots=4, mapping=mapping)
    assert_bits(got, want)
    q = nominal_q()
    for cols in groups.values():
        sub = lambda a: np.ascontiguousarray(np.asarray(a)[..., cols])
        ostreams = [dict(idx=d["idx"], z=sub(d["z"]), R=d["R"], **({"quat": sub(d["quat"])} if d.get("quat") is not None else {}))
                    for d in streams]
        ref = oracle.run_ensemble(sub(sc["vec"]), sub(sc["quat"]), sub(sc["cov"]), None, 0, q, sub(sc["st"]["imu"]), ostreams,
                                  deleted(arrivals, miss, cols[0]), n_threads=NTHREADS)
        e = max_errors(got[0][:, cols], got[1][:, cols], got[2][:, cols], ref["vec"], ref["quat"], ref["cov"])
        ll = ref["loglik"]
        e["ll"] = float(np.max(np.abs(got[3][cols] - ll) / np.maximum(1.0, np.abs(ll))))
        assert max(e.values()) < 1e-8, e


@pytest.mark.gpu
def test_launch_groups_pieces_column_maps_and_float_rows():
    """Automatic launch groups with pieces against one group (40,000 filters); a NaN in a shared column of a column map skips
    every filter that reads it, as the expanded rows do; float rows widen NaN to NaN."""
    rng = np.random.default_rng(12)
    # launch groups and pieces
    N, T = 40_000, 60
    sc = scenario(N, T)
    streams = base(sc)
    miss = {0: rng.random((streams[0]["z"].shape[0], N)) < 0.2, 1: rng.random((streams[1]["z"].shape[0], N)) < 0.2}
    flagged = with_nans(streams, miss, rng)
    ops = [tuple(e) for e in sc["st"]["events"]]
    one, v1, _ = run(sc, flagged, ops, True, mapping=1, launch_groups=1)
    grp, v2, _ = run(sc, flagged, ops, True, mapping=1, launch_groups=0, piece_ops=16)
    assert v1 & MASK_VARIANT and v2 & MASK_VARIANT
    assert_bits(grp, one)
    # column maps and float rows
    N, T, cols = 256, 150, 8
    sc = scenario(N, T)
    st = sc["st"]
    f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)
    z_shared = f32(st["legodo"][:, :, :cols]).astype(np.float64)
    rows = z_shared.shape[0]
    z_shared[rng.integers(0, rows, 20), rng.integers(0, 3, 20), rng.integers(0, cols, 20)] = np.nan
    cmap = (np.arange(N) * 5 % cols).astype(np.int32)
    expanded = np.ascontiguousarray(z_shared[:, :, cmap])
    pose = dict(idx=synth.POSE_IDX, z=st["pose_z"], R=st["R_pose"], quat=st["pose_q"])
    ops = [tuple(e) for e in st["events"]]
    ref, _, _ = run(sc, [dict(idx=synth.LEGODO_IDX, z=expanded, R=st["R_legodo"]), pose], ops, True, mapping=1)
    miss = {0: np.isnan(expanded).any(axis=1)}
    assert miss[0].any() and not miss[0].all()
    want, _, _ = references(sc, [dict(idx=synth.LEGODO_IDX, z=np.nan_to_num(expanded), R=st["R_legodo"]), pose], ops, miss, mapping=1)
    assert_bits(ref, want)
    imu32 = f32(st["imu"])
    for mapping in (1, 4):
        for kind in ("mapped", "float32"):
            with RBISBatch(N, mapping=mapping) as b:
                b.set_process_noise(*nominal_q())
                b.set_state(sc["vec"], sc["quat"], sc["cov"])
                if kind == "mapped":
                    b.set_column_map(0, cmap, cols)
                    streams = [MeasStream(synth.LEGODO_IDX, z_shared, st["R_legodo"], skip_nan_rows=True),
                               MeasStream(synth.POSE_IDX, st["pose_z"], st["R_pose"], quat=st["pose_q"], skip_nan_rows=True)]
                    b.run_fused(ops, imu=st["imu"], streams=streams)
                else:
                    streams = [MeasStream(synth.LEGODO_IDX, f32(expanded), st["R_legodo"], skip_nan_rows=True),
                               MeasStream(synth.POSE_IDX, f32(st["pose_z"]), st["R_pose"], quat=f32(st["pose_q"]), skip_nan_rows=True)]
                    b.run_fused(ops, imu=imu32, streams=streams)
                assert b.last_kernel_variant & MASK_VARIANT
                got = b.get_state()
            if kind == "mapped":
                assert_bits(got, ref)
            else:
                assert np.isnan(f32(expanded)).sum() == np.isnan(expanded).sum()
                widened = [dict(idx=synth.LEGODO_IDX, z=f32(expanded).astype(np.float64), R=st["R_legodo"]),
                           dict(pose, z=f32(st["pose_z"]).astype(np.float64), quat=f32(st["pose_q"]).astype(np.float64))]
                sc32 = dict(sc, st=dict(st, imu=imu32.astype(np.float64)))
                w, _, _ = run(sc32, widened, ops, True, mapping=mapping)
                assert_bits(got, w)


@pytest.mark.gpu
def test_error_cases():
    N, T = 64, 40
    sc = scenario(N, T)
    st = sc["st"]
    ops = st["events"]
    with RBISBatch(N) as b:
        b.set_process_noise(*nominal_q())
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        before = b.launch_count
        for bad in (2, 1 | 8, -1):
            prep = b.prepare_fused(ops, imu=st["imu"], streams=gpu(base(sc), True))
            prep[5][0].flags = bad
            with pytest.raises(capi.RBISError, match="unknown flags"):
                b.run_prepared(prep)
        d = synth.synth_spec_inputs(sc["truth"], 0, T)
        spec = SynthSpec(synth.SEED, d["imu_mean"], d["imu_step"], d["streams"], mode=1)
        for s in (0, 1):
            streams = [MeasStream(synth.LEGODO_IDX, None, st["R_legodo"]), MeasStream(synth.POSE_IDX, None, st["R_pose"], quat=True)]
            streams[s].skip_nan_rows = True
            with pytest.raises(capi.RBISError, match="synthesised"):
                b.run_fused_synth(ops, streams, spec)
        assert b.launch_count == before   # rejected before anything was enqueued
        b.run_fused(ops, imu=st["imu"], streams=gpu(base(sc), True))
        assert b.last_kernel_variant & MASK_VARIANT
