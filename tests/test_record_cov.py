"""Records of covariance blocks (rbis_record_t::cov_blocks) and ensemble statistics over record rows
(rbis_batch_stats_records_enqueue), include/rbis_batch.h.  A record row's covariance part must hold, bit for bit, what a snapshot
at the same program position holds in those slots; the statistics of a record row must equal, bit for bit, the statistics of
such a snapshot; and a row with vec, quat and all seven blocks must give the filter_state_t messages of the reference."""
import ctypes as C
import os

import numpy as np
import pytest

from pronto_b200 import (MeasStream, RBISBatch, SynthSpec, capi, filter_states_from_record, record_cov_blocks, record_fields,
                         record_layout, reduce_chunks, synth)
from pronto_b200.parity import max_errors

from common import gpu_streams, nominal_q, oracle_streams, scenario

NTHREADS = min(16, os.cpu_count() or 1)
STEP_TOL = 1e-9
ALL = (1 << capi.REC_FIELDS) - 1
STATE = record_fields(vec=range(21), quat=True, loglik=True)   # fields 0..25
POSE = record_fields(vec=(9, 10, 11), quat=True)
BLOCK_SETS = [  # (fields, covariance blocks)
    (ALL, range(7)),
    (STATE, (1, 2, 3)),          # the NEES block
    (0, (0, 3, 6)),              # omega / p / accel bias: parked and exactly-zero slots of the decoupled kernels, no fields
    (POSE, (2, 3)),              # the pose covariance
]


def cov_index(blocks):
    return [3 * b + c for b in sorted(blocks) for c in range(3)]


def expected_row(vec, quat, cov, ll, fields, blocks):
    """[k][N] a record row holds for a state as get_state / get_snapshot return it (full covariance [441][N])."""
    full = np.concatenate([vec, quat, ll[None], cov[[i + 21 * i for i in range(21)]]])
    rows = [full[f] for f in range(capi.REC_FIELDS) if fields >> f & 1]
    idx = cov_index(blocks)
    for jj, j in enumerate(idx):
        rows += [cov[i + 21 * j] for i in idx[:jj + 1]]
    return np.stack(rows)


def k_of(fields, blocks):
    return len(record_layout(fields, blocks))


def device_out(rows, fields, blocks, N):
    import torch

    return torch.full((rows, k_of(fields, blocks), N), float("nan"), dtype=torch.float64, device="cuda")


def pinned_out(rows, fields, blocks, N):
    import torch

    return torch.full((rows, k_of(fields, blocks), N), float("nan"), dtype=torch.float64).pin_memory()


def as_np(t):
    return t.cpu().numpy() if hasattr(t, "cpu") else np.asarray(t)


def rec_op(row):
    return (capi.OP_RECORD, 0, int(row), 0, 0.0)


def snap_op(slot):
    return (capi.OP_SNAPSHOT, 0, int(slot), 0, 0.0)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _setup(b, sc):
    b.set_process_noise(*nominal_q())
    b.set_state(sc["vec"], sc["quat"], sc["cov"])


def _equal_state(a, b):
    for x, y in zip(a[:4], b[:4]):
        assert np.array_equal(bits(x), bits(y))


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
def test_cov_blocks_takes_the_place_of_reserved(rbis_lib):
    class Old(C.Structure):
        _fields_ = [("fields", C.c_uint64), ("out", C.c_void_p), ("rows", C.c_int64), ("mem", C.c_int32), ("reserved", C.c_int32)]

    assert capi.Record.cov_blocks.offset == Old.reserved.offset
    assert capi.Record.cov_blocks.size == Old.reserved.size == 4
    assert C.sizeof(capi.Record) == C.sizeof(Old)


def test_layout_positions_follow_the_packed_formula(rbis_lib):
    rng = np.random.default_rng(7)
    assert len(record_layout(0, range(7))) == 231
    assert record_layout(POSE, (3,))[7:] == ["cov9_9", "cov9_10", "cov10_10", "cov9_11", "cov10_11", "cov11_11"]
    for _ in range(300):
        fields = int(rng.integers(0, 1 << 47)) & int(rng.choice([ALL, STATE, POSE, 0]))
        blocks = sorted(set(rng.integers(0, 7, rng.integers(0, 5)).tolist()))
        if not fields and not blocks:
            continue
        names = record_layout(fields, blocks)
        kf, nb = bin(fields).count("1"), 3 * len(blocks)
        assert len(names) == kf + nb * (nb + 1) // 2
        assert names[:kf] == record_layout(fields) if fields else kf == 0
        idx = cov_index(blocks)
        for jj in range(nb):
            for ii in range(jj + 1):
                assert names[kf + jj * (jj + 1) // 2 + ii] == f"cov{idx[ii]}_{idx[jj]}"
        cov = [n for n in names[kf:]]
        back = sorted({int(n[3:].split("_")[0]) // 3 for n in cov})
        assert back == blocks
    assert record_cov_blocks((0, 6)) == 0x41
    for bad in ((7,), (-1,)):
        with pytest.raises(ValueError):
            record_cov_blocks(bad)
    with pytest.raises(ValueError):
        record_layout(0, ())


def test_filter_state_messages_from_a_synthetic_row(rbis_lib):
    N = 5
    rng = np.random.default_rng(3)
    vec, quat, ll = rng.normal(size=(21, N)), rng.normal(size=(4, N)), rng.normal(size=N)
    A = rng.normal(size=(N, 21, 21))
    full = np.einsum("nij,nkj->nik", A, A)                 # symmetric per filter
    cov = np.ascontiguousarray(full.transpose(2, 1, 0).reshape(441, N))   # element (i, j) at i + 21 j
    for fields in (STATE, ALL, record_fields(vec=range(21), quat=True)):
        row = expected_row(vec, quat, cov, ll, fields, range(7))
        msgs = filter_states_from_record(row, fields, utime=1234, first=1, count=3)
        for k in range(3):
            n = 1 + k
            m = msgs[k]
            assert m.utime == 1234 and m.num_states == 21 and m.num_cov_elements == 441
            assert np.array_equal(np.array(m.state), vec[:, n])
            assert np.array_equal(np.array(m.quat), quat[:, n])
            want = np.array([full[n][e % 21, e // 21] for e in range(441)])   # column-major, both triangles
            assert np.array_equal(np.array(m.cov), want)
    row = expected_row(vec, quat, cov, ll, STATE, range(7))
    for fields, blocks in ((POSE, range(7)), (STATE, range(6))):
        with pytest.raises(capi.RBISError, match="rbis error -1"):
            filter_states_from_record(row, fields, blocks)
    with pytest.raises(capi.RBISError, match="rbis error -1"):
        filter_states_from_record(row, STATE, range(7), first=4, count=2)


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
def _rewind_program(N=64, T=200):
    from test_record import _rewind_program as rp

    return rp(N, T)


def _insert(ops, at, extra):
    from test_record import _insert as ins

    return ins(ops, at, extra)


@pytest.mark.gpu
@pytest.mark.parametrize("mapping", [1, 2, 4, 8, 16])
@pytest.mark.parametrize("dense_only", [False, True])
def test_records_equal_snapshots(mapping, dense_only):
    """Before the first IMU step (at -1), right after every RESTORE and after IMU / MEAS ops: every covariance-block record row
    equals the selected entries of a SNAPSHOT at the same position, bit for bit."""
    sc, streams, ops, at = _rewind_program()
    st, N = sc["st"], sc["vec"].shape[1]
    assert at[0] == -1 and any(ops[i][0] == capi.OP_RESTORE for i in at if i >= 0)
    R = len(at)
    prog = _insert(ops, at, lambda j: [rec_op(j), snap_op(3 + j)])
    for fields, blocks in BLOCK_SETS:
        out = device_out(R, fields, blocks, N)
        with RBISBatch(N, snapshot_slots=3 + R, mapping=mapping, dense_only=dense_only) as b:
            _setup(b, sc)
            b.set_record(out, fields, blocks)
            b.run_fused(prog, imu=st["imu"], streams=streams)
            assert b.last_kernel_variant & 8
            assert bool(b.last_kernel_variant & 2) == (not dense_only)
            want = np.stack([expected_row(*b.get_snapshot(3 + j), fields, blocks) for j in range(R)])
        assert np.array_equal(bits(as_np(out)), bits(want)), (fields, blocks)


@pytest.mark.gpu
@pytest.mark.parametrize("mapping", [1, 4])
def test_covariance_records_do_not_perturb_the_filter(mapping):
    sc, streams, ops, at = _rewind_program()
    st, N = sc["st"], sc["vec"].shape[1]
    out = device_out(len(at), ALL, range(7), N)
    with RBISBatch(N, snapshot_slots=3, mapping=mapping) as b:
        _setup(b, sc)
        b.run_fused(ops, imu=st["imu"], streams=streams)
        plain = b.get_state()
        _setup(b, sc)
        b.set_record(out, ALL, range(7))
        b.run_fused(_insert(ops, at, lambda j: [rec_op(j)]), imu=st["imu"], streams=streams)
        recorded = b.get_state()
    _equal_state(plain, recorded)
    assert not np.isnan(as_np(out)).any()


def _check_against_snapshots(make_batch, run, N, rows, fields=STATE, blocks=(1, 2, 3), where=device_out):
    """run(b, prog_fn) runs a program whose record j is followed by a snapshot into slot j; -> the record rows equal those
    snapshots, and the same program with the record output in pinned host memory gives the same bits."""
    outs = []
    for w in (where, pinned_out) if where is device_out else (where,):
        out = w(rows, fields, blocks, N)
        with make_batch() as b:
            b.set_record(out, fields, blocks)
            run(b)
            b.wait(b.record())
            want = np.stack([expected_row(*b.get_snapshot(j), fields, blocks) for j in range(rows)])
            got = as_np(out).copy()
        assert np.array_equal(bits(got), bits(want))
        outs.append(got)
    for o in outs[1:]:
        assert np.array_equal(bits(o), bits(outs[0]))


@pytest.mark.gpu
def test_every_path_launch_groups_pieces_and_host_output():
    N, T = 40_000, 100
    sc = scenario(N, T)
    st = sc["st"]
    prog, rows = [], 0
    for e, event in enumerate(st["events"]):
        prog.append(event)
        if e % 25 == 0:
            prog += [rec_op(rows), snap_op(rows)]
            rows += 1
    assert len(prog) >= 2 * 64
    for groups in (1, 0):
        def run(b):
            _setup(b, sc)
            b.run_fused(prog, imu=st["imu"], streams=gpu_streams(st))
        _check_against_snapshots(lambda: RBISBatch(N, mapping=1, launch_groups=groups, piece_ops=64, snapshot_slots=rows), run, N,
                                 rows, fields=ALL, blocks=range(7))


@pytest.mark.gpu
@pytest.mark.parametrize("mapping", [1, 4])
def test_every_path_synthesis_nan_rows_and_column_maps(mapping):
    from test_missing_rows import gpu, with_nans

    N, T = 300, 120
    sc = scenario(N, T, tumbling=True)
    st = sc["st"]
    prog, rows = [], 0
    for e, event in enumerate(st["events"]):
        prog.append(event)
        if e % 9 == 0:
            prog += [rec_op(rows), snap_op(rows)]
            rows += 1
    # fused synthesis
    d = synth.synth_spec_inputs(sc["truth"], 0, T)

    def run_syn(b):
        _setup(b, sc)
        spec = SynthSpec(synth.SEED, d["imu_mean"], d["imu_step"], d["streams"], mode=1)
        b.run_fused_synth(prog, [MeasStream(synth.LEGODO_IDX, None, st["R_legodo"]), MeasStream(synth.POSE_IDX, None, st["R_pose"], quat=True)],
                          spec)
        assert b.last_kernel_variant & 12 == 12
    _check_against_snapshots(lambda: RBISBatch(N, mapping=mapping, snapshot_slots=rows), run_syn, N, rows, fields=ALL, blocks=range(7))
    # streams that skip NaN rows (MASK kernels)
    rng = np.random.default_rng(4)
    miss = {0: rng.random((st["legodo"].shape[0], N)) < 0.2}
    flagged = gpu(with_nans(oracle_streams(st), miss, rng), True)

    def run_nan(b):
        _setup(b, sc)
        b.run_fused(prog, imu=st["imu"], streams=flagged)
        assert b.last_kernel_variant & 512
    _check_against_snapshots(lambda: RBISBatch(N, mapping=mapping, snapshot_slots=rows), run_nan, N, rows)
    # column maps: records stay per filter
    C_, G_ = 16, 8
    M = C_ * G_
    sc2 = scenario(C_, 80)
    st2 = sc2["st"]
    cmap = (np.arange(M) % C_).astype(np.int32)
    ex = lambda a: np.ascontiguousarray(a[..., cmap])
    prog2, rows2 = [], 0
    for e, event in enumerate(st2["events"]):
        prog2.append(event)
        if e % 7 == 0:
            prog2 += [rec_op(rows2), snap_op(rows2)]
            rows2 += 1

    def run_map(b):
        b.set_process_noise(*nominal_q())
        b.set_state(ex(sc2["vec"]), ex(sc2["quat"]), ex(sc2["cov"]))
        for w in (-1, 0, 1):
            b.set_column_map(w, cmap, C_)
        b.run_fused(prog2, imu=st2["imu"], streams=gpu_streams(st2))
    _check_against_snapshots(lambda: RBISBatch(M, mapping=mapping, snapshot_slots=rows2), run_map, M, rows2, fields=ALL, blocks=range(7))


@pytest.mark.gpu
@pytest.mark.parametrize("tumbling", [False, True])
def test_full_covariance_records_against_the_oracle(oracle, tumbling):
    N, T = 150, 220
    sc = scenario(N, T, tumbling=tumbling)
    st = sc["st"]
    ev = st["events"]
    ref = oracle.run_ensemble(sc["vec"], sc["quat"], sc["cov"], None, 0, nominal_q(), st["imu"], oracle_streams(st), ev,
                              n_threads=NTHREADS, trace=True)
    prog = []
    for e, event in enumerate(ev):
        prog += [event, rec_op(e)]
    out = device_out(len(ev), STATE, range(7), N)
    with RBISBatch(N) as b:
        _setup(b, sc)
        b.set_record(out, STATE, range(7))
        b.run_fused(prog, imu=st["imu"], streams=gpu_streams(st))
        b.synchronize()
    rec = as_np(out)
    slot = np.array([(j * (j + 1) // 2 + i if i <= j else i * (i + 1) // 2 + j) for j in range(21) for i in range(21)])
    worst = 0.0
    for e in range(len(ev)):
        cov = rec[e, 26 + slot]   # element (i, j) at i + 21 j
        err = max_errors(rec[e, 0:21], rec[e, 21:25], cov, ref["trace_vec"][e], ref["trace_quat"][e], np.asarray(ref["trace_cov"][e]))
        worst = max(worst, err["vec"], err["quat"], err["cov"])
    assert worst <= STEP_TOL, worst


def _stats_program(sc, every=10):
    st = sc["st"]
    prog, rows = [], 0
    for e, event in enumerate(st["events"]):
        prog.append(event)
        if e % every == every - 1:
            prog += [rec_op(rows), snap_op(rows)]
            rows += 1
    tv, tq = synth.truth_state_at(sc["truth"], 0)
    tvs = np.stack([np.asarray(tv, dtype=np.float64) + 1e-3 * k for k in range(rows)])
    tqs = np.tile(np.asarray(tq, dtype=np.float64), (rows, 1))
    return prog, rows, tvs, tqs


def _pinned(shape):
    import torch

    return torch.full(shape, float("nan"), dtype=torch.float64).pin_memory()


@pytest.mark.gpu
@pytest.mark.parametrize("N", [1000, 3000])
@pytest.mark.parametrize("chunk", [32, 256, 1024])
def test_stats_of_records_equal_stats_of_snapshots(N, chunk):
    import torch

    sc = scenario(N, 80)
    st = sc["st"]
    prog, rows, tv, tq = _stats_program(sc)
    cov = sc["cov"].copy()
    vec = sc["vec"].copy()
    vec[4, 17] = np.nan   # one poisoned filter: counted non-finite on both paths
    nch = (N + chunk - 1) // chunk
    for blocks in ((1, 2, 3), range(7)):
        out = device_out(rows, STATE, blocks, N)
        with RBISBatch(N, snapshot_slots=rows) as b:
            b.set_process_noise(*nominal_q())
            b.set_state(vec, sc["quat"], cov)
            b.set_record(out, STATE, blocks)
            b.run_fused(prog, imu=st["imu"], streams=gpu_streams(st))
            chunks, totals = _pinned((rows, nch, capi.NUM_STATS)), _pinned((rows, capi.NUM_STATS))
            b.wait(b.stats_records_enqueue(0, tv, tq, chunks, totals, chunk=chunk))
            snaps = []
            for r in range(rows):
                o = _pinned((nch, capi.NUM_STATS))
                b.wait(b.stats_snapshot_enqueue(r, tv[r], tq[r], o, chunk=chunk))
                snaps.append(o.numpy().copy())
            # a sub-range of rows: row r of the call is record row first_row + r
            sub = _pinned((2, nch, capi.NUM_STATS))
            b.wait(b.stats_records_enqueue(1, tv[1:3], tq[1:3], sub, None, chunk=chunk))
        got = chunks.numpy()
        assert np.array_equal(bits(got), bits(np.stack(snaps)))
        assert np.array_equal(bits(sub.numpy()), bits(got[1:3]))
        assert not got[..., 48:].any()   # reserved statistics are zero, also for chunks of fewer than 96 filters
        assert all(got[r, :, 45].sum() == 1.0 for r in range(rows))
        assert all(got[r, :, 46].sum() == N for r in range(rows))
        for r in range(rows):
            assert np.array_equal(bits(totals.numpy()[r]), bits(reduce_chunks(got[r])))
        del out
        torch.cuda.synchronize()


@pytest.mark.gpu
def test_stats_of_records_are_ordered_against_later_calls():
    """A pass enqueued right before a call that records different values into the SAME buffer still returns the first call's
    statistics; with two alternating buffers and no synchronise, every row is right."""
    N, T, CH = 20_000, 120, 30
    sc = scenario(N, T)
    chunk = 256
    nch = (N + chunk - 1) // chunk
    calls = []
    for k0 in range(0, T, CH):
        st = synth.make_streams(sc["truth"], N, k0, CH)
        prog, r = [], 0
        for e in st["events"]:
            prog.append(e)
            if e[0] == capi.OP_IMU and e[2] % 10 == 9:
                prog.append(rec_op(r))
                r += 1
        calls.append((st, prog, r))
    rows = max(c[2] for c in calls)
    tv = np.stack([np.linspace(0, 1, 21) * (1 + 0.1 * r) for r in range(rows)])
    tq = np.tile([1.0, 0.0, 0.0, 0.0], (rows, 1))

    def run(n_bufs, sync):
        outs = [device_out(rows, STATE, (1, 2, 3), N) for _ in range(n_bufs)]
        res = []
        with RBISBatch(N, mapping=1, launch_groups=6, piece_ops=64) as b:
            _setup(b, sc)
            for c, (st, prog, r) in enumerate(calls):
                b.set_record(outs[c % n_bufs], STATE, (1, 2, 3))
                b.run_fused(prog, imu=st["imu"], streams=gpu_streams(st))
                o = _pinned((r, nch, capi.NUM_STATS))
                t = b.stats_records_enqueue(0, tv[:r], tq[:r], o, None, chunk=chunk)
                if sync:
                    b.wait(t)
                res.append(o)
            b.synchronize()
            return [o.numpy().copy() for o in res]

    ref = run(1, True)
    for n_bufs in (1, 2):
        got = run(n_bufs, False)
        for g, w in zip(got, ref):
            assert np.array_equal(bits(g), bits(w))
    assert len({bits(g).tobytes() for g in ref}) == len(ref)   # the calls' statistics differ


@pytest.mark.gpu
def test_stats_of_records_errors_leave_handle_and_ensemble_unchanged():
    import torch

    N, T = 256, 30
    sc = scenario(N, T)
    st = sc["st"]
    ev = st["events"]
    tv, tq = np.zeros((2, 21)), np.tile([1.0, 0, 0, 0], (2, 1))
    nch = N // 256
    chunks = _pinned((2, nch, capi.NUM_STATS))
    with RBISBatch(N) as b:
        _setup(b, sc)
        b.run_fused(ev[:10], imu=st["imu"], streams=gpu_streams(st))
        before = b.get_state()
        with pytest.raises(capi.RBISError, match="rbis error -4: .*no record set"):
            b.stats_records_enqueue(0, tv, tq, chunks, chunk=256)
        launches = b.launch_count
        good = device_out(4, STATE, (1, 2, 3), N)
        cases = [(pinned_out(4, STATE, (1, 2, 3), N), STATE, (1, 2, 3), 0, "device memory"),
                 (device_out(4, STATE & ~(1 << 25), (1, 2, 3), N), STATE & ~(1 << 25), (1, 2, 3), 0, "fields 0..25"),
                 (device_out(4, STATE, (1, 3), N), STATE, (1, 3), 0, "blocks 1, 2 and 3"),
                 (good, STATE, (1, 2, 3), 3, "outside"),
                 (good, STATE, (1, 2, 3), -1, "outside")]
        for out, fields, blocks, first, msg in cases:
            b.set_record(out, fields, blocks)
            with pytest.raises(capi.RBISError, match=f"rbis error -1: .*{msg}"):
                b.stats_records_enqueue(first, tv, tq, chunks, chunk=256)
        assert b.launch_count == launches
        # cov_blocks bit 7 is refused and leaves the current set in place
        rec = capi.Record()
        rec.fields, rec.out, rec.rows, rec.mem, rec.cov_blocks = STATE, good.data_ptr(), 4, capi.MEM_DEVICE, 0x8E
        assert b.lib.rbis_batch_set_record(b.h, C.byref(rec)) == -1
        rec.fields, rec.cov_blocks = 0, 0
        assert b.lib.rbis_batch_set_record(b.h, C.byref(rec)) == -1
        rec.cov_blocks = 0x2
        assert b.lib.rbis_batch_set_record(b.h, C.byref(rec)) == 0   # covariance only
        b.set_record(good, STATE, (1, 2, 3))
        _equal_state(before, b.get_state())
        assert np.isnan(as_np(good)).all()
        b.run_fused([rec_op(2), rec_op(3)], imu=st["imu"], streams=gpu_streams(st))
        b.wait(b.stats_records_enqueue(2, tv, tq, chunks, chunk=256))
        assert not np.isnan(chunks.numpy()).any()
        _equal_state(before, b.get_state())
        torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("mapping", [1, 4])
def test_filter_states_from_record_equal_get_filter_states(mapping):
    sc, streams, ops, at = _rewind_program()
    st, N = sc["st"], sc["vec"].shape[1]
    cut = at[len(at) // 2]
    out = device_out(1, STATE, range(7), N)
    with RBISBatch(N, snapshot_slots=3, mapping=mapping) as b:
        _setup(b, sc)
        b.set_record(out, STATE, range(7))
        b.run_fused(list(ops[:cut + 1]) + [rec_op(0)], imu=st["imu"], streams=streams)
        b.synchronize()
        want = (capi.FilterState * N)()
        capi.check(b.lib.rbis_batch_get_filter_states(b.h, 0, N, want))
        utime = b.get_state()[4]
    got = filter_states_from_record(as_np(out)[0], STATE, range(7), utime=utime)
    assert C.sizeof(got) == C.sizeof(want)
    assert bytes(got) == bytes(want)
