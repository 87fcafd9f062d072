"""Innovation sets (rbis_batch_set_innovations, rbis_batch_stats_innovations_enqueue, include/rbis_batch.h).

Every MEAS op on a stream with an innovation set writes, per filter, the NIS y^T S^-1 y, the innovation y = z - x-[idx] and
S(a,a) = P-(idx_a, idx_a) + R(a,a) of its update, from the prior state.  The yardsticks: numpy formed from the oracle's traced
priors (and the oracle's own log-likelihood step, log det S + NIS), bit identity across every kernel mapping and launch path,
no effect on anything else, and a numpy restatement of the statistics tree."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from pronto_b200 import MeasStream, RBISBatch, SynthSpec, capi, innovation_layout, reduce_chunks, synth

from common import nominal_q, scenario

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NTHREADS = min(16, os.cpu_count() or 1)
ALL = capi.INNOV_NIS | capi.INNOV_Y | capi.INNOV_S_DIAG
YAW_IDX = [17, 8]
REC_ALL = (1 << capi.REC_FIELDS) - 1
INNOV_VARIANT = 1024


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
def test_header_constants_match_capi():
    with open(os.path.join(ROOT, "include", "rbis_batch.h")) as f:
        text = f.read()
    for name, v in (("NIS", capi.INNOV_NIS), ("Y", capi.INNOV_Y), ("S_DIAG", capi.INNOV_S_DIAG)):
        assert re.search(rf"#define RBIS_INNOV_{name}\s+{v}\b", text), name
    assert "int rbis_batch_set_innovations(rbis_batch_t* h, int32_t stream, const rbis_innovation_t* spec);" in text


def test_innovation_struct_layout():
    assert C.sizeof(capi.Innovation) == 24
    assert (capi.Innovation.fields.offset, capi.Innovation.m.offset, capi.Innovation.out.offset, capi.Innovation.rows.offset) == (0, 4, 8, 16)
    assert capi.Innovation.fields.size == 4 and capi.Innovation.m.size == 4


def test_innovation_layout():
    assert innovation_layout(3, ALL) == ["nis", "y0", "y1", "y2", "s0", "s1", "s2"]
    assert innovation_layout(2, capi.INNOV_NIS) == ["nis"]
    assert innovation_layout(2, capi.INNOV_Y | capi.INNOV_S_DIAG) == ["y0", "y1", "s0", "s1"]
    assert innovation_layout(9, capi.INNOV_S_DIAG) == [f"s{a}" for a in range(9)]
    for m, f in ((0, ALL), (10, ALL), (3, 0), (3, 8)):
        with pytest.raises(ValueError):
            innovation_layout(m, f)


def test_chi2_bounds_of_the_kernel_match_scipy():
    """The 2.5 % / 97.5 % quantiles the statistics kernel counts against, to the digits stored."""
    from scipy.stats import chi2

    with open(os.path.join(ROOT, "pronto_b200", "csrc", "rbis_stats.cuh")) as f:
        text = f.read()
    for name, p in (("c_chi2_lo", 0.025), ("c_chi2_hi", 0.975)):
        body = re.search(rf"{name}\[9\] = \{{([^}}]*)\}}", text).group(1)
        vals = [v.strip() for v in body.split(",")]
        assert len(vals) == 9
        for m, s in enumerate(vals, start=1):
            digits = len(s.replace(".", "").lstrip("0"))
            want = chi2.ppf(p, m)
            assert float(f"{want:.{digits}g}") == float(s), (name, m, s, want)


# ------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------
def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def same_bits(a, b):
    return np.array_equal(bits(a), bits(b))


def yaw_streams(sc, k_block, k_diag, seed=5):
    """Two yaw locks on [17, 8] with the measured orientation, added to leg odometry (0) and pose (1): stream 2 with a
    correlated 2x2 R per row (one correlated block), stream 3 with a per-filter diagonal R (two one-row chunks).  Returns
    (stream dicts, arrival-ordered events)."""
    rng = np.random.default_rng(seed)
    truth, st = sc["truth"], sc["st"]
    N = sc["vec"].shape[1]
    out = [dict(idx=synth.LEGODO_IDX, z=st["legodo"], R=st["R_legodo"]),
           dict(idx=synth.POSE_IDX, z=st["pose_z"], R=st["R_pose"], quat=st["pose_q"])]
    for s, ks in ((2, k_block), (3, k_diag)):
        k = np.asarray(ks, dtype=int)
        z = np.zeros((len(k), 2, N))
        z[:, 0] = synth.NOMINAL["bg"][2] + 1e-4 * rng.normal(size=(len(k), N))
        q = np.ascontiguousarray(np.repeat(truth["quat"][k][:, :, None], N, axis=2))
        if s == 2:
            R = np.empty((len(k), 2, 2))
            for i in range(len(k)):
                a, c = (1e-4 * (1 + i % 3)) ** 2, (0.002 * (1 + i % 2)) ** 2
                R[i] = [[a, 0.4 * np.sqrt(a * c)], [0.4 * np.sqrt(a * c), c]]
            out.append(dict(idx=YAW_IDX, z=z, quat=q, R=R))
        else:
            R = np.stack([np.full(N, 2e-4 ** 2), np.full(N, 0.003 ** 2)]) * (1 + rng.random((2, N)))
            out.append(dict(idx=YAW_IDX, z=z, quat=q, R=np.ascontiguousarray(R), per_filter_diag=True))
    at = {}
    for s, ks in ((2, k_block), (3, k_diag)):
        for r, kk in enumerate(ks):
            at.setdefault(int(kk), []).append((s, r))
    ev = []
    for e in st["events"]:
        ev.append(tuple(e))
        if e[0] == capi.OP_IMU:
            for s, r in at.get(int(st["steps"][e[2]]), []):
                ev.append((capi.OP_MEAS, s, r, e[3], 0.0))
    return out, ev


def gpu(streams, skip=False, f=lambda a: a):
    return [MeasStream(d["idx"], f(d["z"]), d["R"], quat=None if d.get("quat") is None else f(d["quat"]),
                       per_filter_diag=d.get("per_filter_diag", False), skip_nan_rows=skip) for d in streams]


def n_rows(streams):
    return [d["z"].shape[0] for d in streams]


def innov_out(rows, m, N, fields=ALL):
    import torch

    return torch.full((max(rows, 1), len(innovation_layout(m, fields)), N), float("nan"), dtype=torch.float64, device="cuda")


def run(sc, streams, ops, sets=None, rec=0, skip=False, maps=None, f=lambda a: a, N=None, **cfg):
    """One handle: innovation sets on the streams in `sets` ({stream: fields}, default all streams with ALL), optional records.
    -> dict(state, innov {s: numpy}, rec, variant)."""
    N = sc["vec"].shape[1] if N is None else N
    sets = {s: ALL for s in range(len(streams))} if sets is None else sets
    import torch

    with RBISBatch(N, **cfg) as b:
        b.set_process_noise(*nominal_q())
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        for w, cmap, cols in (maps or ()):
            b.set_column_map(w, cmap, cols)
        outs = {}
        for s, fl in sets.items():
            outs[s] = innov_out(n_rows(streams)[s], len(streams[s]["idx"]), N, fl)
            b.set_innovations(s, outs[s], len(streams[s]["idx"]), fl)
        ro = None
        if rec:
            ro = torch.full((rec, capi.REC_FIELDS, N), float("nan"), dtype=torch.float64, device="cuda")
            b.set_record(ro, REC_ALL)
        b.run_fused(ops, imu=f(sc["st"]["imu"]), streams=gpu(streams, skip, f))
        b.synchronize()
        return dict(state=b.get_state(), innov={s: o.cpu().numpy() for s, o in outs.items()},
                    rec=None if ro is None else ro.cpu().numpy(), variant=b.last_kernel_variant)


def same_innov(a, b):
    assert a.keys() == b.keys()
    for s in a:
        assert same_bits(a[s], b[s]), s


def subtract_quats(q1, q2):
    """Log(q2^-1 q1) for [4][N] quaternions (oracle/rbis_numpy.py:subtract_quats, vectorised)."""
    from oracle import rbis_numpy as rn

    return np.stack([rn.subtract_quats(q1[:, n], q2[:, n]) for n in range(q1.shape[1])], axis=1)


def oracle_events(streams, ev):
    """The oracle takes one shared R per stream: every row of a per-row R stream becomes a stream of its own."""
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
    out = []
    for e in ev:
        if e[0] == capi.OP_MEAS:
            e = (e[0], where[e[1]], e[2]) + tuple(e[3:]) if e[1] in where else (e[0], where[(e[1], e[2])], 0) + tuple(e[3:])
        out.append(e)
    return split, out


def bundle(sc, vec, quat, cov):
    return dict(sc, vec=vec, quat=quat, cov=cov)


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_innovations_against_the_oracle(oracle):
    """y, S(a,a) and NIS of every MEAS op against numpy formed from the oracle's traced priors, and log det S + NIS against
    the oracle's own log-likelihood step: aligned triples, pose with orientation (m = 6), a yaw lock with a correlated R per row
    (one correlated block) and one with a per-filter diagonal R (one-row chunks)."""
    N, T = 64, 240
    sc = scenario(N, T, tumbling=True)
    streams, ev = yaw_streams(sc, range(5, T, 11), range(9, T, 13))
    got = run(sc, streams, ev)
    assert got["variant"] & 8
    split, oev = oracle_events(streams, ev)
    ref = oracle.run_ensemble(sc["vec"], sc["quat"], sc["cov"], None, 0, nominal_q(), sc["st"]["imu"], split, oev,
                              n_threads=NTHREADS, trace=True)
    worst = dict(y=0.0, s=0.0, nis=0.0, ll=0.0)
    seen = set()
    for e, op in enumerate(ev):
        if op[0] != capi.OP_MEAS:
            continue
        s, r = op[1], op[2]
        d = streams[s]
        idx = np.asarray(d["idx"])
        m = len(idx)
        if e == 0:
            pv, pq, pc, pll = sc["vec"], sc["quat"], sc["cov"], np.zeros(N)
        else:
            pv, pq, pc, pll = ref["trace_vec"][e - 1], ref["trace_quat"][e - 1], ref["trace_cov"][e - 1], ref["trace_loglik"][e - 1]
        P = pc.reshape(21, 21, N)   # element (r, c) at r + 21 c: P[c, r]
        y = d["z"][r] - pv[idx]
        if d.get("quat") is not None:
            dq = subtract_quats(d["quat"][r], pq)
            for a, i in enumerate(idx):
                if 6 <= i <= 8:
                    y[a] = dq[i - 6]
        R = np.asarray(d["R"])
        nis, logdet, sdiag = np.empty(N), np.empty(N), np.empty((m, N))
        for n in range(N):
            Rn = R[r] if R.ndim == 3 else np.diag(R[:, n]) if d.get("per_filter_diag") else R
            S = Rn + P[np.ix_(idx, idx, [n])][:, :, 0].T
            sdiag[:, n] = np.diag(S)
            nis[n] = y[:, n] @ np.linalg.solve(S, y[:, n])
            logdet[n] = np.log(np.linalg.det(S))
        g = got["innov"][s][r]
        rel = lambda a, b: float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))
        worst["y"] = max(worst["y"], float(np.max(np.abs(g[1:1 + m] - y) / np.maximum(np.abs(y), 1e-3 * np.abs(y).max() + 1e-300))))
        worst["s"] = max(worst["s"], rel(g[1 + m:], sdiag))
        worst["nis"] = max(worst["nis"], float(np.max(np.abs(g[0] - nis) / np.maximum(1.0, nis))))
        step = -(ref["trace_loglik"][e] - pll)
        worst["ll"] = max(worst["ll"], float(np.max(np.abs(logdet + g[0] - step) / np.maximum(1.0, np.abs(step)))))
        seen.add(s)
    assert seen == {0, 1, 2, 3}
    assert worst["y"] <= 1e-9 and worst["s"] <= 1e-9 and worst["nis"] <= 1e-9 and worst["ll"] <= 1e-9, worst


@pytest.mark.gpu
def test_bits_do_not_depend_on_mapping_or_kernel_variant():
    N, T = 300, 200
    sc = scenario(N, T, tumbling=True)
    streams, ev = yaw_streams(sc, range(5, T, 11), range(9, T, 13))
    ref = run(sc, streams, ev, mapping=1)
    assert ref["variant"] & 2   # decoupled
    for cfg in (dict(mapping=1, dense_only=True), dict(mapping=1, lane_filters_per_cta=256), dict(mapping=1, lane_filters_per_cta=128),
                dict(mapping=2), dict(mapping=4), dict(mapping=8), dict(mapping=16), dict(mapping=4, dense_only=True)):
        got = run(sc, streams, ev, **cfg)
        same_innov(got["innov"], ref["innov"])
    # triples only: the lane kernels without the one-row / correlated paths
    ref = run(sc, streams[:2], [e for e in ev if e[0] != capi.OP_MEAS or e[1] < 2])
    assert not ref["variant"] & 1
    got = run(sc, streams[:2], [e for e in ev if e[0] != capi.OP_MEAS or e[1] < 2], mapping=1, dense_only=True)
    same_innov(got["innov"], ref["innov"])


@pytest.mark.gpu
@pytest.mark.parametrize("mapping", [1, 4])
def test_innovation_sets_change_nothing_else(mapping):
    """State, quaternion, covariance, log-likelihood and records are bit-identical with and without innovation sets."""
    N, T = 257, 200
    sc = scenario(N, T, tumbling=True)
    streams, ev = yaw_streams(sc, range(5, T, 11), range(9, T, 13))
    prog, row = [], 0
    for i, e in enumerate(ev):
        prog.append(e)
        if i % 5 == 4:
            prog.append((capi.OP_RECORD, 0, row, 0, 0.0))
            row += 1
    for p, rec in ((ev, 0), (prog, row)):
        a = run(sc, streams, p, sets={}, rec=rec, mapping=mapping)
        b = run(sc, streams, p, rec=rec, mapping=mapping)
        c = run(sc, streams, p, sets={1: capi.INNOV_NIS, 3: capi.INNOV_Y}, rec=rec, mapping=mapping)
        # programs that only record run the REC kernels without the innovation path (+1024)
        assert bool(a["variant"] & 8) == bool(rec) and not a["variant"] & INNOV_VARIANT
        assert b["variant"] & (8 | INNOV_VARIANT) == 8 | INNOV_VARIANT and c["variant"] & (8 | INNOV_VARIANT) == 8 | INNOV_VARIANT
        for x in (b, c):
            for u, v in zip(a["state"][:4], x["state"][:4]):
                assert same_bits(u, v)
            if rec:
                assert same_bits(a["rec"], x["rec"])
        assert same_bits(c["innov"][1], b["innov"][1][:, :1])
        assert same_bits(c["innov"][3], b["innov"][3][:, 1:3])


@pytest.mark.gpu
def test_launch_groups_and_pieces_give_the_same_rows():
    N, T = 3000, 300
    sc = scenario(N, T)
    streams, ev = yaw_streams(sc, range(5, T, 11), range(9, T, 13))
    ref = run(sc, streams, ev)
    for cfg in (dict(launch_groups=4, piece_ops=64), dict(launch_groups=3, piece_ops=100, mapping=4)):
        got = run(sc, streams, ev, **cfg)
        same_innov(got["innov"], ref["innov"])


@pytest.mark.gpu
@pytest.mark.parametrize("mapping", [1, 8])
def test_skipped_rows_hold_nan(mapping):
    """Filters that skip a row write NaN into all its entries; filters that skip nothing write the rows of the unflagged program,
    and every filter's rows before its first skip are those of the unflagged program."""
    N, T = 200, 240
    sc = scenario(N, T)
    streams, ev = yaw_streams(sc, range(5, T, 11), range(9, T, 13))
    rng = np.random.default_rng(4)
    flagged = []
    first = {}
    for s, d in enumerate(streams):
        d = dict(d)
        z = d["z"].copy()
        miss = (rng.random((z.shape[0], N)) < 0.15) & (np.arange(N) % 3 == 0)
        cols = [a for a, i in enumerate(d["idx"]) if not (d.get("quat") is not None and 6 <= i <= 8)]
        r, n = np.nonzero(miss)
        z[r, np.asarray(cols)[rng.integers(0, len(cols), len(r))], n] = np.nan
        d["z"] = z
        flagged.append(d)
        first[s] = miss
    got = run(sc, flagged, ev, skip=True, mapping=mapping)
    ref = run(sc, streams, ev, mapping=mapping)
    assert got["variant"] & 512 and got["variant"] & 8
    # the op index of each filter's first skip
    first_skip = np.full(N, len(ev))
    for e, op in enumerate(ev):
        if op[0] == capi.OP_MEAS:
            hit = first[op[1]][op[2]] & (first_skip == len(ev))
            first_skip[hit] = e
    clean = first_skip == len(ev)
    assert clean.sum() > N // 2 and (~clean).sum() > 10
    for e, op in enumerate(ev):
        if op[0] != capi.OP_MEAS:
            continue
        s, r = op[1], op[2]
        g, w = got["innov"][s][r], ref["innov"][s][r]
        miss = first[s][r]
        assert np.isnan(g[:, miss]).all()
        before = e <= first_skip
        keep = ~miss & before
        assert same_bits(g[:, keep], w[:, keep])


@pytest.mark.gpu
@pytest.mark.parametrize("materialize", [False, True])
def test_fused_synthesis_equals_synthesize_then_run_fused(materialize):
    import torch

    N, T = 300, 220
    sc = scenario(N, T)
    st = sc["st"]
    ev = st["events"]
    d = synth.synth_spec_inputs(sc["truth"], 0, T)
    rows = [st["legodo"].shape[0], st["pose_z"].shape[0]]
    outs = [[innov_out(rows[s], (3, 6)[s], N) for s in range(2)] for _ in range(2)]
    with RBISBatch(N, synth_materialize=materialize) as b:
        b.set_process_noise(*nominal_q())
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        spec = SynthSpec(synth.SEED, d["imu_mean"], d["imu_step"], d["streams"], mode=1)
        for s in range(2):
            b.set_innovations(s, outs[0][s], (3, 6)[s])
        b.run_fused_synth(ev, [MeasStream(synth.LEGODO_IDX, None, st["R_legodo"]), MeasStream(synth.POSE_IDX, None, st["R_pose"], quat=True)],
                          spec)
        assert bool(b.last_kernel_variant & 4) == (not materialize) and b.last_kernel_variant & 8
        gen = b.synthesize(spec)
        b.set_process_noise(*nominal_q())
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        for s in range(2):
            b.set_innovations(s, outs[1][s], (3, 6)[s])
        b.run_fused(ev, imu=gen["imu"], streams=[MeasStream(synth.LEGODO_IDX, gen["z"][0], st["R_legodo"]),
                                                  MeasStream(synth.POSE_IDX, gen["z"][1], st["R_pose"], quat=gen["quat"][1])])
        b.synchronize()
    for s in range(2):
        a, c = outs[0][s].cpu().numpy(), outs[1][s].cpu().numpy()
        assert not np.isnan(a).any()
        assert same_bits(a, c)
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("mapping", [1, 4])
def test_rewinds_hold_the_replayed_values(mapping):
    """Late pose fixes planned into RESTORE + replay: every row equals the in-order program's row over the same history."""
    from pronto_b200.schedule import program_from_arrivals

    N, T = 256, 400
    sc = scenario(N, T)
    streams, ev = yaw_streams(sc, range(5, T, 11), range(9, T, 13))
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
    got = run(sc, streams, ops, snapshot_slots=4, mapping=mapping)
    ref = run(sc, streams, ev, snapshot_slots=4, mapping=mapping)
    same_innov(got["innov"], ref["innov"])
    for u, v in zip(got["state"][:4], ref["state"][:4]):
        assert same_bits(u, v)


@pytest.mark.gpu
@pytest.mark.parametrize("mapping", [1, 4])
def test_column_maps_and_float_rows(mapping):
    """Innovations stay per filter under column maps; float rows are widened exactly."""
    C_, G_ = 16, 8
    M = C_ * G_
    sc = scenario(C_, 160)
    cmap = (np.arange(M) % C_).astype(np.int32)
    ex = lambda a: np.ascontiguousarray(a[..., cmap])
    f32 = lambda a: np.ascontiguousarray(ex(a), dtype=np.float32)
    streams = [dict(idx=synth.LEGODO_IDX, z=sc["st"]["legodo"], R=sc["st"]["R_legodo"]),
               dict(idx=synth.POSE_IDX, z=sc["st"]["pose_z"], R=sc["st"]["R_pose"], quat=sc["st"]["pose_q"])]
    big = bundle(sc, ex(sc["vec"]), ex(sc["quat"]), ex(sc["cov"]))
    ev = sc["st"]["events"]
    mapped = run(big, streams, ev, N=M, maps=[(w, cmap, C_) for w in (-1, 0, 1)], mapping=mapping)
    expanded = run(big, streams, ev, N=M, f=ex, mapping=mapping)
    floats = run(big, streams, ev, N=M, f=f32, mapping=mapping)
    widened = run(big, streams, ev, N=M, f=lambda a: f32(a).astype(np.float64), mapping=mapping)
    assert not np.isnan(mapped["innov"][0]).any()
    same_innov(mapped["innov"], expanded["innov"])
    same_innov(floats["innov"], widened["innov"])


@pytest.mark.gpu
def test_ensemble_average_nis_is_near_m():
    """4,096 filters whose noise matches R and Q: the ensemble-average NIS over the run lies within 25 % of m for every stream
    (loose on purpose: the filter is not exactly consistent, SURVEY.md Appendix B)."""
    N, T = 4096, 1000
    sc = scenario(N, T)
    streams = [dict(idx=synth.LEGODO_IDX, z=sc["st"]["legodo"], R=sc["st"]["R_legodo"]),
               dict(idx=synth.POSE_IDX, z=sc["st"]["pose_z"], R=sc["st"]["R_pose"], quat=sc["st"]["pose_q"])]
    got = run(sc, streams, sc["st"]["events"], sets={0: capi.INNOV_NIS, 1: capi.INNOV_NIS})
    for s, m in ((0, 3), (1, 6)):
        nis = got["innov"][s][:, 0]
        assert np.isfinite(nis).all()
        anis = float(nis.mean())
        assert abs(anis - m) <= 0.25 * m, (s, anis)


def stats_reference(rows, m, fields, chunk):
    """numpy restatement of innov_stats_kernel: per row [n_chunks][96], the fixed binary tree of each chunk."""
    from scipy.stats import chi2  # noqa: F401  (bounds come from the kernel's table, checked against scipy above)

    with open(os.path.join(ROOT, "pronto_b200", "csrc", "rbis_stats.cuh")) as f:
        text = f.read()
    lo = [float(v) for v in re.search(r"c_chi2_lo\[9\] = \{([^}]*)\}", text).group(1).split(",")][m - 1]
    hi = [float(v) for v in re.search(r"c_chi2_hi\[9\] = \{([^}]*)\}", text).group(1).split(",")][m - 1]
    R, k, N = rows.shape
    nch = (N + chunk - 1) // chunk
    out = np.zeros((R, nch, capi.NUM_STATS))
    with np.errstate(invalid="ignore", over="ignore"):
        for r in range(R):
            val = np.zeros((33, nch * chunk))
            nis = rows[r, 0]
            fin = np.isfinite(nis)
            v = val[:, :N]
            v[0] = np.where(fin, nis, 0.0)
            v[1] = np.where(fin, nis * nis, 0.0)
            v[2] = fin
            v[3] = fin & (nis >= lo) & (nis <= hi)
            v[4] = ~fin
            v[5] = 1.0
            if fields & capi.INNOV_Y:
                for a in range(m):
                    y = rows[r, 1 + a]
                    v[6 + a] = np.where(fin, y, 0.0)
                    v[15 + a] = np.where(fin, y * y, 0.0)
                    if fields & capi.INNOV_S_DIAG:
                        v[24 + a] = np.where(fin, (y * y) / rows[r, 1 + m + a], 0.0)
            t = val.reshape(33, nch, chunk).copy()
            w = chunk
            while w > 1:
                w //= 2
                t = t[:, :, :w] + t[:, :, w:2 * w]
            out[r, :, :33] = t[:, :, 0].T
    return out


def _pinned(shape):
    import torch

    return torch.full(shape, float("nan"), dtype=torch.float64).pin_memory()


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [32, 256, 1024])
def test_stats_equal_a_numpy_restatement_of_the_tree(chunk):
    """With a poisoned filter and skipped rows: every table bit for bit, totals equal rbis_stats_reduce_chunks, and the
    fields-only-NIS and NIS + y sets give their prefix of the statistics."""
    N, T = 3000, 120
    sc = scenario(N, T)
    vec = sc["vec"].copy()
    vec[4, 17] = np.nan
    streams = [dict(idx=synth.LEGODO_IDX, z=sc["st"]["legodo"].copy(), R=sc["st"]["R_legodo"]),
               dict(idx=synth.POSE_IDX, z=sc["st"]["pose_z"], R=sc["st"]["R_pose"], quat=sc["st"]["pose_q"])]
    streams[0]["z"][::3, 1, 100:160] = np.nan
    ev = sc["st"]["events"]
    nch = (N + chunk - 1) // chunk
    for fields in (ALL, capi.INNOV_NIS, capi.INNOV_NIS | capi.INNOV_Y):
        with RBISBatch(N) as b:
            b.set_process_noise(*nominal_q())
            b.set_state(vec, sc["quat"], sc["cov"])
            outs = []
            for s, m in ((0, 3), (1, 6)):
                outs.append(innov_out(streams[s]["z"].shape[0], m, N, fields))
                b.set_innovations(s, outs[s], m, fields)
            b.run_fused(ev, imu=sc["st"]["imu"], streams=gpu(streams, skip=True))
            res = []
            for s, m in ((0, 3), (1, 6)):
                R = streams[s]["z"].shape[0]
                ch, tot = _pinned((R, nch, capi.NUM_STATS)), _pinned((R, capi.NUM_STATS))
                b.wait(b.stats_innovations_enqueue(s, 0, ch, tot, chunk=chunk))
                sub = _pinned((R - 1, nch, capi.NUM_STATS))   # a sub-range: row r of the call is row 1 + r
                b.wait(b.stats_innovations_enqueue(s, 1, sub, None, chunk=chunk))
                res.append((ch.numpy().copy(), tot.numpy().copy(), sub.numpy().copy()))
            b.synchronize()
            rows = [o.cpu().numpy() for o in outs]
        for s, m in ((0, 3), (1, 6)):
            ch, tot, sub = res[s]
            want = stats_reference(rows[s], m, fields, chunk)
            assert same_bits(ch, want), (fields, s)
            assert same_bits(sub, ch[1:])
            assert (ch[..., 5].sum(axis=1) == N).all()
            assert (ch[..., 4].sum(axis=1) >= 1).all()   # the poisoned filter
            for r in range(ch.shape[0]):
                assert same_bits(tot[r], reduce_chunks(ch[r]))
        assert res[0][0][::3, :, 4].sum(axis=1).min() >= 61   # skipped rows count as non-finite


@pytest.mark.gpu
def test_pending_stats_are_not_overwritten_by_later_calls():
    """A pass enqueued right before calls that write the same rows of the same buffer still returns the first call's values."""
    N, T, CH = 20_000, 120, 30
    sc = scenario(N, T)
    chunk = 256
    nch = (N + chunk - 1) // chunk
    calls = [synth.make_streams(sc["truth"], N, k0, CH) for k0 in range(0, T, CH)]

    def go(n_bufs, sync):
        import torch

        R = calls[0]["legodo"].shape[0]
        bufs = [torch.full((R, 7, N), float("nan"), dtype=torch.float64, device="cuda") for _ in range(n_bufs)]
        res = []
        with RBISBatch(N, launch_groups=6, piece_ops=64) as b:
            b.set_process_noise(*nominal_q())
            b.set_state(sc["vec"], sc["quat"], sc["cov"])
            for c, st in enumerate(calls):
                b.set_innovations(0, bufs[c % n_bufs], 3)
                b.run_fused(st["events"], imu=st["imu"], streams=[MeasStream(synth.LEGODO_IDX, st["legodo"], st["R_legodo"]),
                                                                  MeasStream(synth.POSE_IDX, st["pose_z"], st["R_pose"], quat=st["pose_q"])])
                o = _pinned((R, nch, capi.NUM_STATS))
                t = b.stats_innovations_enqueue(0, 0, o, None, chunk=chunk)
                if sync:
                    b.wait(t)
                res.append(o)
            b.synchronize()
            return [o.numpy().copy() for o in res]

    ref = go(1, True)
    for n_bufs in (1, 2):
        for g, w in zip(go(n_bufs, False), ref):
            assert same_bits(g, w)
    assert len({bits(g).tobytes() for g in ref}) == len(ref)


@pytest.mark.gpu
def test_errors_are_refused_before_anything_is_enqueued():
    import torch

    N, T = 64, 60
    sc = scenario(N, T)
    st = sc["st"]
    streams = [MeasStream(synth.LEGODO_IDX, st["legodo"], st["R_legodo"]), MeasStream(synth.POSE_IDX, st["pose_z"], st["R_pose"], quat=st["pose_q"])]
    rows = st["legodo"].shape[0]
    with RBISBatch(N) as b:
        b.set_process_noise(*nominal_q())
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        before = b.get_state()
        launches = b.launch_count
        lib, h = b.lib, b.h
        good = torch.zeros((rows, 7, N), dtype=torch.float64, device="cuda")

        def spec(fields=ALL, m=3, out=good.data_ptr(), n=rows):
            s = capi.Innovation()
            s.fields, s.m, s.out, s.rows = fields, m, out, n
            return C.byref(s)

        host = np.zeros((rows, 7, N))
        for stream, sp in ((-1, spec()), (8, spec()), (0, spec(fields=0)), (0, spec(fields=8)), (0, spec(m=0)), (0, spec(m=10)),
                           (0, spec(out=None)), (0, spec(out=host.ctypes.data)), (0, spec(n=0))):
            assert lib.rbis_batch_set_innovations(h, stream, sp) == -1   # RBIS_ERR_INVALID
        # m mismatch with the call's stream, and a MEAS row outside [0, rows)
        b.set_innovations(1, torch.zeros((20, 13, N), dtype=torch.float64, device="cuda"), 6)
        b.set_innovations(0, torch.zeros((2, 7, N), dtype=torch.float64, device="cuda"), 3)
        with pytest.raises(Exception):
            b.run_fused(st["events"], imu=st["imu"], streams=streams)
        b.set_innovations(0, good, 3)
        b.set_innovations(1, torch.zeros((20, 7, N), dtype=torch.float64, device="cuda"), 3, ALL)
        with pytest.raises(Exception):
            b.run_fused(st["events"], imu=st["imu"], streams=streams)
        # statistics: no set, no NIS field, rows out of range, bad chunk
        b.clear_innovations(1)
        o = _pinned((1, 1, capi.NUM_STATS))
        with pytest.raises(Exception):
            b.stats_innovations_enqueue(1, 0, o, chunk=1024)
        b.set_innovations(1, torch.zeros((20, 12, N), dtype=torch.float64, device="cuda"), 6, capi.INNOV_Y | capi.INNOV_S_DIAG)
        with pytest.raises(Exception):
            b.stats_innovations_enqueue(1, 0, o, chunk=1024)
        with pytest.raises(Exception):
            b.stats_innovations_enqueue(0, rows, o, chunk=1024)
        with pytest.raises(Exception):
            b.stats_innovations_enqueue(0, 0, _pinned((1, 2, capi.NUM_STATS)), chunk=48)
        b.synchronize()
        assert b.launch_count == launches
        after = b.get_state()
        for u, v in zip(before[:4], after[:4]):
            assert same_bits(u, v)
        # the single-update entry points ignore innovation sets, and so does a call with fewer streams than the set's slot
        b.clear_innovations(1)
        b.set_innovations(5, torch.zeros((1, 5, N), dtype=torch.float64, device="cuda"), 2)
        z = np.ascontiguousarray(st["legodo"][0])
        b.indexed_update(synth.LEGODO_IDX, z, st["R_legodo"])
        assert not b.last_kernel_variant & (8 | INNOV_VARIANT)
        b.clear_innovations(0)
        b.clear_innovations(1)
        b.run_fused(st["events"], imu=st["imu"], streams=streams)
        assert not b.last_kernel_variant & 8
        b.synchronize()
