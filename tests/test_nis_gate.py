"""NIS gates (rbis_batch_set_nis_gate, RBIS_INNOV_APPLIED, include/rbis_batch.h).

A gated stream makes every filter reject a row whose prior NIS y^T S^-1 y exceeds its threshold; a rejected filter keeps its
values exactly as for a missing row.  The yardsticks: the same program with the rejected rows made NaN under
RBIS_STREAM_SKIP_NAN_ROWS (bit for bit), numpy's NIS from the oracle's traced priors, an oracle replay whose per-filter
decisions numpy makes, bit identity across every mapping and launch path, and a numpy restatement of the statistics."""
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
APPLIED_SET = capi.INNOV_NIS | capi.INNOV_APPLIED
MASK_VARIANT, GATE_VARIANT = 512, 2048
REC_ALL = (1 << capi.REC_FIELDS) - 1


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
def test_header_constants_match_capi():
    with open(os.path.join(ROOT, "include", "rbis_batch.h")) as f:
        text = f.read()
    assert re.search(rf"#define RBIS_INNOV_APPLIED\s+{capi.INNOV_APPLIED}\b", text)
    assert capi.INNOV_APPLIED == 8
    assert "int rbis_batch_set_nis_gate(rbis_batch_t* h, int32_t stream, const rbis_nis_gate_t* gate);" in text
    assert "rbis_batch_set_nis_gate" in capi.PROTOTYPES


def test_nis_gate_struct_layout():
    assert C.sizeof(capi.NisGate) == 16
    assert (capi.NisGate.nis_max.offset, capi.NisGate.nis_max_per_filter.offset) == (0, 8)
    assert capi.NisGate.nis_max.size == 8 and capi.NisGate.nis_max_per_filter.size == 8


def test_innovation_layout_with_applied():
    assert innovation_layout(3, ALL | capi.INNOV_APPLIED) == ["nis", "y0", "y1", "y2", "s0", "s1", "s2", "applied"]
    assert innovation_layout(2, APPLIED_SET) == ["nis", "applied"]
    assert innovation_layout(1, capi.INNOV_Y | capi.INNOV_APPLIED) == ["y0", "applied"]
    for m, f in ((3, capi.INNOV_APPLIED), (3, 16), (3, ALL | 16)):
        with pytest.raises(ValueError):
            innovation_layout(m, f)


# ------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------
def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def same_bits(a, b):
    return np.array_equal(bits(a), bits(b))


def assert_state_bits(got, want, cols=None):
    for x, y in zip(got[:4], want[:4]):
        x, y = np.asarray(x), np.asarray(y)
        if cols is not None:
            x, y = x[..., cols], y[..., cols]
        assert same_bits(x, y)


def base_streams(sc):
    st = sc["st"]
    return [dict(idx=synth.LEGODO_IDX, z=st["legodo"], R=st["R_legodo"]),
            dict(idx=synth.POSE_IDX, z=st["pose_z"], R=st["R_pose"], quat=st["pose_q"])]


def with_outliers(streams, rng, frac=0.02, size=5.0, which=(1,)):
    """Copies of the streams with `size` metres added to the position rows (pose, indices 9..11) or to every readable value
    (leg odometry) of a random `frac` of the (row, filter) pairs.  -> (streams, {stream: bool [rows][N]})."""
    out, hit = [], {}
    for s, d in enumerate(streams):
        d = dict(d)
        if s in which:
            z = np.array(d["z"], dtype=np.float64, copy=True)
            h = rng.random((z.shape[0], z.shape[2])) < frac
            cols = [a for a, i in enumerate(d["idx"]) if 9 <= i <= 11] or list(range(len(d["idx"])))
            for a in cols:
                z[:, a, :] += np.where(h, size * rng.choice([-1.0, 1.0], size=h.shape), 0.0)
            d["z"] = z
            hit[s] = h
        out.append(d)
    return out, hit


def gpu(streams, skip=False, f=lambda a: a):
    return [MeasStream(d["idx"], f(d["z"]), d["R"], quat=None if d.get("quat") is None else f(d["quat"]),
                       per_filter_diag=d.get("per_filter_diag", False), skip_nan_rows=skip) for d in streams]


def run(sc, streams, ops, gates=None, sets=None, skip=False, rec=0, maps=None, f=lambda a: a, N=None, **cfg):
    """One handle.  gates: {stream: threshold (float) or per-filter numpy [N]}; sets: {stream: innovation fields} (default:
    NIS + APPLIED on every gated stream).  -> dict(state, innov {s: numpy}, rec, variant)."""
    import torch

    N = sc["vec"].shape[1] if N is None else N
    gates = gates or {}
    sets = {s: APPLIED_SET for s in gates} if sets is None else sets
    with RBISBatch(N, **cfg) as b:
        b.set_process_noise(*nominal_q())
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        for w, cmap, cols in (maps or ()):
            b.set_column_map(w, cmap, cols)
        for s, g in gates.items():
            if np.ndim(g) == 0:
                b.set_nis_gate(s, float(g))
            else:
                b.set_nis_gate(s, per_filter=torch.as_tensor(np.ascontiguousarray(g, dtype=np.float64), device="cuda"))
        outs = {}
        for s, fl in sets.items():
            m = len(streams[s]["idx"])
            outs[s] = torch.full((max(streams[s]["z"].shape[0], 1), len(innovation_layout(m, fl)), N), float("nan"),
                                 dtype=torch.float64, device="cuda")
            b.set_innovations(s, outs[s], m, fl)
        ro = None
        if rec:
            ro = torch.full((rec, capi.REC_FIELDS, N), float("nan"), dtype=torch.float64, device="cuda")
            b.set_record(ro, REC_ALL)
        b.run_fused(ops, imu=f(sc["st"]["imu"]), streams=gpu(streams, skip, f))
        b.synchronize()
        return dict(state=b.get_state(), innov={s: o.cpu().numpy() for s, o in outs.items()},
                    rec=None if ro is None else ro.cpu().numpy(), variant=b.last_kernel_variant)


def nan_rows(streams, rejected):
    """Copies of the streams whose z is NaN (every readable value) where rejected[s][row, n]."""
    out = []
    for s, d in enumerate(streams):
        d = dict(d)
        if s in rejected:
            z = np.array(d["z"], dtype=np.float64, copy=True)
            r, n = np.nonzero(rejected[s])
            for a, i in enumerate(d["idx"]):
                if not (d.get("quat") is not None and 6 <= i <= 8):
                    z[r, a, n] = np.nan
            d["z"] = z
        out.append(d)
    return out


def chi2_thr(m, p):
    from scipy.stats import chi2

    return float(chi2.ppf(p, m))


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
MAPPINGS = [dict(mapping=1), dict(mapping=1, dense_only=True), dict(mapping=2), dict(mapping=4), dict(mapping=8),
            dict(mapping=16), dict(mapping=4, dense_only=True)]


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", MAPPINGS, ids=lambda c: "-".join(f"{k}{v}" for k, v in c.items()))
def test_open_gate_changes_nothing(cfg):
    """A gate of +inf: state, covariance and log-likelihood bit-identical to the ungated program, APPLIED all 1."""
    N, T = 300, 240
    sc = scenario(N, T, tumbling=True)
    streams = base_streams(sc)
    ops = sc["st"]["events"]
    ref = run(sc, streams, ops, **cfg)
    got = run(sc, streams, ops, gates={0: np.inf, 1: np.inf}, **cfg)
    assert not ref["variant"] & GATE_VARIANT
    assert got["variant"] == ref["variant"] | MASK_VARIANT | GATE_VARIANT | 8 | 1024   # GATE, and INNOV for the APPLIED sets
    assert_state_bits(got["state"], ref["state"])
    for s in (0, 1):
        assert (got["innov"][s][:, 1] == 1.0).all()
        assert np.isfinite(got["innov"][s][:, 0]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", MAPPINGS, ids=lambda c: "-".join(f"{k}{v}" for k, v in c.items()))
def test_rejected_equals_missing(cfg):
    """Outliers in 3 % of the (row, filter) pairs of both streams, gates at chi2(0.999): the filters that rejected rows end,
    bit for bit, where the ungated program ends with those rows NaN under RBIS_STREAM_SKIP_NAN_ROWS."""
    N, T = 300, 300
    rng = np.random.default_rng(3)
    sc = scenario(N, T, tumbling=True)
    streams, hit = with_outliers(base_streams(sc), rng, frac=0.03, size=2.0, which=(0, 1))
    ops = sc["st"]["events"]
    got = run(sc, streams, ops, gates={0: chi2_thr(3, 0.999), 1: chi2_thr(6, 0.999)}, **cfg)
    rejected = {s: got["innov"][s][:, 1] == 0.0 for s in (0, 1)}
    for s in (0, 1):
        assert set(np.unique(got["innov"][s][:, 1])) <= {0.0, 1.0}
        assert rejected[s][hit[s]].mean() > 0.5       # the gate catches most outliers ...
        assert rejected[s][~hit[s]].mean() < 0.05     # ... and few clean rows
    ref = run(sc, nan_rows(streams, rejected), ops, skip=True, **cfg)
    assert_state_bits(got["state"], ref["state"])


def one_row_yaw(sc, ks, seed=9):
    """A one-row yaw lock on chi_z (index 8) with the measured orientation and a shared 1x1 R."""
    N = sc["vec"].shape[1]
    k = np.asarray(ks, dtype=int)
    q = np.ascontiguousarray(np.repeat(sc["truth"]["quat"][k][:, :, None], N, axis=2))
    return dict(idx=[8], z=np.zeros((len(k), 1, N)), quat=q, R=np.array([[0.003 ** 2]]))


def gate_streams(sc, T):
    """Leg odometry, pose, the two yaw locks of the innovation tests (correlated per-row R, per-filter diagonal R) and a one-row
    yaw lock -> (streams, events)."""
    from test_innovations import yaw_streams

    streams, ev = yaw_streams(sc, range(5, T, 11), range(9, T, 13))
    streams.append(one_row_yaw(sc, range(7, T, 17)))
    at = {int(k): r for r, k in enumerate(range(7, T, 17))}
    out = []
    for e in ev:
        out.append(tuple(e))
        if e[0] == capi.OP_IMU and int(sc["st"]["steps"][e[2]]) in at:
            out.append((capi.OP_MEAS, 4, at[int(sc["st"]["steps"][e[2]])], e[3], 0.0))
    return streams, out


def numpy_nis(d, r, pv, pq, pc):
    """y^T S^-1 y of row r of stream d for every filter, from the prior (pv [21][N], pq [4][N], pc [441][N])."""
    from test_innovations import subtract_quats

    N = pv.shape[1]
    idx = np.asarray(d["idx"])
    P = pc.reshape(21, 21, N)
    y = d["z"][r] - pv[idx]
    if d.get("quat") is not None:
        dq = subtract_quats(d["quat"][r], pq)
        for a, i in enumerate(idx):
            if 6 <= i <= 8:
                y[a] = dq[i - 6]
    R = np.asarray(d["R"])
    nis = np.empty(N)
    for n in range(N):
        Rn = R[r] if R.ndim == 3 else np.diag(R[:, n]) if d.get("per_filter_diag") else R
        S = Rn + P[np.ix_(idx, idx, [n])][:, :, 0].T
        nis[n] = y[:, n] @ np.linalg.solve(S, y[:, n])
    return nis


@pytest.mark.gpu
def test_nis_against_numpy_and_decisions_against_the_oracle(oracle):
    """Aligned triples, pose with orientation, a one-row yaw lock, a correlated per-row R and a per-filter diagonal R, with
    outliers: (a) an open gate's NIS equals numpy's from the oracle's traced priors to 1e-9 relative; (b) with finite gates,
    the final states equal an oracle replay per filter whose accept / reject decisions numpy makes from that replay's own
    priors, at the parity tolerances; no NIS lies within 1e-6 relative of its threshold."""
    from pronto_b200.parity import max_errors
    from test_innovations import oracle_events

    N, T = 24, 240
    rng = np.random.default_rng(21)
    sc = scenario(N, T, tumbling=True)
    streams, ev = gate_streams(sc, T)
    streams, _ = with_outliers(streams, rng, frac=0.05, size=1.0, which=(0, 1))
    S_ = len(streams)
    # (a) open gates: the gate's NIS on every row against numpy
    got = run(sc, streams, ev, gates={s: np.inf for s in range(S_)})
    split, oev = oracle_events(streams, ev)
    ref = oracle.run_ensemble(sc["vec"], sc["quat"], sc["cov"], None, 0, nominal_q(), sc["st"]["imu"], split, oev,
                              n_threads=NTHREADS, trace=True)
    worst = 0.0
    for e, op in enumerate(ev):
        if op[0] != capi.OP_MEAS:
            continue
        pv, pq, pc = ((sc["vec"], sc["quat"], sc["cov"]) if e == 0 else
                      (ref["trace_vec"][e - 1], ref["trace_quat"][e - 1], ref["trace_cov"][e - 1]))
        want = numpy_nis(streams[op[1]], op[2], pv, pq, pc)
        worst = max(worst, float(np.max(np.abs(got["innov"][op[1]][op[2], 0] - want) / np.maximum(np.abs(want), 1e-300))))
    assert worst <= 1e-9, worst
    # (b) finite gates: per filter, replay through the oracle and reject the first accepted row numpy's NIS fails, until none
    thr = {0: chi2_thr(3, 0.999), 1: chi2_thr(6, 0.999), 2: chi2_thr(2, 0.99), 3: chi2_thr(2, 0.99), 4: chi2_thr(1, 0.99)}
    gated = run(sc, streams, ev, gates=thr)
    one = lambda d, n: dict(d, z=d["z"][..., n:n + 1], quat=None if d.get("quat") is None else d["quat"][..., n:n + 1],
                            R=(np.asarray(d["R"])[:, n:n + 1] if d.get("per_filter_diag") else d["R"]))
    margin, n_rej = np.inf, 0
    fv, fq, fc, fl = (np.empty_like(sc["vec"]), np.empty_like(sc["quat"]), np.empty_like(sc["cov"]), np.empty(N))
    for n in range(N):
        sn = [one(d, n) for d in streams]
        keep = list(ev)
        while True:
            sp, oe = oracle_events(sn, keep)
            r1 = oracle.run_ensemble(sc["vec"][:, n:n + 1], sc["quat"][:, n:n + 1], sc["cov"][:, n:n + 1], None, 0, nominal_q(),
                                     sc["st"]["imu"][..., n:n + 1], sp, oe, trace=True)
            bad = None
            for e, op in enumerate(keep):
                if op[0] != capi.OP_MEAS:
                    continue
                pv, pq, pc = ((sc["vec"][:, n:n + 1], sc["quat"][:, n:n + 1], sc["cov"][:, n:n + 1]) if e == 0 else
                              (r1["trace_vec"][e - 1], r1["trace_quat"][e - 1], r1["trace_cov"][e - 1]))
                v = float(numpy_nis(sn[op[1]], op[2], pv, pq, pc)[0])
                margin = min(margin, abs(v - thr[op[1]]) / thr[op[1]])
                if not v <= thr[op[1]]:
                    bad = e
                    break
            if bad is None:
                break
            del keep[bad]
            n_rej += 1
        fv[:, n], fq[:, n], fc[:, n], fl[n] = r1["vec"][:, 0], r1["quat"][:, 0], r1["cov"][:, 0], r1["loglik"][0]
        want_rej = {s: set() for s in range(S_)}
        kept = {(o[1], o[2]) for o in keep if o[0] == capi.OP_MEAS}
        for o in ev:
            if o[0] == capi.OP_MEAS and (o[1], o[2]) not in kept:
                want_rej[o[1]].add(o[2])
        for s in range(S_):
            assert set(np.nonzero(gated["innov"][s][:, 1, n] == 0.0)[0].tolist()) == want_rej[s], (n, s)
    assert n_rej > 0
    assert margin > 1e-6, margin
    gv, gq, gP, gll, _ = gated["state"]
    err = max_errors(gv, gq, gP, fv, fq, fc)
    assert err["vec"] < 1e-8 and err["quat"] < 1e-8 and err["cov"] < 1e-8, err
    assert float(np.max(np.abs(gll - fl) / np.maximum(1.0, np.abs(fl)))) < 1e-8


@pytest.mark.gpu
@pytest.mark.parametrize("mapping", [1, 4])
def test_decisions_do_not_depend_on_how_the_program_runs(mapping):
    """A per-filter threshold sweep equals one scalar-threshold run per threshold; launch groups, pieces, column maps and float
    rows give the same decisions and values."""
    C_, G_ = 64, 4
    M = C_ * G_
    rng = np.random.default_rng(5)
    sc = scenario(C_, 200, tumbling=True)
    streams, _ = with_outliers(base_streams(sc), rng, frac=0.05, size=1.0, which=(0, 1))
    ev = sc["st"]["events"]
    cmap = (np.arange(M) % C_).astype(np.int32)
    ex = lambda a: np.ascontiguousarray(a[..., cmap])
    big = dict(sc, vec=ex(sc["vec"]), quat=ex(sc["quat"]), cov=ex(sc["cov"]))
    exp_streams = [dict(d, z=ex(d["z"]), quat=None if d.get("quat") is None else ex(d["quat"])) for d in streams]
    big_exp = dict(big, st=dict(sc["st"], imu=ex(sc["st"]["imu"])))
    levels = [chi2_thr(6, p) for p in (0.9, 0.99, 0.999, 0.9999)]
    thr = np.array([levels[n // C_] for n in range(M)])
    gates = lambda t: {0: chi2_thr(3, 0.999), 1: t}
    sweep = run(big_exp, exp_streams, ev, gates=gates(thr), mapping=mapping)
    for g, t in enumerate(levels):
        one = run(big_exp, exp_streams, ev, gates=gates(t), mapping=mapping)
        cols = np.arange(g * C_, (g + 1) * C_)
        assert_state_bits(sweep["state"], one["state"], cols)
        for s in (0, 1):
            assert same_bits(sweep["innov"][s][..., cols], one["innov"][s][..., cols])
    assert (sweep["innov"][1][:, 1] == 0.0).sum(axis=0)[:C_].sum() > (sweep["innov"][1][:, 1] == 0.0).sum(axis=0)[-C_:].sum()
    for cfg, kw in ((dict(launch_groups=4, piece_ops=64), {}), (dict(launch_groups=3, piece_ops=100), {}),
                    ({}, dict(maps=[(w, cmap, C_) for w in (-1, 0, 1)]))):
        src = (big, streams) if kw else (big_exp, exp_streams)
        other = run(*src, ev, gates=gates(thr), mapping=mapping, **cfg, **kw)
        assert_state_bits(other["state"], sweep["state"])
        for s in (0, 1):
            assert same_bits(other["innov"][s], sweep["innov"][s])
    f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)
    floats = run(big_exp, exp_streams, ev, gates=gates(thr), mapping=mapping, f=f32)
    widened = run(big_exp, exp_streams, ev, gates=gates(thr), mapping=mapping, f=lambda a: f32(a).astype(np.float64))
    assert_state_bits(floats["state"], widened["state"])
    for s in (0, 1):
        assert same_bits(floats["innov"][s], widened["innov"][s])


@pytest.mark.gpu
@pytest.mark.parametrize("mapping", [1, 8])
def test_missing_rows_and_nan_rows(mapping):
    """SKIP_NAN_ROWS with a gate: missing rows report NaN APPLIED, the others are gated; without the flag a NaN row is rejected
    by the gate.  Both equal the ungated SKIP_NAN_ROWS program with the rejected rows NaN as well."""
    N, T = 256, 240
    rng = np.random.default_rng(8)
    sc = scenario(N, T, tumbling=True)
    streams, _ = with_outliers(base_streams(sc), rng, frac=0.03, size=1.0, which=(0, 1))
    miss = {s: rng.random((streams[s]["z"].shape[0], N)) < 0.1 for s in (0, 1)}
    holed = nan_rows(streams, miss)
    ev = sc["st"]["events"]
    gates = {0: chi2_thr(3, 0.999), 1: chi2_thr(6, 0.999)}
    sets = {0: ALL | capi.INNOV_APPLIED, 1: ALL | capi.INNOV_APPLIED}
    flagged = run(sc, holed, ev, gates=gates, sets=sets, skip=True, mapping=mapping)
    unflagged = run(sc, holed, ev, gates=gates, sets=sets, skip=False, mapping=mapping)
    for s, m in ((0, 3), (1, 6)):
        fa, ua = flagged["innov"][s][:, -1], unflagged["innov"][s][:, -1]
        assert np.isnan(fa[miss[s]]).all() and set(np.unique(fa[~miss[s]])) <= {0.0, 1.0}
        assert (fa[~miss[s]] == 0.0).any()
        assert (ua[miss[s]] == 0.0).all()                      # NaN NIS: rejected
        assert (ua[~miss[s]] == fa[~miss[s]]).all()
        assert np.isnan(flagged["innov"][s][:, :-1][np.broadcast_to(miss[s][:, None], (miss[s].shape[0], 2 * m + 1, N))]).all()
        rej = fa == 0.0
        assert np.isfinite(flagged["innov"][s][:, 1:1 + 2 * m].transpose(1, 0, 2)[:, rej]).all()  # y, S(a,a) written when rejected
    assert_state_bits(flagged["state"], unflagged["state"])
    ref = run(sc, nan_rows(holed, {s: flagged["innov"][s][:, -1] == 0.0 for s in (0, 1)}), ev, skip=True, mapping=mapping)
    assert_state_bits(flagged["state"], ref["state"])


@pytest.mark.gpu
@pytest.mark.parametrize("mapping", [1, 4])
def test_rewinds_regate_replayed_rows_and_records_equal_snapshots(mapping):
    """Late pose fixes planned into RESTORE + replay: every replayed row is gated again against its replayed prior, so the
    program ends where the in-order gated program ends; RECORD ops inside gated programs equal snapshots."""
    from pronto_b200.schedule import program_from_arrivals

    N, T = 256, 400
    rng = np.random.default_rng(13)
    sc = scenario(N, T)
    streams, _ = with_outliers(base_streams(sc), rng, frac=0.03, size=1.0)
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
    gates = {0: chi2_thr(3, 0.999), 1: chi2_thr(6, 0.999)}
    got = run(sc, streams, ops, gates=gates, snapshot_slots=4, mapping=mapping)
    ref = run(sc, streams, ev, gates=gates, snapshot_slots=4, mapping=mapping)
    assert (ref["innov"][1][:, 1] == 0.0).any()
    assert_state_bits(got["state"], ref["state"])
    for s in (0, 1):
        assert same_bits(got["innov"][s], ref["innov"][s])
    # records inside a gated program against snapshots at the same positions
    import torch

    prog = []
    for i, o in enumerate(ev[:400]):
        prog.append(o)
        if i % 40 == 39:
            prog += [(capi.OP_RECORD, 0, i // 40, 0, 0.0), (capi.OP_SNAPSHOT, 0, 0, 0, 0.0)]
    with RBISBatch(N, snapshot_slots=1, mapping=mapping) as b:
        b.set_process_noise(*nominal_q())
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        for s, t in gates.items():
            b.set_nis_gate(s, t)
        ro = torch.full((10, capi.REC_FIELDS, N), float("nan"), dtype=torch.float64, device="cuda")
        b.set_record(ro, REC_ALL)
        for k in range(10):
            b.run_fused(prog[k * 42:(k + 1) * 42], imu=sc["st"]["imu"], streams=gpu(streams))
            assert b.last_kernel_variant & GATE_VARIANT
            b.synchronize()
            v, q, _, ll = b.get_snapshot(0)
            r = ro[k].cpu().numpy()
            assert same_bits(r[:21], v) and same_bits(r[21:25], q) and same_bits(r[25], ll)


@pytest.mark.gpu
@pytest.mark.parametrize("materialize", [False, True])
def test_synthesised_inputs(materialize):
    """run_fused_synth with a gate equals synthesize + gated run_fused bit for bit (the gated call materialises its rows)."""
    N, T = 300, 220
    sc = scenario(N, T)
    st = sc["st"]
    ev = st["events"]
    d = synth.synth_spec_inputs(sc["truth"], 0, T)
    gates = {0: chi2_thr(3, 0.99), 1: chi2_thr(6, 0.99)}
    import torch

    outs = [[torch.full((r, 2, N), float("nan"), dtype=torch.float64, device="cuda") for r in (st["legodo"].shape[0], st["pose_z"].shape[0])]
            for _ in range(2)]
    with RBISBatch(N, synth_materialize=materialize) as b:
        b.set_process_noise(*nominal_q())
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        spec = SynthSpec(synth.SEED, d["imu_mean"], d["imu_step"], d["streams"], mode=1)
        for s, t in gates.items():
            b.set_nis_gate(s, t)
            b.set_innovations(s, outs[0][s], (3, 6)[s], APPLIED_SET)
        b.run_fused_synth(ev, [MeasStream(synth.LEGODO_IDX, None, st["R_legodo"]), MeasStream(synth.POSE_IDX, None, st["R_pose"], quat=True)],
                          spec)
        assert not b.last_kernel_variant & 4 and b.last_kernel_variant & GATE_VARIANT
        a = b.get_state()
        gen = b.synthesize(spec)
        b.set_process_noise(*nominal_q())
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        for s in gates:
            b.set_innovations(s, outs[1][s], (3, 6)[s], APPLIED_SET)
        b.run_fused(ev, imu=gen["imu"], streams=[MeasStream(synth.LEGODO_IDX, gen["z"][0], st["R_legodo"]),
                                                  MeasStream(synth.POSE_IDX, gen["z"][1], st["R_pose"], quat=gen["quat"][1])])
        b.synchronize()
        c = b.get_state()
    assert_state_bits(a, c)
    for s in (0, 1):
        x, y = outs[0][s].cpu().numpy(), outs[1][s].cpu().numpy()
        assert not np.isnan(x).any() and same_bits(x, y)


@pytest.mark.gpu
def test_rejected_fraction_of_consistent_filters():
    """4,096 filters whose noise matches R and Q, gated at chi2_m(0.99): the rejected fraction of every row (after the first
    fifth of the run) lies within 5 sigma of 1 % under the binomial."""
    N, T = 4096, 1000
    sc = scenario(N, T)
    got = run(sc, base_streams(sc), sc["st"]["events"], gates={0: chi2_thr(3, 0.99), 1: chi2_thr(6, 0.99)})
    tol = 5 * np.sqrt(0.01 * 0.99 / N)
    for s in (0, 1):
        a = got["innov"][s][:, 1]
        a = a[a.shape[0] // 5:]
        assert set(np.unique(a)) <= {0.0, 1.0}
        frac = (a == 0.0).mean(axis=1)
        assert np.all(np.abs(frac - 0.01) <= tol), (s, float(frac.min()), float(frac.max()), float(frac.mean()))


@pytest.mark.gpu
def test_gate_keeps_nees_consistent_under_pose_outliers():
    """2 % of the pose rows carry a 5 m error: the gated ensemble's average NEES of position stays near 3 (chi2(3)), the ungated
    one does not."""
    N, T = 1024, 600
    rng = np.random.default_rng(17)
    sc = scenario(N, T)
    streams, _ = with_outliers(base_streams(sc), rng, frac=0.02, size=5.0)
    ev = sc["st"]["events"]
    tv, _ = synth.truth_state_at(sc["truth"], T - 1)
    res = {}
    for name, g in (("gated", {0: chi2_thr(3, 0.999), 1: chi2_thr(6, 0.999)}), ("ungated", None)):
        v, q, P, ll, _ = run(sc, streams, ev, gates=g)["state"]
        e = v[9:12] - tv[9:12, None]
        Pp = P.reshape(21, 21, N)[9:12, 9:12]
        res[name] = float(np.mean([e[:, n] @ np.linalg.solve(Pp[:, :, n], e[:, n]) for n in range(N)]))
    assert res["gated"] < 4.5, res
    assert res["ungated"] > 10 * res["gated"], res


def innov_stats_reference(rows, m, fields, chunk):
    """The innovation statistics tree of tests/test_innovations.py plus entry [33], filters with APPLIED == 0."""
    from test_innovations import stats_reference

    out = stats_reference(rows, m, fields & ~capi.INNOV_APPLIED, chunk)
    R, k, N = rows.shape
    nch = (N + chunk - 1) // chunk
    if fields & capi.INNOV_APPLIED:
        for r in range(R):
            v = np.zeros(nch * chunk)
            v[:N] = rows[r, k - 1] == 0.0
            t = v.reshape(nch, chunk)
            w = chunk
            while w > 1:
                w //= 2
                t = t[:, :w] + t[:, w:2 * w]
            out[r, :, 33] = t[:, 0]
    return out


def _pinned(shape):
    import torch

    return torch.full(shape, float("nan"), dtype=torch.float64).pin_memory()


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [32, 1024])
def test_statistics_count_rejections(chunk):
    """Entry [33] counts the rejected filters of each row and every other entry equals the innovation tree; tables of sets
    without APPLIED stay as they were."""
    N, T = 3000, 120
    rng = np.random.default_rng(4)
    sc = scenario(N, T)
    streams, _ = with_outliers(base_streams(sc), rng, frac=0.05, size=1.0, which=(0, 1))
    streams[0]["z"][::3, 1, 100:160] = np.nan
    ev = sc["st"]["events"]
    nch = (N + chunk - 1) // chunk
    for fields in (ALL | capi.INNOV_APPLIED, APPLIED_SET, ALL):
        with RBISBatch(N) as b:
            b.set_process_noise(*nominal_q())
            b.set_state(sc["vec"], sc["quat"], sc["cov"])
            outs = []
            import torch

            for s, m in ((0, 3), (1, 6)):
                b.set_nis_gate(s, chi2_thr(m, 0.999))
                outs.append(torch.full((streams[s]["z"].shape[0], len(innovation_layout(m, fields)), N), float("nan"),
                                       dtype=torch.float64, device="cuda"))
                b.set_innovations(s, outs[s], m, fields)
            b.run_fused(ev, imu=sc["st"]["imu"], streams=gpu(streams, skip=True))
            res = []
            for s in (0, 1):
                R = streams[s]["z"].shape[0]
                ch, tot = _pinned((R, nch, capi.NUM_STATS)), _pinned((R, capi.NUM_STATS))
                b.wait(b.stats_innovations_enqueue(s, 0, ch, tot, chunk=chunk))
                res.append((ch.numpy().copy(), tot.numpy().copy()))
            b.synchronize()
            rows = [o.cpu().numpy() for o in outs]
        for s, m in ((0, 3), (1, 6)):
            ch, tot = res[s]
            assert same_bits(ch, innov_stats_reference(rows[s], m, fields, chunk)), (fields, s)
            for r in range(ch.shape[0]):
                assert same_bits(tot[r], reduce_chunks(ch[r]))
            if fields & capi.INNOV_APPLIED:
                assert ch[..., 33].sum() == (rows[s][:, -1] == 0.0).sum() > 0
            else:
                assert (ch[..., 33] == 0).all()


@pytest.mark.gpu
def test_errors_are_refused_before_anything_is_enqueued():
    import torch

    N, T = 64, 60
    sc = scenario(N, T)
    st = sc["st"]
    streams = gpu(base_streams(sc))
    with RBISBatch(N) as b:
        b.set_process_noise(*nominal_q())
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        before = b.launch_count
        lib = capi.load()
        good = torch.full((N,), 10.0, dtype=torch.float64, device="cuda")

        def gate(nis_max=10.0, per=None):
            g = capi.NisGate()
            g.nis_max, g.nis_max_per_filter = nis_max, per
            return C.byref(g)

        host = np.full(N, 10.0)
        for stream, g in ((-1, gate()), (8, gate()), (0, gate(np.nan)), (0, gate(0.0)), (0, gate(-1.0)), (0, gate(-np.inf)),
                          (0, gate(10.0, host.ctypes.data))):
            assert lib.rbis_batch_set_nis_gate(b.h, stream, g) != 0, stream
        with pytest.raises(capi.RBISError):
            b.set_nis_gate(0, per_filter=torch.full((N,), 10.0, dtype=torch.float64))   # host tensor
        with pytest.raises(ValueError):
            b.set_nis_gate(0, per_filter=torch.full((N + 1,), 10.0, dtype=torch.float64, device="cuda"))
        assert lib.rbis_batch_set_nis_gate(b.h, 0, gate(np.nan, good.data_ptr())) == 0   # nis_max unused with thresholds
        assert lib.rbis_batch_set_nis_gate(b.h, 0, gate(np.inf)) == 0
        assert lib.rbis_batch_set_nis_gate(b.h, 0, None) == 0
        out = torch.zeros((1, 1, N), dtype=torch.float64, device="cuda")
        spec = capi.Innovation()
        spec.fields, spec.m, spec.out, spec.rows = capi.INNOV_APPLIED, 3, out.data_ptr(), 1
        assert lib.rbis_batch_set_innovations(b.h, 0, C.byref(spec)) != 0
        spec.fields = 16 | capi.INNOV_NIS
        assert lib.rbis_batch_set_innovations(b.h, 0, C.byref(spec)) != 0
        assert b.launch_count == before
        # the single-update entry points ignore gates: a gate of 1e-300 rejects everything in a fused call, nothing here
        b.set_nis_gate(0, 1e-300)
        v0 = b.get_state()[0].copy()
        z = np.ascontiguousarray(st["legodo"][0])
        b.indexed_update(synth.LEGODO_IDX, z, st["R_legodo"])
        assert b.last_kernel_variant >= 0 and not b.last_kernel_variant & GATE_VARIANT
        assert not same_bits(b.get_state()[0], v0)
        # a call with fewer streams than the gated slot ignores it
        b.set_nis_gate(1, 1e-300)
        b.clear_nis_gate(0)
        b.run_fused([e for e in st["events"] if e[0] == capi.OP_IMU or e[1] == 0], imu=st["imu"], streams=streams[:1])
        assert not b.last_kernel_variant & GATE_VARIANT
        b.synchronize()
