"""EKF smoother ("next" row 1 of SURVEY.md 8f): ekfSmoothingStep (MSE/rbis.cpp:234-266) and
MavStateEstimator::EKFSmoothBackwardsPass (MSE/mav_state_est.cpp:98-189).

CPU: the oracle's restatement against the reference's own compiled sources (oracle/_ref, where available) and against
an independent numpy statement of the recursion; the host-side traversal planner (rbis_smooth_plan) against the
oracle's traversal.  GPU: rbis_batch_smooth_backward against the oracle on the same forward pass.
"""
import os

import numpy as np
import pytest

from pronto_b200 import RBISBatch, capi, smoother, synth

from common import gpu_streams, nominal_q, oracle_streams, random_ensemble, scenario

NTHREADS = min(16, os.cpu_count() or 1)


def _events(T, trailing_measurement):
    sc = scenario(3, T, tumbling=True)
    ev = list(sc["st"]["events"])
    if trailing_measurement:  # end the history on a leg-odometry update (step T-1 is odd: append step T's pair)
        while ev[-1][0] == capi.OP_IMU:
            ev.pop()
    return sc, ev


def _np_smoothing_step(o, npred, nxt, cur, dt):
    """rbis.cpp:234-266 written with numpy (Ac from the oracle's linearisation)."""
    Ad = np.eye(21) + o.linearization(cur[0], cur[1]) * dt
    S = npred[2].copy()
    for b0 in (15, 18):
        if (np.diag(npred[2])[b0:b0 + 3] < 1e-11).any():
            S[b0:b0 + 3, b0:b0 + 3] = np.eye(3)
    L = np.linalg.solve(S, Ad @ cur[2]).T
    cov = cur[2] + L @ (nxt[2] - npred[2]) @ L.T
    resid = nxt[0] - npred[0]
    resid[6:9] = o.state_error(nxt[0], nxt[1], npred[0], npred[1])[6:9]
    return L @ resid, cov


def test_smoothing_step_oracle_vs_numpy_and_reference(oracle):
    vec, quat, cov = random_ensemble(4, seed=21)
    P = lambda n, s=1.0: cov[:, n].reshape(21, 21).T * s
    npred = (vec[:, 0], quat[:, 0], P(0))
    nxt = (vec[:, 0] + 0.01 * vec[:, 1], quat[:, 1], P(0, 0.8))
    cur = (vec[:, 2], quat[:, 2], P(2))
    sv, sq, sP = oracle.ekf_smoothing_step(npred, nxt, cur, 1e-3)
    innov, ncov = _np_smoothing_step(oracle, npred, nxt, cur, 1e-3)
    assert np.max(np.abs(sP - ncov)) < 1e-12 * np.max(np.abs(ncov))
    keep = [k for k in range(21) if k not in (6, 7, 8)]
    assert np.max(np.abs((sv - cur[0])[keep] - innov[keep])) < 1e-12
    # zero-uncertainty biases: the identity replacement of rbis.cpp:243-250
    npred0 = (npred[0], npred[1], npred[2].copy())
    npred0[2][15:18, :] = 0; npred0[2][:, 15:18] = 0
    sv0, sq0, sP0 = oracle.ekf_smoothing_step(npred0, nxt, cur, 1e-3)
    _, ncov0 = _np_smoothing_step(oracle, npred0, nxt, cur, 1e-3)
    assert np.max(np.abs(sP0 - ncov0)) < 1e-11 * np.max(np.abs(ncov0))
    if oracle.build_ref() is None:
        pytest.skip("oracle/_ref not available")
    with oracle.reference():
        oracle.set_constants()
        rv, rq, rP = oracle.ekf_smoothing_step(npred, nxt, cur, 1e-3)
        rv0, rq0, rP0 = oracle.ekf_smoothing_step(npred0, nxt, cur, 1e-3)
    for a, b in ((sv, rv), (sq, rq), (sP, rP), (sv0, rv0), (sP0, rP0)):
        assert np.max(np.abs(a - b)) < 1e-12


@pytest.mark.parametrize("trailing", [False, True])
def test_backwards_pass_oracle_equals_reference(oracle, ref_next, trailing):
    """Live against oracle/_ref where it is built; otherwise against what it computed on these very inputs
    (tests/golden/make_reference_golden_next.py:smoothing_events builds the same 3-filter, 61-step history)."""
    sc, ev = _events(61, trailing)
    st = sc["st"]
    a = oracle.smooth_ensemble(sc["vec"], sc["quat"], sc["cov"], 0, nominal_q(), st["imu"], oracle_streams(st), ev, 1e-3)
    if oracle.build_ref() is None:
        name = "trailing" if trailing else "plain"
        b = {f"post_{k}": ref_next[f"smooth_{name}_{k}"] for k in ("vec", "quat", "cov")}
    else:
        with oracle.reference():
            oracle.set_constants()
            b = oracle.smooth_ensemble(sc["vec"], sc["quat"], sc["cov"], 0, nominal_q(), st["imu"], oracle_streams(st), ev, 1e-3)
    for k in ("post_vec", "post_quat", "post_cov"):
        assert np.max(np.abs(a[k] - b[k])) < 1e-12, k
    filt = oracle.run_ensemble(sc["vec"], sc["quat"], sc["cov"], None, 0, nominal_q(), st["imu"], oracle_streams(st), ev, trace=True)
    assert np.max(np.abs(a["post_vec"] - filt["trace_vec"])) > 1e-3  # the pass did smooth something


def _replay_plan(oracle, filt, init, ev, dt, n):
    """Run the planned steps with the oracle's single smoothing step on filter n -> per-update posterior."""
    _, is_ins, slot = smoother.forward_program(ev)
    np_slot, n_slot, steps, alias = smoother.plan(is_ins, slot)
    post = {0: init}
    for u in range(1, len(is_ins)):
        post[u] = (filt["trace_vec"][u - 1][:, n], filt["trace_quat"][u - 1][:, n], filt["trace_cov"][u - 1][:, n].reshape(21, 21).T)
    nxt_pred, nxt = post[np_slot], post[n_slot]
    for s in steps:
        cur, cur_pred = post[int(s["cur_slot"])], post[int(s["cur_pred_slot"])]
        sm = oracle.ekf_smoothing_step(nxt_pred, nxt, cur, dt)
        post[int(s["out_slot"])] = sm
        nxt, nxt_pred = sm, cur_pred
    return post, alias


@pytest.mark.parametrize("trailing", [False, True])
def test_plan_reproduces_the_reference_traversal(oracle, rbis_lib, trailing):
    sc, ev = _events(41, trailing)
    st = sc["st"]
    sm = oracle.smooth_ensemble(sc["vec"], sc["quat"], sc["cov"], 0, nominal_q(), st["imu"], oracle_streams(st), ev, 1e-3)
    filt = oracle.run_ensemble(sc["vec"], sc["quat"], sc["cov"], None, 0, nominal_q(), st["imu"], oracle_streams(st), ev, trace=True)
    n = 1
    init = (sc["vec"][:, n], sc["quat"][:, n], sc["cov"][:, n].reshape(21, 21).T)
    post, alias = _replay_plan(oracle, filt, init, ev, 1e-3, n)
    for u in range(1, len(ev) + 1):
        pv, pq, pP = post[int(alias[u])]
        assert np.max(np.abs(pv - sm["post_vec"][u - 1][:, n])) < 1e-13, u
        assert np.max(np.abs(pP.T.reshape(-1) - sm["post_cov"][u - 1][:, n])) < 1e-15, u


def test_plan_rejects_a_history_without_imu_steps(rbis_lib):
    with pytest.raises(capi.RBISError):
        smoother.plan(np.zeros(4, dtype=np.uint8), np.arange(4, dtype=np.int32))


@pytest.fixture(scope="module")
def ref_next():
    return np.load(os.path.join(os.path.dirname(__file__), "golden", "rbis_reference_golden_next.npz"))


def _golden_case(trailing):
    sys_path = os.path.join(os.path.dirname(__file__), "golden")
    import importlib.util

    spec = importlib.util.spec_from_file_location("make_reference_golden_next", os.path.join(sys_path, "make_reference_golden_next.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.smoothing_events(trailing)


@pytest.mark.parametrize("name,trailing", [("plain", False), ("trailing", True)])
def test_oracle_backwards_pass_matches_reference_golden(oracle, ref_next, name, trailing):
    """Fixture made by the reference's own compiled sources (tests/golden/make_reference_golden_next.py)."""
    sc, ev = _golden_case(trailing)
    st = sc["st"]
    a = oracle.smooth_ensemble(sc["vec"], sc["quat"], sc["cov"], 0, nominal_q(), st["imu"], oracle_streams(st), ev, 1e-3)
    for k in ("vec", "quat", "cov"):
        assert np.max(np.abs(a[f"post_{k}"] - ref_next[f"smooth_{name}_{k}"])) < 1e-12, k


@pytest.mark.gpu
@pytest.mark.parametrize("name,trailing", [("plain", False), ("trailing", True)])
def test_gpu_backward_pass_matches_reference_golden(ref_next, name, trailing):
    sc, ev = _golden_case(trailing)
    st = sc["st"]
    N = sc["vec"].shape[1]
    ops, is_ins, slot = smoother.forward_program(ev)
    with RBISBatch(N, snapshot_slots=len(is_ins)) as b:
        b.set_process_noise(*nominal_q())
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        b.run_fused(ops, imu=st["imu"], streams=gpu_streams(st))
        alias = smoother.smooth(b, is_ins, slot, 1e-3)
        for u in range(1, len(is_ins)):
            gv, gq, gP, _ = b.get_snapshot(int(alias[u]))
            rv, rq, rP = (ref_next[f"smooth_{name}_{k}"][u - 1] for k in ("vec", "quat", "cov"))
            assert np.max(np.abs(gv - rv) / np.maximum(1.0, np.abs(rv))) < 1e-9, u
            assert np.max(np.abs(gq - rq)) < 1e-9, u
            d = np.sqrt(np.abs(rP.reshape(21, 21, N)[np.arange(21), np.arange(21)]))
            scale = np.maximum(d[:, None, :] * d[None, :, :], 1e-30).reshape(441, N)
            assert np.max(np.abs(gP - rP) / scale) < 1e-7, u


@pytest.mark.gpu
@pytest.mark.parametrize("trailing,N", [(False, 37), (True, 130)])
def test_gpu_backward_pass_matches_oracle(oracle, trailing, N):
    T = 121
    sc = scenario(N, T, tumbling=True)
    st = sc["st"]
    ev = list(st["events"])
    if trailing:
        while ev[-1][0] == capi.OP_IMU:
            ev.pop()
    ref = oracle.smooth_ensemble(sc["vec"], sc["quat"], sc["cov"], 0, nominal_q(), st["imu"], oracle_streams(st), ev, 1e-3,
                                 n_threads=NTHREADS)
    ops, is_ins, slot = smoother.forward_program(ev)
    with RBISBatch(N, snapshot_slots=len(is_ins)) as b:
        b.set_process_noise(*nominal_q())
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        b.run_fused(ops, imu=st["imu"], streams=gpu_streams(st))
        alias = smoother.smooth(b, is_ins, slot, 1e-3)
        worst = dict(vec=0.0, quat=0.0, cov=0.0)
        for u in sorted(set(range(1, len(is_ins), 7)) | {1, len(is_ins) - 1}):
            gv, gq, gP, _ = b.get_snapshot(int(alias[u]))
            rv, rq, rP = ref["post_vec"][u - 1], ref["post_quat"][u - 1], ref["post_cov"][u - 1]
            worst["vec"] = max(worst["vec"], float(np.max(np.abs(gv - rv) / np.maximum(1.0, np.abs(rv)))))
            worst["quat"] = max(worst["quat"], float(np.max(np.abs(gq - rq))))
            d = np.sqrt(np.abs(rP.reshape(21, 21, N)[np.arange(21), np.arange(21)]))
            scale = np.maximum(d[:, None, :] * d[None, :, :], 1e-30).reshape(441, N)
            worst["cov"] = max(worst["cov"], float(np.max(np.abs(gP - rP) / scale)))
    assert worst["vec"] < 1e-9 and worst["quat"] < 1e-9 and worst["cov"] < 1e-7, worst


@pytest.mark.gpu
def test_gpu_backward_pass_is_reproducible():
    """Warp-level shared-memory hand-offs in rbis_smooth_kernel: two runs from the same forward pass give the same bits
    (compute-sanitizer's racecheck is not available on the GPU pool)."""
    N, T = 300, 80
    sc = scenario(N, T)
    st = sc["st"]
    ev = list(st["events"])
    ops, is_ins, slot = smoother.forward_program(ev)
    outs = []
    with RBISBatch(N, snapshot_slots=len(is_ins)) as b:
        b.set_process_noise(*nominal_q())
        for rep in range(3):
            b.set_state(sc["vec"], sc["quat"], sc["cov"])
            b.run_fused(ops, imu=st["imu"], streams=gpu_streams(st))
            alias = smoother.smooth(b, is_ins, slot, 1e-3)
            outs.append(b.get_snapshot(int(alias[1])))
    for o in outs[1:]:
        for x, y in zip(o, outs[0]):
            assert np.array_equal(x, y)


@pytest.mark.gpu
def test_gpu_smoother_errors():
    with RBISBatch(8, snapshot_slots=3) as b:
        steps = np.zeros(1, dtype=smoother.STEP_DTYPE)
        with pytest.raises(capi.RBISError):
            b.smooth_backward(0, 1, steps, 1e-3)  # empty slots
        with pytest.raises(capi.RBISError):
            b.get_snapshot(5)
