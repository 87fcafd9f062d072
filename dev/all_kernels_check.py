#!/usr/bin/env python
"""dev/all_kernels_check.py -- one small pass through every fused-kernel family with a bit-identity check (compute-sanitizer is closed on the GPU pool):
lane-per-filter decoupled + dense, warp-group 4 / 8 lanes, SYN instantiations, snapshot / restore, snapshot statistics, the
REC instantiations (RBIS_OP_RECORD), the MASK instantiations (RBIS_STREAM_SKIP_NAN_ROWS, with and without records) and the
innovation sets (rbis_batch_set_innovations, REC instantiations: in-order, rewound, synthesised and masked programs) over the same
mappings and variants."""
import os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import torch
from common import gpu_streams, nominal_q, scenario, random_ensemble
from pronto_b200 import MeasStream, RBISBatch, SynthSpec, capi, synth

N, T = 37, 24
sc = scenario(N, T, tumbling=True)
st = sc["st"]
ev = list(st["events"])
half = len(ev) // 2
prog = ev[:half] + [(capi.OP_SNAPSHOT, 0, 0, ev[half - 1][3], 0.0)] + ev[half:] + [(capi.OP_RESTORE, 0, 0, ev[half - 1][3], 0.0)] + ev[half:]
tv, tq = synth.truth_state_at(sc["truth"], T - 1)
ref = None
for cfg in (dict(mapping=1, lane_filters_per_cta=384), dict(mapping=1, lane_filters_per_cta=128), dict(mapping=1, dense_only=True),
            dict(mapping=4), dict(mapping=8), dict(mapping=4, dense_only=True)):
    with RBISBatch(N, snapshot_slots=2, **cfg) as b:
        b.set_process_noise(*nominal_q())
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        b.run_fused(prog, imu=st["imu"], streams=gpu_streams(st))
        out = torch.empty((1, capi.NUM_STATS), dtype=torch.float64, pin_memory=True).numpy()
        b.run_fused([(capi.OP_SNAPSHOT, 0, 1, ev[-1][3], 0.0)], imu=st["imu"], streams=gpu_streams(st))
        b.wait(b.stats_snapshot_enqueue(1, tv, tq, out, chunk=64))
        got = b.get_state()
    if ref is None:
        ref = got
    same = all(np.array_equal(x, y) for x, y in zip(got[:4], ref[:4]))
    print(cfg, "variant", "same bits" if same else "DIFFERENT", flush=True)
    assert same
d = synth.synth_spec_inputs(sc["truth"], 0, T)
for cfg in (dict(mapping=1), dict(mapping=4), dict(mapping=8), dict(mapping=1, synth_materialize=True)):
    with RBISBatch(N, **cfg) as b:
        b.set_process_noise(*nominal_q())
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        b.run_fused_synth(ev, [MeasStream(synth.LEGODO_IDX, None, st["R_legodo"]), MeasStream(synth.POSE_IDX, None, st["R_pose"], quat=True)],
                          SynthSpec(synth.SEED, d["imu_mean"], d["imu_step"], d["streams"], mode=1))
        got = b.get_state()
    if cfg == dict(mapping=1):
        ref = got
    same = all(np.array_equal(x, y) for x, y in zip(got[:4], ref[:4]))
    print("synth", cfg, "same bits" if same else "DIFFERENT", flush=True)
    assert same
# records: a RECORD of every field after every op of the same programs, through the REC instantiations
rec_prog, rows = [], 0
for o in prog:
    rec_prog += [o, (capi.OP_RECORD, 0, rows, 0, 0.0)]
    rows += 1
ALL = (1 << capi.REC_FIELDS) - 1
ref_rec = ref_state = None
for cfg in (dict(mapping=1, lane_filters_per_cta=384), dict(mapping=1, lane_filters_per_cta=128), dict(mapping=1, dense_only=True),
            dict(mapping=4), dict(mapping=8), dict(mapping=4, dense_only=True)):
    out = torch.full((rows, capi.REC_FIELDS, N), float("nan"), dtype=torch.float64, device="cuda")
    with RBISBatch(N, snapshot_slots=2, **cfg) as b:
        b.set_process_noise(*nominal_q())
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        b.set_record(out, ALL)
        b.run_fused(rec_prog, imu=st["imu"], streams=gpu_streams(st))
        variant = b.last_kernel_variant
        got = b.get_state()
    rec = out.cpu().numpy()
    if ref_rec is None:
        ref_rec, ref_state = rec, got
    same = np.array_equal(rec, ref_rec) and all(np.array_equal(x, y) for x, y in zip(got[:4], ref_state[:4])) and not np.isnan(rec).any()
    print("record", cfg, "variant", variant, "same bits" if same else "DIFFERENT", flush=True)
    assert same and variant & 8
syn_rec = [x for i, o in enumerate(ev) for x in (o, (capi.OP_RECORD, 0, i, 0, 0.0))]
ref_rec = None
for cfg in (dict(mapping=1), dict(mapping=4), dict(mapping=8), dict(mapping=1, synth_materialize=True)):
    out = torch.full((rows, capi.REC_FIELDS, N), float("nan"), dtype=torch.float64, device="cuda")
    with RBISBatch(N, **cfg) as b:
        b.set_process_noise(*nominal_q())
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        b.set_record(out, ALL)
        b.run_fused_synth(syn_rec, [MeasStream(synth.LEGODO_IDX, None, st["R_legodo"]), MeasStream(synth.POSE_IDX, None, st["R_pose"], quat=True)],
                          SynthSpec(synth.SEED, d["imu_mean"], d["imu_step"], d["streams"], mode=1))
        variant = b.last_kernel_variant
        b.synchronize()
    rec = out.cpu().numpy()[:len(ev)]
    if ref_rec is None:
        ref_rec = rec
    same = np.array_equal(rec, ref_rec) and not np.isnan(rec).any()
    print("record synth", cfg, "variant", variant, "same bits" if same else "DIFFERENT", flush=True)
    assert same and variant & 8
# missing rows: per-filter NaN dropouts on both streams through the MASK (and MASK + REC) instantiations; a flagged program
# without NaN gives the unflagged bits
rng = np.random.default_rng(3)
lego, pose_z = st["legodo"].copy(), st["pose_z"].copy()
lego[rng.random(lego.shape) < 0.1] = np.nan
pose_z[:, 0][rng.random(pose_z[:, 0].shape) < 0.2] = np.nan


def masked(z_lego, z_pose):
    return [MeasStream(synth.LEGODO_IDX, z_lego, st["R_legodo"], skip_nan_rows=True),
            MeasStream(synth.POSE_IDX, z_pose, st["R_pose"], quat=st["pose_q"], skip_nan_rows=True)]


ref_mask = None
for cfg in (dict(mapping=1, lane_filters_per_cta=384), dict(mapping=1, lane_filters_per_cta=128), dict(mapping=1, dense_only=True),
            dict(mapping=4), dict(mapping=8), dict(mapping=4, dense_only=True)):
    for with_rec in (False, True):
        out = torch.full((rows, capi.REC_FIELDS, N), float("nan"), dtype=torch.float64, device="cuda")
        with RBISBatch(N, snapshot_slots=2, **cfg) as b:
            b.set_process_noise(*nominal_q())
            b.set_state(sc["vec"], sc["quat"], sc["cov"])
            b.run_fused(prog, imu=st["imu"], streams=masked(st["legodo"], st["pose_z"]))
            clean = b.get_state()
            b.set_state(sc["vec"], sc["quat"], sc["cov"])
            if with_rec:
                b.set_record(out, ALL)
            b.run_fused(rec_prog if with_rec else prog, imu=st["imu"], streams=masked(lego, pose_z))
            variant = b.last_kernel_variant
            got = b.get_state()
        if ref_mask is None:
            ref_mask = got
        same = all(np.array_equal(x, y) for x, y in zip(got[:4], ref_mask[:4])) and all(np.array_equal(x, y) for x, y in zip(clean[:4], ref_state[:4]))
        same = same and not np.isnan(got[0]).any()
        print("masked", cfg, "records" if with_rec else "", "variant", variant, "same bits" if same else "DIFFERENT", flush=True)
        assert same and variant & 512
# innovation sets: NIS, y and S(a,a) of every MEAS op of both streams; the rows of the rewound program equal those of the same
# program's replay, the state equals the program without innovation sets
INNOV = capi.INNOV_NIS | capi.INNOV_Y | capi.INNOV_S_DIAG


def innov_bufs():
    return [torch.full((st["legodo"].shape[0], 7, N), float("nan"), dtype=torch.float64, device="cuda"),
            torch.full((st["pose_z"].shape[0], 13, N), float("nan"), dtype=torch.float64, device="cuda")]


ref_innov = {}
for cfg in (dict(mapping=1, lane_filters_per_cta=384), dict(mapping=1, lane_filters_per_cta=128), dict(mapping=1, dense_only=True),
            dict(mapping=4), dict(mapping=8), dict(mapping=4, dense_only=True)):
    for key, streams, want_state in (("plain", gpu_streams(st), ref_state), ("masked", masked(lego, pose_z), ref_mask)):
        bufs = innov_bufs()
        with RBISBatch(N, snapshot_slots=2, **cfg) as b:
            b.set_process_noise(*nominal_q())
            b.set_state(sc["vec"], sc["quat"], sc["cov"])
            for s_, m_ in ((0, 3), (1, 6)):
                b.set_innovations(s_, bufs[s_], m_, INNOV)
            b.run_fused(prog, imu=st["imu"], streams=streams)
            variant = b.last_kernel_variant
            got = b.get_state()
        rows_ = [x.cpu().numpy() for x in bufs]
        ref_innov.setdefault(key, rows_)
        same = all(np.array_equal(x, y, equal_nan=True) for x, y in zip(rows_, ref_innov[key]))
        same = same and all(np.array_equal(x, y) for x, y in zip(got[:4], want_state[:4]))
        same = same and (key == "masked" or not any(np.isnan(x).any() for x in rows_))
        print("innovations", key, cfg, "variant", variant, "same bits" if same else "DIFFERENT", flush=True)
        assert same and variant & 8
ref_innov = None
for cfg in (dict(mapping=1), dict(mapping=4), dict(mapping=8), dict(mapping=1, synth_materialize=True)):
    bufs = innov_bufs()
    with RBISBatch(N, **cfg) as b:
        b.set_process_noise(*nominal_q())
        b.set_state(sc["vec"], sc["quat"], sc["cov"])
        for s_, m_ in ((0, 3), (1, 6)):
            b.set_innovations(s_, bufs[s_], m_, INNOV)
        b.run_fused_synth(ev, [MeasStream(synth.LEGODO_IDX, None, st["R_legodo"]), MeasStream(synth.POSE_IDX, None, st["R_pose"], quat=True)],
                          SynthSpec(synth.SEED, d["imu_mean"], d["imu_step"], d["streams"], mode=1))
        variant = b.last_kernel_variant
        b.synchronize()
    rows_ = [x.cpu().numpy() for x in bufs]
    if ref_innov is None:
        ref_innov = rows_
    same = all(np.array_equal(x, y) for x, y in zip(rows_, ref_innov)) and not any(np.isnan(x).any() for x in rows_)
    print("innovations synth", cfg, "variant", variant, "same bits" if same else "DIFFERENT", flush=True)
    assert same and variant & 8
print("ok")
