#!/usr/bin/env python
"""dev/gate_bench.py -- cost of the NIS gates (rbis_batch_set_nis_gate) inside the fused launches.

BASELINE shape (65,536 filters, 1 kHz IMU, 500 Hz leg odometry, 10 Hz pose fixes, 200-step fused launches, inputs resident
in HBM as bench.py keeps them).  The same programs under five settings:
  none         -- no gate: the program bench.py times;
  flag0        -- RBIS_STREAM_SKIP_NAN_ROWS on both streams and no NaN anywhere: the MASK kernels' cost;
  gate         -- NIS gates on both streams at chi2_m(0.999), clean rows (GATE kernels);
  gate_out     -- as `gate`, with 2 % of the pose rows (per filter) moved by 5 m;
  gate_innov   -- as `gate`, plus NIS + APPLIED innovation sets on both streams.
All run in one process, alternating, --reps times each.  A run is --launches calls from a synchronise to a wait on a ticket
recorded after the last call, timed with the host clock.  Prints one JSON line: filter-steps/s of every run, the median per
case, its run-to-run spread and its ratio to `none`, the rejected fractions of the first call, and the card and its power
limit read in the same run."""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--filters", type=int, default=65_536)
    ap.add_argument("--chunk-steps", type=int, default=200)
    ap.add_argument("--chunks", type=int, default=24, help="resident input chunks (each ~0.8 GB at the default size)")
    ap.add_argument("--launches", type=int, default=48, help="fused launches per timed run (cycling through the chunks)")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()

    import torch
    from scipy.stats import chi2

    import bench
    from row_noise_bench import card
    from pronto_b200 import MeasStream, RBISBatch, capi, innovation_layout, synth

    if not torch.cuda.is_available():
        raise SystemExit("gate_bench.py: no CUDA device")
    dev = torch.device("cuda", 0)
    p = synth.NOMINAL
    N, Tc = args.filters, args.chunk_steps
    R_lego = np.eye(3) * p["r_vxyz"] ** 2
    R_pose = np.diag([p["r_xyz"] ** 2] * 3 + [p["r_chi"] ** 2] * 3)
    wl = bench.Workload(N, Tc, args.chunks, dev, 0x5EED, R_lego, R_pose)
    gen = torch.Generator(device=dev)
    gen.manual_seed(0x6A7E)
    ms = (3, 6)
    thr = [float(chi2.ppf(0.999, m)) for m in ms]

    def streams(c, flag, outliers):
        pz = wl.chunks[c]["pose_z"]
        if outliers:   # 5 m on the position rows of 2 % of the (row, filter) pairs
            pz = pz.clone()
            hit = torch.rand((pz.shape[0], N), generator=gen, device=dev) < 0.02
            for a in range(3):
                pz[:, a] += 5.0 * hit
        return [MeasStream(synth.LEGODO_IDX, wl.chunks[c]["legodo"], R_lego, skip_nan_rows=flag),
                MeasStream(synth.POSE_IDX, pz, R_pose, quat=wl.chunks[c]["pose_q"], skip_nan_rows=flag)]

    cases = {"none": (False, False, False, False), "flag0": (True, False, False, False), "gate": (False, True, False, False),
             "gate_out": (False, True, True, False), "gate_innov": (False, True, False, True)}
    rows = [int(max(o["row"] for o in wl.progs[0] if o["kind"] == capi.OP_MEAS and o["stream"] == s)) + 1 for s in (0, 1)]
    fields = capi.INNOV_NIS | capi.INNOV_APPLIED
    bufs = [torch.empty((rows[s], len(innovation_layout(ms[s], fields)), N), dtype=torch.float64, device=dev) for s in (0, 1)]
    q4 = (p["q_gyro"], p["q_accel"], p["q_gyro_bias"], p["q_accel_bias"])
    name, power_limit, sm_max = card()
    res = {k: [] for k in cases}
    variants, rejected = {}, {}
    with RBISBatch(N) as b:
        b.set_process_noise(*q4)
        preps = {k: [b.prepare_fused(wl.progs[c], imu=wl.chunks[c]["imu"], streams=streams(c, flag, out)) for c in range(args.chunks)]
                 for k, (flag, _, out, _) in cases.items()}
        torch.cuda.synchronize()

        def run(k, launches=args.launches):
            _, gated, _, innov = cases[k]
            for s in (0, 1):
                if gated:
                    b.set_nis_gate(s, thr[s])
                if innov:
                    b.set_innovations(s, bufs[s], ms[s], fields)
            for i in range(launches):
                b.run_prepared(preps[k][i % args.chunks])
            b.wait(b.record())
            for s in (0, 1):
                b.clear_nis_gate(s)
                b.clear_innovations(s)

        for k in cases:   # warm-up of every program
            b.set_state(wl.vec0, wl.quat0, wl.cov0)
            run(k)
            variants[k] = b.last_kernel_variant
        for k in ("gate", "gate_out"):   # rejected fractions of one call, read through an innovation set
            b.set_state(wl.vec0, wl.quat0, wl.cov0)
            for s in (0, 1):
                b.set_innovations(s, bufs[s], ms[s], fields)
                b.set_nis_gate(s, thr[s])
            b.run_prepared(preps[k][0])
            b.synchronize()
            rejected[k] = [float((bufs[s][:, 1] == 0.0).double().mean()) for s in (0, 1)]
            for s in (0, 1):
                b.clear_nis_gate(s)
                b.clear_innovations(s)
        for rep in range(args.reps):
            order = list(cases) if rep % 2 == 0 else list(cases)[::-1]
            for k in order:
                b.set_state(wl.vec0, wl.quat0, wl.cov0)
                b.synchronize()
                t0 = time.perf_counter()
                run(k)
                res[k].append(N * Tc * args.launches / (time.perf_counter() - t0))
    med = {k: float(np.median(v)) for k, v in res.items()}
    out = dict(metric="gate_filter_steps_per_s", filters=N, chunk_steps=Tc, launches_per_run=args.launches, reps=args.reps,
               card=name, power_limit_w=power_limit, sm_max_mhz=sm_max, thresholds=thr,
               filter_steps_per_s={k: [round(x) for x in v] for k, v in res.items()},
               median={k: round(v) for k, v in med.items()},
               spread_rel={k: (max(v) - min(v)) / float(np.median(v)) for k, v in res.items()},
               ratio_vs_none={k: med[k] / med["none"] for k in cases}, kernel_variant=variants, rejected_fraction=rejected,
               time=time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime()))
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
