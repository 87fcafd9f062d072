#!/usr/bin/env python
"""dev/dropout_bench.py -- cost of rows missing per filter (RBIS_STREAM_SKIP_NAN_ROWS) in the fused launches.

BASELINE shape (65,536 filters, 1 kHz IMU, 500 Hz leg odometry, 10 Hz pose fixes, 200-step fused launches, inputs resident
in HBM as bench.py keeps them).  The same programs over the same rows, four cases:
  clear    -- no flag: the program bench.py times;
  flag0    -- both streams flagged, no NaN anywhere: the price of the MASK instantiations alone;
  drop10   -- flagged, 10 % of the leg-odometry rows missing, drawn per filter and row;
  drop50   -- flagged, 50 % missing.
All run in one process, alternating, --reps times each.  A run is --launches calls from a synchronise to a wait on a ticket
recorded after the last call, timed with the host clock.  Prints one JSON line: filter-steps/s of every run, the median per case
and its ratio to `clear`, the kernel variants, and the card and its power limit read in the same run."""
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
    ap.add_argument("--chunks", type=int, default=8, help="resident input chunks per case (each ~0.8 GB at the default size)")
    ap.add_argument("--launches", type=int, default=48, help="fused launches per timed run (cycling through the chunks)")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()

    import torch

    import bench
    from row_noise_bench import card
    from pronto_b200 import MeasStream, RBISBatch, synth

    if not torch.cuda.is_available():
        raise SystemExit("dropout_bench.py: no CUDA device")
    dev = torch.device("cuda", 0)
    p = synth.NOMINAL
    N, Tc = args.filters, args.chunk_steps
    R_lego = np.eye(3) * p["r_vxyz"] ** 2
    R_pose = np.diag([p["r_xyz"] ** 2] * 3 + [p["r_chi"] ** 2] * 3)
    wl = bench.Workload(N, Tc, args.chunks, dev, 0x5EED, R_lego, R_pose)
    gen = torch.Generator(device=dev)
    gen.manual_seed(0xD0)

    def streams(c, frac, flag):
        z = wl.chunks[c]["legodo"]
        if frac > 0:   # one NaN in a random column of each missing (row, filter)
            z = z.clone()
            rows = z.shape[0]
            miss = torch.rand((rows, N), generator=gen, device=dev) < frac
            col = torch.randint(0, 3, (rows, N), generator=gen, device=dev)
            for a in range(3):
                z[:, a][miss & (col == a)] = float("nan")
        return [MeasStream(synth.LEGODO_IDX, z, R_lego, skip_nan_rows=flag),
                MeasStream(synth.POSE_IDX, wl.chunks[c]["pose_z"], R_pose, quat=wl.chunks[c]["pose_q"], skip_nan_rows=flag)]

    cases = {"clear": (0.0, False), "flag0": (0.0, True), "drop10": (0.1, True), "drop50": (0.5, True)}
    q4 = (p["q_gyro"], p["q_accel"], p["q_gyro_bias"], p["q_accel_bias"])
    name, power_limit, sm_max = card()
    res = {k: [] for k in cases}
    variants = {}
    with RBISBatch(N) as b:
        b.set_process_noise(*q4)
        preps = {k: [b.prepare_fused(wl.progs[c], imu=wl.chunks[c]["imu"], streams=streams(c, frac, flag)) for c in range(args.chunks)]
                 for k, (frac, flag) in cases.items()}
        torch.cuda.synchronize()

        def run(k):
            for i in range(args.launches):
                b.run_prepared(preps[k][i % args.chunks])
            b.wait(b.record())

        finals = {}
        for k in cases:   # warm-up of every program; flag0 must give the bits of clear
            b.set_state(wl.vec0, wl.quat0, wl.cov0)
            run(k)
            variants[k] = b.last_kernel_variant
            finals[k] = b.get_state()
        same = all(np.array_equal(x, y) for x, y in zip(finals["flag0"][:4], finals["clear"][:4]))
        for rep in range(args.reps):
            order = list(cases) if rep % 2 == 0 else list(cases)[::-1]
            for k in order:
                b.set_state(wl.vec0, wl.quat0, wl.cov0)
                b.synchronize()
                t0 = time.perf_counter()
                run(k)
                res[k].append(N * Tc * args.launches / (time.perf_counter() - t0))
    med = {k: float(np.median(v)) for k, v in res.items()}
    out = dict(metric="dropout_filter_steps_per_s", filters=N, chunk_steps=Tc, launches_per_run=args.launches, reps=args.reps,
               card=name, power_limit_w=power_limit, sm_max_mhz=sm_max,
               filter_steps_per_s={k: [round(x) for x in v] for k, v in res.items()},
               median={k: round(v) for k, v in med.items()},
               spread_rel={k: (max(v) - min(v)) / float(np.median(v)) for k, v in res.items()},
               ratio_vs_clear={k: med[k] / med["clear"] for k in cases}, kernel_variant=variants, flag0_same_bits=same,
               time=time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime()))
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
