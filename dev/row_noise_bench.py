#!/usr/bin/env python
"""dev/row_noise_bench.py -- cost of a measurement covariance that changes from row to row (RBIS_R_PER_ROW_FULL).

BASELINE shape (65,536 filters, 1 kHz IMU, 500 Hz leg odometry, 10 Hz pose fixes, 200-step fused launches, inputs resident
in HBM as bench.py keeps them), two programs that differ only in the leg-odometry R:
  shared   -- one R for every row (RBIS_R_SHARED_FULL), the program bench.py times;
  per_row  -- R switching between LegOdoCommon's certain and uncertain value on a seeded pattern (10 % uncertain), one
              RBIS_R_PER_ROW_FULL stream.
Both run in one process, alternating, --reps times each.  Prints one JSON line: filter-steps/s of every run and the
median, host enqueue time per call (mean of the first six calls after a synchronise, as bench.py measures it), the
per-row table bytes uploaded per call, the card and its power limit read in the same run.  Also checks that a per-row
stream whose rows all equal the shared R gives the shared program's bits."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    import torch

    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        return name, float(out[0]), float(out[1])
    except Exception:
        return name, None, None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--filters", type=int, default=65_536)
    ap.add_argument("--chunk-steps", type=int, default=200)
    ap.add_argument("--chunks", type=int, default=24, help="resident input chunks (each ~0.8 GB at the default size)")
    ap.add_argument("--launches", type=int, default=48, help="fused launches per timed run (cycling through the chunks)")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--uncertain", type=float, default=0.1, help="share of leg-odometry rows with the uncertain R")
    args = ap.parse_args()

    import torch

    import bench
    from pronto_b200 import MeasStream, RBISBatch, synth

    if not torch.cuda.is_available():
        raise SystemExit("row_noise_bench.py: no CUDA device")
    dev = torch.device("cuda", 0)
    p = synth.NOMINAL
    N, Tc = args.filters, args.chunk_steps
    R_lego = np.eye(3) * p["r_vxyz"] ** 2
    R_unc = np.eye(3) * (5 * p["r_vxyz"]) ** 2   # LegOdoCommon's r_vxyz_uncertain, here 5 x r_vxyz
    R_pose = np.diag([p["r_xyz"] ** 2] * 3 + [p["r_chi"] ** 2] * 3)
    wl = bench.Workload(N, Tc, args.chunks, dev, 0x5EED, R_lego, R_pose)
    rng = np.random.default_rng(0x0D0)
    programs = {"shared": wl.streams, "per_row": [], "per_row_equal": []}
    table_bytes = []
    for c in range(args.chunks):
        lego, pose = wl.streams[c]
        rows = lego.z.shape[0]
        R = np.repeat(R_lego[None], rows, axis=0)
        R[rng.random(rows) < args.uncertain] = R_unc
        programs["per_row"].append([MeasStream(synth.LEGODO_IDX, lego.z, R), pose])
        programs["per_row_equal"].append([MeasStream(synth.LEGODO_IDX, lego.z, np.repeat(R_lego[None], rows, axis=0)), pose])
        table_bytes.append(rows * 3 * 3 * 8)   # a per-row table without correlated chunks holds the m x m matrix only
    q4 = (p["q_gyro"], p["q_accel"], p["q_gyro_bias"], p["q_accel_bias"])
    name, power_limit, sm_max = card()
    res = {k: [] for k in ("shared", "per_row")}
    enq = {k: [] for k in ("shared", "per_row")}
    with RBISBatch(N) as b:
        b.set_process_noise(*q4)
        stream = torch.cuda.ExternalStream(b.cuda_stream, device=dev)
        preps = {k: [b.prepare_fused(wl.progs[c], imu=wl.chunks[c]["imu"], streams=v[c]) for c in range(args.chunks)]
                 for k, v in programs.items()}
        cyc = {k: [v[i % args.chunks] for i in range(args.launches)] for k, v in preps.items()}
        # bit identity of equal rows, and a warm-up of every program
        outs = {}
        for k in ("shared", "per_row_equal", "per_row"):
            b.set_state(wl.vec0, wl.quat0, wl.cov0)
            for pr in preps[k][:4]:
                b.run_prepared(pr)
            b.synchronize()
            outs[k] = (b.get_state(), b.last_kernel_variant)
        identical = all(np.array_equal(x, y) for x, y in zip(outs["shared"][0][:4], outs["per_row_equal"][0][:4])) and \
            outs["shared"][1] == outs["per_row_equal"][1]
        for rep in range(args.reps):
            for k in (("shared", "per_row") if rep % 2 == 0 else ("per_row", "shared")):
                b.set_state(wl.vec0, wl.quat0, wl.cov0)
                b.synchronize()
                e0, e1 = bench.timed_launches(b, cyc[k], stream, 0, args.launches)
                b.synchronize()
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1)
                res[k].append(N * Tc * args.launches / (ms * 1e-3))
                enq[k].append(bench.timed_launches.enqueue_ms * 1e3)
                variant = b.last_kernel_variant
    med = {k: float(np.median(v)) for k, v in res.items()}
    spread = {k: (max(v) - min(v)) / float(np.median(v)) for k, v in res.items()}
    out = dict(metric="row_noise_filter_steps_per_s", filters=N, chunk_steps=Tc, launches_per_run=args.launches, reps=args.reps,
               uncertain_share=args.uncertain, card=name, power_limit_w=power_limit, sm_max_mhz=sm_max,
               filter_steps_per_s={k: [round(x) for x in v] for k, v in res.items()},
               median={k: round(v) for k, v in med.items()}, spread_rel=spread,
               per_row_vs_shared=med["per_row"] / med["shared"],
               enqueue_us_per_call={k: float(np.mean(v)) for k, v in enq.items()},
               table_bytes_per_call=float(np.mean(table_bytes)), kernel_variant=variant,
               equal_rows_bit_identical_to_shared=bool(identical), time=time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime()))
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
