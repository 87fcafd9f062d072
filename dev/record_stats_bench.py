#!/usr/bin/env python
"""dev/record_stats_bench.py -- a NEES / error time series of a Monte-Carlo run from records instead of snapshots.

BASELINE shape (65,536 filters, 1 kHz IMU, 500 Hz leg odometry, 10 Hz pose fixes, 200-step fused launches, inputs resident in
HBM as bench.py keeps them).  One point every --every steps (20 per launch) of the statistics against the truth:
  none        -- no records, no statistics: the program bench.py times;
  rec_stats   -- a RECORD of vec + quat + loglik + covariance blocks {v, chi, p} (71 doubles per filter and row) into one of
                 two alternating device buffers, and ONE rbis_batch_stats_records_enqueue per call over the call's rows;
  snap_stats  -- today's route: a SNAPSHOT into one of 2 x 20 ring slots, and one rbis_batch_stats_snapshot_enqueue per point;
  full_cov    -- a RECORD of vec + quat + loglik + all seven covariance blocks (257 doubles per filter and row) into device
                 memory, no statistics.
All run in one process, alternating, --reps times each.  A run is --launches calls from a synchronise to the end of a
synchronise after the last call (every stream drained, the statistics' copies included), timed with CUDA events on the handle's
stream.  Prints one JSON line: filter-steps/s of every run, the median per case and its ratio to `none`, the bytes each case
writes per launch, whether the two statistics routes agree bit for bit, and the card and its power limit read in the same run."""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def with_points(ops, every, kind, slot0=0):
    """A `kind` op (RECORD rows / SNAPSHOT slots slot0, slot0 + 1, ..) after every `every`-th IMU op; -> (ops, points)."""
    from pronto_b200 import capi

    out, k, n_imu = [], 0, 0
    for o in ops:
        out.append(tuple(o.tolist()))
        if o["kind"] == capi.OP_IMU:
            n_imu += 1
            if n_imu % every == 0:
                out.append((kind, 0, slot0 + k, 0, 0.0))
                k += 1
    return out, k


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--filters", type=int, default=65_536)
    ap.add_argument("--chunk-steps", type=int, default=200)
    ap.add_argument("--chunks", type=int, default=8, help="resident input chunks (each ~0.8 GB at the default size)")
    ap.add_argument("--launches", type=int, default=24, help="fused launches per timed run (cycling through the chunks)")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--every", type=int, default=10, help="steps between statistics points")
    ap.add_argument("--chunk", type=int, default=1024, help="statistics chunk (filters)")
    args = ap.parse_args()

    import torch

    import bench
    from row_noise_bench import card
    from pronto_b200 import RBISBatch, capi, record_fields, record_layout, synth

    if not torch.cuda.is_available():
        raise SystemExit("record_stats_bench.py: no CUDA device")
    dev = torch.device("cuda", 0)
    p = synth.NOMINAL
    N, Tc = args.filters, args.chunk_steps
    R_lego = np.eye(3) * p["r_vxyz"] ** 2
    R_pose = np.diag([p["r_xyz"] ** 2] * 3 + [p["r_chi"] ** 2] * 3)
    wl = bench.Workload(N, Tc, args.chunks, dev, 0x5EED, R_lego, R_pose)
    rec_progs = [with_points(wl.progs[c], args.every, capi.OP_RECORD) for c in range(args.chunks)]
    P = rec_progs[0][1]
    snap_progs = [[with_points(wl.progs[c], args.every, capi.OP_SNAPSHOT, slot0=P * h)[0] for c in range(args.chunks)] for h in (0, 1)]
    state = record_fields(vec=range(21), quat=True, loglik=True)
    nees_blocks, all_blocks = (1, 2, 3), range(7)
    k_nees, k_full = len(record_layout(state, nees_blocks)), len(record_layout(state, all_blocks))
    bufs = [torch.empty((P, k_nees, N), dtype=torch.float64, device=dev) for _ in range(2)]
    full = torch.empty((P, k_full, N), dtype=torch.float64, device=dev)
    nch = (N + args.chunk - 1) // args.chunk
    # truth of each point: the chunk's truth at the point's step
    truth = []
    for c in range(args.chunks):
        tv, tq = zip(*[synth.truth_state_at(wl.truth, c * Tc + (k + 1) * args.every - 1) for k in range(P)])
        truth.append((np.ascontiguousarray(np.stack(tv)), np.ascontiguousarray(np.stack(tq))))
    out_rec = [torch.empty((P, nch, capi.NUM_STATS), dtype=torch.float64).pin_memory() for _ in range(args.launches)]
    out_snap = [torch.empty((P, nch, capi.NUM_STATS), dtype=torch.float64).pin_memory() for _ in range(args.launches)]
    q4 = (p["q_gyro"], p["q_accel"], p["q_gyro_bias"], p["q_accel_bias"])
    name, power_limit, sm_max = card()
    cases = ["none", "rec_stats", "snap_stats", "full_cov"]
    res = {k: [] for k in cases}
    with RBISBatch(N, snapshot_slots=2 * P) as b:
        b.set_process_noise(*q4)
        preps = {"none": wl.prepare(b)}
        preps["rec"] = [b.prepare_fused(rec_progs[c][0], imu=wl.chunks[c]["imu"], streams=wl.streams[c]) for c in range(args.chunks)]
        preps["snap"] = [[b.prepare_fused(snap_progs[h][c], imu=wl.chunks[c]["imu"], streams=wl.streams[c]) for c in range(args.chunks)]
                         for h in (0, 1)]
        stream = torch.cuda.ExternalStream(b.cuda_stream)

        def run(k):
            for i in range(args.launches):
                c = i % args.chunks
                tv, tq = truth[c]
                if k == "none":
                    b.run_prepared(preps["none"][c])
                elif k == "rec_stats":
                    b.set_record(bufs[i % 2], state, nees_blocks)
                    b.run_prepared(preps["rec"][c])
                    b.stats_records_enqueue(0, tv, tq, out_rec[i], chunk=args.chunk)
                elif k == "snap_stats":
                    h = i % 2
                    b.run_prepared(preps["snap"][h][c])
                    for j in range(P):
                        b.stats_snapshot_enqueue(P * h + j, tv[j], tq[j], out_snap[i][j], chunk=args.chunk)
                else:
                    b.set_record(full, state, all_blocks)
                    b.run_prepared(preps["rec"][c])
            b.synchronize()

        for k in cases:   # warm-up of every program
            b.set_state(wl.vec0, wl.quat0, wl.cov0)
            run(k)
        consistent = all(torch.equal(out_rec[i], out_snap[i]) for i in range(args.launches))
        for rep in range(args.reps):
            order = cases if rep % 2 == 0 else cases[::-1]
            for k in order:
                b.set_state(wl.vec0, wl.quat0, wl.cov0)
                b.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                run(k)   # ends in a synchronise of every stream of the handle
                e1.record(stream)
                e1.synchronize()
                res[k].append(N * Tc * args.launches / (e0.elapsed_time(e1) * 1e-3))
    med = {k: float(np.median(v)) for k, v in res.items()}
    spread = {k: (max(v) - min(v)) / float(np.median(v)) for k, v in res.items()}
    written = {"rec_stats": P * k_nees * N * 8, "snap_stats": P * 257 * N * 8,
               "full_cov": P * k_full * N * 8}
    out = dict(metric="record_stats_filter_steps_per_s", filters=N, chunk_steps=Tc, points_per_launch=P, every_steps=args.every,
               stats_chunk=args.chunk, launches_per_run=args.launches, reps=args.reps, card=name, power_limit_w=power_limit,
               sm_max_mhz=sm_max, filter_steps_per_s={k: [round(x) for x in v] for k, v in res.items()},
               median={k: round(v) for k, v in med.items()}, spread_rel=spread,
               ratio_vs_no_records={k: med[k] / med["none"] for k in cases[1:]},
               bytes_written_per_launch=written, stats_routes_bit_identical=bool(consistent),
               time=time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime()))
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
