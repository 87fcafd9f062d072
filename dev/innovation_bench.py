#!/usr/bin/env python
"""dev/innovation_bench.py -- cost of the innovation sets (rbis_batch_set_innovations) inside the fused launches.

BASELINE shape (65,536 filters, 1 kHz IMU, 500 Hz leg odometry, 10 Hz pose fixes, 200-step fused launches, inputs resident
in HBM as bench.py keeps them).  The same programs under four settings:
  none       -- no innovation set: the program bench.py times;
  nis        -- NIS of both measurement streams;
  all        -- NIS + y + S(a,a) of both streams;
  all_stats  -- as `all`, plus one statistics pass per call and stream (rbis_batch_stats_innovations_enqueue) over the call's
                rows, the calls alternating between two sets of buffers so that no call waits for a pass.
All run in one process, alternating, --reps times each.  A run is --launches calls from a synchronise to a wait on a ticket
recorded after the last call (and after its statistics passes), timed with the host clock.  Prints one JSON line: filter-steps/s
of every run, the median per case and its ratio to `none`, the bytes written per launch, and the card and its power limit read
in the same run."""
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

    import bench
    from row_noise_bench import card
    from pronto_b200 import RBISBatch, capi, innovation_layout, synth

    if not torch.cuda.is_available():
        raise SystemExit("innovation_bench.py: no CUDA device")
    dev = torch.device("cuda", 0)
    p = synth.NOMINAL
    N, Tc = args.filters, args.chunk_steps
    R_lego = np.eye(3) * p["r_vxyz"] ** 2
    R_pose = np.diag([p["r_xyz"] ** 2] * 3 + [p["r_chi"] ** 2] * 3)
    wl = bench.Workload(N, Tc, args.chunks, dev, 0x5EED, R_lego, R_pose)
    ms = (3, 6)
    rows = [int(max(o["row"] for o in wl.progs[0] if o["kind"] == capi.OP_MEAS and o["stream"] == s)) + 1 for s in (0, 1)]
    for c in range(args.chunks):   # every chunk's MEAS rows start at 0: one buffer row per row of a call
        for s in (0, 1):
            assert int(max(o["row"] for o in wl.progs[c] if o["kind"] == capi.OP_MEAS and o["stream"] == s)) + 1 == rows[s]
    ALL = capi.INNOV_NIS | capi.INNOV_Y | capi.INNOV_S_DIAG
    fields = {"nis": capi.INNOV_NIS, "all": ALL, "all_stats": ALL}
    bufs = {k: [[torch.empty((rows[s], len(innovation_layout(ms[s], f)), N), dtype=torch.float64, device=dev) for s in (0, 1)]
                for _ in range(2 if k == "all_stats" else 1)] for k, f in fields.items()}
    chunk = 1024
    nch = (N + chunk - 1) // chunk
    tables = [[torch.empty((rows[s], nch, capi.NUM_STATS), dtype=torch.float64).pin_memory() for s in (0, 1)] for _ in range(2)]
    q4 = (p["q_gyro"], p["q_accel"], p["q_gyro_bias"], p["q_accel_bias"])
    name, power_limit, sm_max = card()
    cases = ["none", "nis", "all", "all_stats"]
    res = {k: [] for k in cases}
    variants = {}
    with RBISBatch(N) as b:
        b.set_process_noise(*q4)
        preps = wl.prepare(b)

        def run(k):
            for i in range(args.launches):
                c = i % args.chunks
                if k != "none":
                    for s in (0, 1):
                        b.set_innovations(s, bufs[k][i % len(bufs[k])][s], ms[s], fields[k])
                b.run_prepared(preps[c])
                if k == "all_stats":
                    for s in (0, 1):
                        b.stats_innovations_enqueue(s, 0, tables[i % 2][s], None, chunk=chunk)
            b.wait(b.record())
            b.synchronize()   # the statistics passes too
            for s in (0, 1):
                b.clear_innovations(s)

        for k in cases:   # warm-up of every program
            b.set_state(wl.vec0, wl.quat0, wl.cov0)
            run(k)
            variants[k] = b.last_kernel_variant if k == "none" else None
        # which kernels the innovation programs run: one call, variant read back
        b.set_state(wl.vec0, wl.quat0, wl.cov0)
        for s in (0, 1):
            b.set_innovations(s, bufs["all"][0][s], ms[s], ALL)
        b.run_prepared(preps[0])
        variants["all"] = b.last_kernel_variant
        b.synchronize()
        anis = [float(bufs["all"][0][s][:, 0].mean()) for s in (0, 1)]
        for s in (0, 1):
            b.clear_innovations(s)
        for rep in range(args.reps):
            order = cases if rep % 2 == 0 else cases[::-1]
            for k in order:
                b.set_state(wl.vec0, wl.quat0, wl.cov0)
                b.synchronize()
                t0 = time.perf_counter()
                run(k)
                dt = time.perf_counter() - t0
                res[k].append(N * Tc * args.launches / dt)
    med = {k: float(np.median(v)) for k, v in res.items()}
    spread = {k: (max(v) - min(v)) / float(np.median(v)) for k, v in res.items()}
    written = {k: sum(rows[s] * len(innovation_layout(ms[s], f)) * N * 8 for s in (0, 1)) for k, f in fields.items()}
    out = dict(metric="innovation_filter_steps_per_s", filters=N, chunk_steps=Tc, meas_rows_per_launch=rows, launches_per_run=args.launches,
               reps=args.reps, card=name, power_limit_w=power_limit, sm_max_mhz=sm_max,
               filter_steps_per_s={k: [round(x) for x in v] for k, v in res.items()},
               median={k: round(v) for k, v in med.items()}, spread_rel=spread,
               ratio_vs_none={k: med[k] / med["none"] for k in cases[1:]},
               innovation_bytes_per_launch=written, kernel_variant=variants, first_call_anis=anis,
               time=time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime()))
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
