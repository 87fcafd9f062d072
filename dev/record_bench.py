#!/usr/bin/env python
"""dev/record_bench.py -- cost of recording the trajectory from inside the fused launches (RBIS_OP_RECORD).

BASELINE shape (65,536 filters, 1 kHz IMU, 500 Hz leg odometry, 10 Hz pose fixes, 200-step fused launches, inputs resident
in HBM as bench.py keeps them).  Programs that differ only in their RECORD ops, one every 10 steps (20 record rows per launch):
  none        -- no records: the program bench.py times;
  pose_dev    -- position (state 9-11) + quaternion, 7 fields, into device memory;
  all_dev     -- all 47 fields into device memory;
  pose_host   -- the 7 pose fields into pinned host memory (device staging + one device-to-host copy per launch);
and, with the input rows drawn inside the kernel (rbis_batch_run_fused_synth, mode 1):
  synth_none  -- no records;
  synth_pose  -- the 7 pose fields into device memory.
All run in one process, alternating, --reps times each.  A run is --launches calls from a synchronise to a wait on a ticket
recorded after the last call, timed with the host clock, so a pose_host run includes its last copy.  Prints one JSON line:
filter-steps/s of every run, the median per case and its ratio to the case without records, the bytes recorded per launch, the
pinned-host copy rate, and the card and its power limit read in the same run."""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def with_records(ops, every):
    """A RECORD op (rows 0, 1, ..) before every IMU op of a step that is a multiple of `every` (but the first), and one at the end."""
    from pronto_b200 import capi

    out, row, n_imu = [], 0, 0
    for o in ops:
        if o["kind"] == capi.OP_IMU:
            if n_imu and n_imu % every == 0:
                out.append((capi.OP_RECORD, 0, row, 0, 0.0))
                row += 1
            n_imu += 1
        out.append(tuple(o.tolist()))
    out.append((capi.OP_RECORD, 0, row, 0, 0.0))
    return out, row + 1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--filters", type=int, default=65_536)
    ap.add_argument("--chunk-steps", type=int, default=200)
    ap.add_argument("--chunks", type=int, default=24, help="resident input chunks (each ~0.8 GB at the default size)")
    ap.add_argument("--launches", type=int, default=48, help="fused launches per timed run (cycling through the chunks)")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--every", type=int, default=10, help="steps between records")
    args = ap.parse_args()

    import torch

    import bench
    from row_noise_bench import card
    from pronto_b200 import MeasStream, RBISBatch, SynthSpec, record_fields, synth
    from pronto_b200.batch import make_ops

    if not torch.cuda.is_available():
        raise SystemExit("record_bench.py: no CUDA device")
    dev = torch.device("cuda", 0)
    p = synth.NOMINAL
    N, Tc = args.filters, args.chunk_steps
    R_lego = np.eye(3) * p["r_vxyz"] ** 2
    R_pose = np.diag([p["r_xyz"] ** 2] * 3 + [p["r_chi"] ** 2] * 3)
    wl = bench.Workload(N, Tc, args.chunks, dev, 0x5EED, R_lego, R_pose)
    progs = [with_records(wl.progs[c], args.every) for c in range(args.chunks)]
    rows = progs[0][1]
    assert all(r == rows for _, r in progs)
    pose, full = record_fields(vec=(9, 10, 11), quat=True), (1 << 47) - 1
    k_pose, k_full = bin(pose).count("1"), bin(full).count("1")
    outs = {"pose_dev": torch.empty((rows, k_pose, N), dtype=torch.float64, device=dev),
            "all_dev": torch.empty((rows, k_full, N), dtype=torch.float64, device=dev),
            "pose_host": torch.empty((rows, k_pose, N), dtype=torch.float64).pin_memory(),
            "synth_pose": torch.empty((rows, k_pose, N), dtype=torch.float64, device=dev)}
    masks = {"pose_dev": pose, "all_dev": full, "pose_host": pose, "synth_pose": pose}
    # synthesised inputs: the noise-free rows of each chunk, the same schedule
    specs = []
    for c in range(args.chunks):
        d = synth.synth_spec_inputs(wl.truth, c * Tc, Tc)
        specs.append(SynthSpec(synth.SEED, d["imu_mean"], d["imu_step"], d["streams"], mode=1))
    syn_streams = [MeasStream(synth.LEGODO_IDX, None, R_lego), MeasStream(synth.POSE_IDX, None, R_pose, quat=True)]
    syn_ops = {"synth_none": wl.progs, "synth_pose": [make_ops(prog) for prog, _ in progs]}
    q4 = (p["q_gyro"], p["q_accel"], p["q_gyro_bias"], p["q_accel_bias"])
    name, power_limit, sm_max = card()
    cases = ["none", "pose_dev", "all_dev", "pose_host", "synth_none", "synth_pose"]
    res = {k: [] for k in cases}
    variants = {}
    with RBISBatch(N) as b:
        b.set_process_noise(*q4)
        preps = {"none": wl.prepare(b)}
        for k in ("pose_dev", "all_dev", "pose_host"):
            preps[k] = [b.prepare_fused(progs[c][0], imu=wl.chunks[c]["imu"], streams=wl.streams[c]) for c in range(args.chunks)]

        def run(k):
            if k in masks:
                b.set_record(outs[k], masks[k])
            for i in range(args.launches):
                c = i % args.chunks
                if k.startswith("synth"):
                    b.run_fused_synth(syn_ops[k][c], syn_streams, specs[c])
                else:
                    b.run_prepared(preps[k][c])
            b.wait(b.record())

        for k in cases:   # warm-up of every program
            b.set_state(wl.vec0, wl.quat0, wl.cov0)
            run(k)
            variants[k] = b.last_kernel_variant
        # the records of the three plain recording programs agree where they overlap
        for k in ("pose_dev", "all_dev", "pose_host"):
            b.set_state(wl.vec0, wl.quat0, wl.cov0)
            b.set_record(outs[k], masks[k])
            b.run_prepared(preps[k][0])
            b.synchronize()
        pos = [9, 10, 11, 21, 22, 23, 24]
        consistent = bool(torch.equal(outs["pose_dev"].cpu(), outs["pose_host"]) and torch.equal(outs["pose_dev"], outs["all_dev"][:, pos]))
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
    rec_bytes = {k: rows * bin(m).count("1") * N * 8 for k, m in masks.items()}
    launch_s = Tc * N / med["pose_host"]
    out = dict(metric="record_filter_steps_per_s", filters=N, chunk_steps=Tc, record_every_steps=args.every, record_rows_per_launch=rows,
               launches_per_run=args.launches, reps=args.reps, card=name, power_limit_w=power_limit, sm_max_mhz=sm_max,
               filter_steps_per_s={k: [round(x) for x in v] for k, v in res.items()},
               median={k: round(v) for k, v in med.items()}, spread_rel=spread,
               ratio_vs_no_records={"pose_dev": med["pose_dev"] / med["none"], "all_dev": med["all_dev"] / med["none"],
                                    "pose_host": med["pose_host"] / med["none"], "synth_pose": med["synth_pose"] / med["synth_none"]},
               record_bytes_per_launch=rec_bytes,
               pose_host_copy_gb_per_s_sustained=rec_bytes["pose_host"] / launch_s / 1e9,
               kernel_variant=variants, records_consistent=consistent,
               time=time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime()))
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
