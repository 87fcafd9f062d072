#!/usr/bin/env python
"""bench.py -- RBIS EKF filter-steps/s on B200 (BASELINE.json metric), one JSON line on stdout.

Headline workload = BASELINE.json configs[2]: IMU 1 kHz + leg-odometry velocity updates 500 Hz (m=3) + pose fixes with
orientation 10 Hz (m=6), fused kernel.  --scaling weak (default): 65,536 filters PER GPU; --scaling strong: 65,536 filters
in total, split over the ranks by contiguous filter ranges (SURVEY.md 8e); the default run reports the strong-scaling number
as an extra leg whenever more than one GPU is used.
One bench "step" = --launches-per-step (5) fused launches, each advancing every filter through a 200-step time chunk, so that
the timed region (K steps) lasts a few hundred milliseconds.  Every launch reads fresh input rows (all chunks of the run are
resident in HBM, each far larger than L2), the state carries over.

  value     filter-steps/s, inputs resident in HBM, CUDA-event timed on the library's stream, barrier + synchronize on
            both sides, max over ranks; the final statistics reduction (rbis_batch_stats_allreduce: device-resident chunk
            table + ncclAllReduce on the library's stream) is inside the timed region.
  e2e       the same metric through the C ABI with HOST (pinned) input buffers: every launch copies its inputs
            host->device and reads the per-chunk statistics back (PCIe bound).
  e2e_synth the Monte-Carlo form of the same call (rbis_batch_run_fused_synth): the host passes the noise-free rows and a
            seed, the per-filter noise is drawn on the device; a 64-filter slice of that very run is checked against the CPU
            oracle fed with the rows the device drew.
  roofline  fused kernel: EXECUTED FP64 flops (ncu instruction counts of profiles/kernel_profile.json, valid only for the
            kernel sources they were captured from) / mean launch time, against the DFMA peak measured in this run; the
            dense algorithmic count of SURVEY.md 8d is reported beside it.
  cpu_baseline  the CPU oracle (restatement of the reference, pinned to the reference's own compiled sources -- DESIGN.md 2)
            on all host threads, 1,024 filters (bounded sample), plus BASELINE.md 3's config-1 run (ONE filter, 60,000
            steps, multimap history, one thread).
  legs      configs[1] (4,096 filters, IMU only), configs[4] (pose fixes 50 steps late: rewind + replay), configs[3]
            (1,048,576-filter parameter sweep, when 4 or 8 GPUs are used), strong scaling (65,536 filters split over the
            ranks), the dense kernel variant, the parameter sweep over shared inputs, the "next" rows.
--impl reference times the CPU path alone on the same workload shape (1,024 filters per step, all host threads).
--dump-outputs DIR writes what the timed steps computed (ensemble state after the last step, reduced statistics) as .npy
files; the inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import gc
import hashlib
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "rbis_ekf_filter_steps_per_s"
UNIT = "filter-steps/s"
F_PROP = 4 * 21 ** 3 + 21 ** 2                     # 37,485  (SURVEY.md 8d)
F_UPD = lambda m: 882 * m + 42 * m * m + 441 + 42 * m
F_CFG3 = (100 * F_PROP + 50 * F_UPD(3) + F_UPD(6)) / 100          # 39,355.47
F_CFG5 = F_CFG3 + (50 * F_PROP + 25 * F_UPD(3)) / 100             # 58,995.72 (replayed steps are not extra filter-steps)
BYTES_PER_STEP = 48 + 24 / 2 + (48 + 32) / 100     # IMU + leg odometry + pose rows actually read (z has 6 columns)
NOMINAL_FP64_TFLOPS = 148 * 64 * 2 * 1.965e9 / 1e12
TOTAL_FILTERS = 65_536
REF_FILTERS = 1024                                  # filters per step of the CPU arms (fixed, stated)
RESIDENT_INPUT_BYTES = 100e9                        # HBM for the input chunks of one run; beyond it they are cycled (180 GB B200)


def kernel_source_sha():
    """sha256 over the CUDA sources the fused kernels are built from: profiles/kernel_profile.json records the value it was
    captured at, and its instruction counts are used only while they match."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "pronto_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cuh", ".cu", ".inc", ".h")) and ("kernels" in f or "group" in f or "fused" in f):
            with open(os.path.join(d, f), "rb") as fh:
                h.update(f.encode() + b"\0" + fh.read())
    return h.hexdigest()[:16]


def kernel_profile(variant):
    """-> (entry or None, reason).  entry: dfma / dmul / dadd warp instructions per warp-step-equivalent (per 32 filter-steps),
    dram bytes per launch with the shape it was captured at."""
    path = os.path.join(ROOT, "profiles", "kernel_profile.json")
    try:
        with open(path) as f:
            prof = json.load(f)
    except Exception as e:
        return None, f"profiles/kernel_profile.json unreadable ({type(e).__name__})"
    sha = kernel_source_sha()
    if prof.get("source_sha") != sha:
        return None, f"profiles/kernel_profile.json was captured at kernel sources {prof.get('source_sha')}, this build is {sha}"
    e = prof.get("variants", {}).get(str(variant))
    if e is None:
        return None, f"no ncu capture for kernel variant {variant} in profiles/kernel_profile.json"
    return e, "ok"


def variant_name(v):
    if v < 0:
        return "none"
    lanes = v >> 4
    base = "decoupled (15x15 active block on chip; chosen at run time because every filter's omega / a covariance couplings are exactly zero, bit-identical to dense)" if v & 2 else "dense (whole 21x21 covariance on chip)"
    mapping = f"warp-group kernel, {lanes} lanes per filter" if lanes else "lane-per-filter kernel"
    return f"{base}; {mapping}" + ("; with one-row / correlated-block paths" if v & 1 else "") + ("; SYN instantiation (input rows drawn in the kernel)" if v & 4 else "")


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --filters per GPU; strong: 65,536 filters in total, split over the ranks (SURVEY.md 8e)")
    ap.add_argument("--filters", type=int, default=TOTAL_FILTERS, help="filters per GPU (weak) / in total (strong)")
    ap.add_argument("--chunk-steps", type=int, default=200, help="IMU steps per fused launch (multiple of 100)")
    ap.add_argument("--launches-per-step", type=int, default=5, help="fused launches per bench step")
    ap.add_argument("--e2e-steps", type=int, default=6)
    ap.add_argument("--cpu-sample-steps", type=int, default=2000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-legs", action="store_true", help="skip the informational legs (other configs, dense variant, next rows)")
    ap.add_argument("--only-legs", default="", help="comma-separated leg names to run (others are skipped); for profiling one leg")
    ap.add_argument("--launch-groups", type=int, default=0, help="0 = library default (automatic)")
    ap.add_argument("--mapping", type=int, default=0, help="lanes per filter (rbis_batch_config_t::mapping); 0 = automatic")
    ap.add_argument("--dense-only", action="store_true", help="force the dense kernel variant (rbis_batch_config_t::dense_only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what they computed (rank 0's ensemble state, the reduced statistics) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    return args


# ------------------------------------------------------------------------------------------------
# synthetic workload
# ------------------------------------------------------------------------------------------------
def chunk_events(Tc, k0):
    """Arrival-ordered events of steps k0..k0+Tc-1 with CHUNK-RELATIVE rows (config-3 schedule)."""
    from pronto_b200 import capi

    ev, li, pi = [], 0, 0
    for i in range(Tc):
        k = k0 + i
        ut = (k + 1) * 1000
        ev.append((capi.OP_IMU, 0, i, ut, 1e-3))
        if k % 2 == 0:
            ev.append((capi.OP_MEAS, 0, li, ut, 0.0)); li += 1
        if k % 100 == 0:
            ev.append((capi.OP_MEAS, 1, pi, ut, 0.0)); pi += 1
    return ev, li, pi


def flops_per_chunk(Tc, n_lego, n_pose):
    return Tc * F_PROP + n_lego * F_UPD(3) + n_pose * F_UPD(6)


def device_chunk(truth, k0, Tc, N, gen, dev):
    """Noisy input rows of one time chunk, generated on the device (synthetic data plumbing)."""
    import torch

    from pronto_b200 import synth

    p = synth.NOMINAL
    steps = np.arange(k0, k0 + Tc)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    sg, sa = math.sqrt(p["q_gyro"] / p["dt"]), math.sqrt(p["q_accel"] / p["dt"])
    imu = torch.randn((Tc, 6, N), dtype=torch.float64, device=dev, generator=gen)
    imu[:, 0:3] *= sg
    imu[:, 3:6] *= sa
    imu[:, 0:3] += t(truth["gyro_in"][steps])[:, :, None]
    imu[:, 3:6] += t(truth["accel_in"][steps])[:, :, None]
    ls, ps = steps[steps % 2 == 0], steps[steps % 100 == 0]
    lego = torch.randn((len(ls), 3, N), dtype=torch.float64, device=dev, generator=gen) * p["r_vxyz"]
    lego += t(truth["v"][ls])[:, :, None]
    pz = torch.zeros((len(ps), 6, N), dtype=torch.float64, device=dev)
    pz[:, 0:3] = torch.randn((len(ps), 3, N), dtype=torch.float64, device=dev, generator=gen) * p["r_xyz"] + t(truth["p"][ps])[:, :, None]
    chi = torch.randn((len(ps), 3, N), dtype=torch.float64, device=dev, generator=gen) * p["r_chi"]
    n = torch.linalg.norm(chi, dim=1, keepdim=True).clamp_min(1e-300)
    dq = torch.cat([torch.cos(0.5 * n), torch.sin(0.5 * n) * chi / n], dim=1)
    tq = t(truth["quat"][ps])[:, :, None]
    w0, x0, y0, z0 = (tq[:, i] for i in range(4))
    w1, x1, y1, z1 = (dq[:, i] for i in range(4))
    pq = torch.stack([w0 * w1 - x0 * x1 - y0 * y1 - z0 * z1, w0 * x1 + x0 * w1 + y0 * z1 - z0 * y1,
                      w0 * y1 + y0 * w1 + z0 * x1 - x0 * z1, w0 * z1 + z0 * w1 + x0 * y1 - y0 * x1], dim=1)
    return dict(imu=imu.contiguous(), legodo=lego.contiguous(), pose_z=pz.contiguous(), pose_q=pq.contiguous())


def initial_state(N, gen, dev):
    import torch

    from pronto_b200 import synth

    p = synth.NOMINAL
    sig = np.zeros(21)
    sig[3:6], sig[6:9], sig[9:12], sig[15:18], sig[18:21] = p["sigma_v"], p["sigma_chi"], p["sigma_p"], p["sigma_bg"], p["sigma_ba"]
    tv = np.zeros(21)
    tv[9:12] = (0, 0, 0.85); tv[15:18] = p["bg"]; tv[18:21] = p["ba"]
    d = torch.randn((21, N), dtype=torch.float64, device=dev, generator=gen) * torch.from_numpy(sig).to(dev)[:, None]
    vec = torch.from_numpy(tv).to(dev)[:, None] + d
    chi = vec[6:9].clone()
    vec[6:9] = 0
    n = torch.linalg.norm(chi, dim=0, keepdim=True).clamp_min(1e-300)
    quat = torch.cat([torch.cos(0.5 * n), torch.sin(0.5 * n) * chi / n], dim=0).contiguous()
    cov = torch.zeros((441, N), dtype=torch.float64, device=dev)
    for i in range(21):
        cov[i + 21 * i] = sig[i] ** 2
    return vec.contiguous(), quat, cov


class ClockSampler:
    """SM clock / throttle-reason sampling during the timed region.  NVML in-process (pynvml) every 20 ms --
    far less intrusive than polling the nvidia-smi binary, which showed up as 5-10 ms hiccups inside the timed
    region; nvidia-smi is the fallback when NVML cannot be loaded."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.nv, self.stop_flag = index, [], None, None, False

    def _physical_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if self.index < len(ids) and ids[self.index].isdigit():
                return int(ids[self.index])
        return self.index

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index())
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            for _ in range(2):  # the first queries are slow (tens of ms): take them before the timed region
                pynvml.nvmlDeviceGetClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
                pynvml.nvmlDeviceGetPowerUsage(self.handle)
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
            return
        except Exception:
            self.nv = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self._physical_index())], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def sample_once(self):
        """One NVML sample from the calling thread (used between launches: the host runs ahead of the GPU there)."""
        self.poll_while(lambda: True, period=0.0, max_samples=1)

    def poll_while(self, busy, period=0.008, stop_after=1e9, max_samples=1 << 30):
        """NVML path: sample from the CALLING thread while busy() holds (the host only waits for the GPU during
        that time, so the queries cannot delay host-side work of the timed region).  No-op on the nvidia-smi path."""
        nv = self.nv
        if nv is None:
            return
        bits = (("hw_slowdown", nv.nvmlClocksThrottleReasonHwSlowdown), ("hw_thermal_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown),
                ("sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwThermalSlowdown), ("sw_power_cap", nv.nvmlClocksThrottleReasonSwPowerCap))
        t_stop = time.time() + stop_after
        taken = 0
        while busy() and time.time() < t_stop and taken < max_samples:
            taken += 1
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM))
                pw = nv.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.rows.append((time.time(), sm, pw, [n for n, b in bits if mask & b]))
            except Exception:
                pass
            if period > 0:
                time.sleep(period)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if self.nv is not None:
            rows = [r for r in self.rows if t0 - 0.02 <= r[0] <= t1 + 0.02] or self.rows
            if not rows:
                return {"sm_mhz": None, "sm_max_mhz": self.max_sm, "reasons": ["no samples"]}
            sm = sorted(r[1] for r in rows)
            return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.max_sm, "power_w_max": max(r[2] for r in rows), "samples": len(rows),
                    "reasons": sorted({n for r in rows for n in r[3]}), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for ts, r in self.rows if t0 - 0.05 <= ts <= t1 + 0.15 and len(r) >= 9] or [r for _, r in self.rows if len(r) >= 9]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(float(r[1]) for r in rows)
        reasons = set()
        for r in rows:
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][2]), "power_w_max": max(float(r[3]) for r in rows),
                "samples": len(rows), "reasons": sorted(reasons), "source": "nvidia-smi"}


# ------------------------------------------------------------------------------------------------
# CPU oracle timing (cpu_baseline leg and --impl reference)
# ------------------------------------------------------------------------------------------------
def cpu_oracle_rate(Tc, n_filters, threads, repeats=1):
    """filter-steps/s of the CPU oracle (all `threads` host threads) on the config-3 schedule.  -> (rate, times, the last
    run's result: run_ensemble's dict)."""
    from oracle import oracle_api
    from pronto_b200 import synth

    sys.path.insert(0, os.path.join(ROOT, "tests"))
    oracle_api.build()
    truth = synth.truth_trajectory(Tc)
    tv = np.zeros(21)
    tv[9:12] = (0, 0, 0.85); tv[15:18] = synth.NOMINAL["bg"]; tv[18:21] = synth.NOMINAL["ba"]
    vec, quat, cov = synth.initial_ensemble(n_filters, tv, np.array([1.0, 0, 0, 0]))
    st = synth.make_streams(truth, n_filters, 0, Tc)
    p = synth.NOMINAL
    q = (p["q_gyro"], p["q_accel"], p["q_gyro_bias"], p["q_accel_bias"])
    streams = [dict(idx=synth.LEGODO_IDX, z=st["legodo"], R=st["R_legodo"]),
               dict(idx=synth.POSE_IDX, z=st["pose_z"], R=st["R_pose"], quat=st["pose_q"])]
    times = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        out = oracle_api.run_ensemble(vec, quat, cov, None, 0, q, st["imu"], streams, st["events"], n_threads=threads)
        times.append(time.perf_counter() - t0)
        assert np.isfinite(out["vec"]).all()
    return n_filters * Tc / min(times), times, out


def cpu_config1_rate():
    """BASELINE.md 3's config-1 run: ONE filter, 60,000 IMU steps at 1 kHz + 30,000 leg-odometry updates, the reference's
    time-ordered multimap history, one thread.  -> (filter-steps/s, seconds)."""
    from oracle import oracle_api
    from pronto_b200 import synth

    oracle_api.build()
    T = 60_000
    truth = synth.truth_trajectory(T)
    tv = np.zeros(21)
    tv[9:12] = (0, 0, 0.85); tv[15:18] = synth.NOMINAL["bg"]; tv[18:21] = synth.NOMINAL["ba"]
    vec, quat, cov = synth.initial_ensemble(1, tv, np.array([1.0, 0, 0, 0]))
    st = synth.make_streams(truth, 1, 0, T, with_pose=False)
    p = synth.NOMINAL
    q = (p["q_gyro"], p["q_accel"], p["q_gyro_bias"], p["q_accel_bias"])
    t0 = time.perf_counter()
    out = oracle_api.run_ensemble(vec, quat, cov, None, 0, q, st["imu"], [dict(idx=synth.LEGODO_IDX, z=st["legodo"], R=st["R_legodo"])],
                                  st["events"], n_threads=1)
    dt = time.perf_counter() - t0
    assert np.isfinite(out["vec"]).all()
    return T / dt, dt


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle restatement; the reference itself needs Eigen, eigen_utils, LCM and
    libbot, none present) on all host threads, a FIXED 1,024 filters x chunk_steps per step.  Rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    threads = os.cpu_count() or 1
    Tc = args.chunk_steps
    n_filters = REF_FILTERS
    K, W = args.steps, args.warmup
    rates = []
    for i in range(W + K):
        r, _, out = cpu_oracle_rate(Tc, n_filters, threads)
        if i >= W:
            rates.append(r)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out["vec"], out["quat"], out["cov"], out["loglik"])
    total_t = sum(n_filters * Tc / r for r in rates)
    value = K * n_filters * Tc / total_t
    sample = f"{n_filters} filters x {Tc} steps per bench step (config-3 schedule), {threads} threads"
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus, "steps": K, "warmup": W,
        "ms_per_step": 1e3 * total_t / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": "configs[2]: IMU 1 kHz + leg-odometry 500 Hz (m=3) + pose fix 10 Hz (m=6)",
                   "filters_per_step": n_filters, "chunk_steps": Tc, "host_threads": threads},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample, "per_thread_value": value / threads},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def bind_to_gpu_numa_node(local, rank):
    """Pin this rank's host threads to the CPUs NVML reports as local to its GPU, BEFORE any pinned buffer is
    allocated: first-touch then places the staging memory on the GPU's NUMA node, which is what decides the
    host->device rate once several ranks copy at the same time."""
    try:
        import pynvml

        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = local
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if local < len(ids) and ids[local].isdigit():
                idx = int(ids[local])
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            log(f"[rank {rank}] bound to {len(cpus)} CPUs local to GPU {idx}")
    except Exception as e:  # affinity is an optimisation only
        log(f"[rank {rank}] no NUMA binding ({type(e).__name__}: {e})")


# ------------------------------------------------------------------------------------------------
class Workload:
    """Config-3 inputs of one rank resident in HBM: n_launches time chunks of Tc steps for N filters."""

    def __init__(self, N, Tc, n_launches, dev, seed, R_lego, R_pose, imu_only=False):
        import torch

        from pronto_b200 import MeasStream, synth
        from pronto_b200.batch import make_ops

        self.N, self.Tc, self.n = N, Tc, n_launches
        self.truth = synth.truth_trajectory(n_launches * Tc)
        gen = torch.Generator(device=dev)
        gen.manual_seed(seed)
        self.vec0, self.quat0, self.cov0 = initial_state(N, gen, dev)
        self.chunks, self.progs, self.streams = [], [], []
        for c in range(n_launches):
            ch = device_chunk(self.truth, c * Tc, Tc, N, gen, dev)
            ev, n_lego, n_pose = chunk_events(Tc, c * Tc)
            if imu_only:
                ev, n_lego, n_pose = [e for e in ev if e[0] == 0], 0, 0
                ch = dict(imu=ch["imu"])
            self.chunks.append(ch)
            self.progs.append(make_ops(ev))
            self.streams.append([] if imu_only else [MeasStream(synth.LEGODO_IDX, ch["legodo"], R_lego),
                                                     MeasStream(synth.POSE_IDX, ch["pose_z"], R_pose, quat=ch["pose_q"])])
        self.flops_chunk = flops_per_chunk(Tc, n_lego, n_pose) * N
        self.in_bytes = sum(int(v.numel()) * 8 for v in self.chunks[0].values())
        torch.cuda.synchronize()

    def prepare(self, b):
        return [b.prepare_fused(self.progs[c], imu=self.chunks[c]["imu"], streams=self.streams[c]) for c in range(self.n)]


DUMP_STATE_FILTERS = 65_536    # filters whose vec / quat / loglik --dump-outputs writes (every filter at the default size)
DUMP_COV_FILTERS = 4_096       # filters whose covariance it writes (441 doubles each)


def dump_outputs(path, vec, quat, cov, loglik, stats=None):
    """--dump-outputs: what a caller of the timed path holds after its last step -- the ensemble state vec [21][N], quat [4][N],
    cov [441][N], loglik [N] (numpy or torch arrays) and, where the path computes them, the reduced statistics -- as float64 .npy
    files.  Larger ensembles are represented by a fixed, seeded sample of filters (their indices are written beside them), so the
    files stay below 32 MB for any --filters."""
    N = vec.shape[-1]

    def sample(k, seed):
        if N <= k:
            return np.arange(N)
        return np.sort(np.random.default_rng(seed).choice(N, size=k, replace=False))

    def pick(t, idx):
        if isinstance(t, np.ndarray):
            return t[..., idx]
        import torch

        return t[..., torch.from_numpy(idx).to(t.device)].cpu().numpy()

    s, sc = sample(DUMP_STATE_FILTERS, 1), sample(DUMP_COV_FILTERS, 2)
    out = {"vec": pick(vec, s), "quat": pick(quat, s), "loglik": pick(loglik, s), "state_filters": s,
           "cov": pick(cov, sc), "cov_filters": sc}
    if stats is not None:
        out["stats"] = stats
    os.makedirs(path, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))
    log(f"[rank 0] wrote {', '.join(sorted(out))} (.npy) to {path}")


def timed_launches(b, preps, stream, first, count, sampler=None):
    """`count` prepared fused launches timed as ONE region on the library's stream (launches overlap through the launch
    groups, so a per-launch event pair would not bracket one launch).  -> (ms total, event0, event1)."""
    import torch

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    t_first = []
    for i in range(count):
        t0 = time.perf_counter()
        b.run_prepared(preps[first + i])
        if i < 6:
            t_first.append(time.perf_counter() - t0)
        if sampler is not None and i >= 2 and i % 6 == 2 and i < count - 1:
            sampler.sample_once()  # clocks under load; the host is several launches ahead of the GPU here
    b.record()
    e1.record(stream)
    # host cost of one rbis_batch_run_fused call: the first six calls after a synchronise, i.e. before the library's 8-deep
    # launch ring makes the host wait for the device (after that a call returns at the device's pace by design)
    timed_launches.enqueue_ms = 1e3 * float(np.mean(t_first)) if t_first else None
    return e0, e1


def run_b200(args):
    import torch
    import torch.distributed as dist

    import __graft_entry__ as ge
    from pronto_b200 import MeasStream, RBISBatch, SynthSpec, capi, measure_fp64_peak, synth
    from pronto_b200.batch import make_ops, reduce_chunks
    from pronto_b200.ensemble import shard_range, summarize
    from pronto_b200.nccl import Communicator

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; pronto_b200 has no CPU path (use --impl reference for the CPU baseline)")
    if not os.path.exists(ge.LIB):
        ge.build_cuda()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    bind_to_gpu_numa_node(local, rank)
    comm = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        comm = Communicator(rank, world, local)   # raw ncclComm_t for the C ABI's statistics all-reduce
    Tc, K, W, L = args.chunk_steps, args.steps, args.warmup, args.launches_per_step
    assert Tc % 100 == 0 and Tc > 0 and L >= 1
    CHUNK = 1024
    strong = args.scaling == "strong"
    if strong:
        lo, hi = shard_range(args.filters, rank, world, CHUNK)
        N, n_total = hi - lo, args.filters
    else:
        N, n_total, lo = args.filters, args.filters * world, rank * args.filters
    p = synth.NOMINAL
    R_lego = np.eye(3) * p["r_vxyz"] ** 2
    R_pose = np.diag([p["r_xyz"] ** 2] * 3 + [p["r_chi"] ** 2] * 3)
    q4 = (p["q_gyro"], p["q_accel"], p["q_gyro_bias"], p["q_accel_bias"])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def new_batch(n, **kw):
        b = RBISBatch(n, device=local, launch_groups=args.launch_groups, mapping=args.mapping, **kw)
        b.set_process_noise(*q4)
        return b

    # ---- FP64 roofline denominator, measured here ----
    dfma_tf, dmma_tf = measure_fp64_peak(local, 4000)
    log(f"[rank {rank}] FP64 peak measured: DFMA {dfma_tf:.2f} TFLOP/s, DMMA(mma.sync m8n8k4) {dmma_tf:.2f} TFLOP/s")

    # ---- synthetic inputs: all launches of the run resident in HBM, up to the fixed RESIDENT_INPUT_BYTES (not the free memory,
    # so that the same arguments give the same inputs, and hence the same outputs, on every run and machine) ----
    n_launches = (W + K) * L
    chunk_bytes = N * Tc * (48 + 12 + 0.8) * 1.02
    resident = max(2, min(n_launches, int(RESIDENT_INPUT_BYTES / chunk_bytes)))
    free_b, _ = torch.cuda.mem_get_info()
    if resident * chunk_bytes > 0.6 * free_b:
        raise SystemExit(f"bench.py: the run's resident inputs ({resident} chunks, {resident * chunk_bytes / 1e9:.1f} GB) need more than 60% "
                         f"of the {free_b / 1e9:.1f} GB free on cuda:{local}; other processes hold the device's memory")
    wl = Workload(N, Tc, resident, dev, 0x5EED + rank, R_lego, R_pose)
    b = new_batch(N, dense_only=args.dense_only)
    b.set_state(wl.vec0, wl.quat0, wl.cov0)
    b.synchronize()
    preps = wl.prepare(b)
    preps = [preps[i % resident] for i in range(n_launches)]   # cycled only when the run does not fit in memory
    stream = torch.cuda.ExternalStream(b.cuda_stream, device=dev)
    tv, tq = synth.truth_state_at(wl.truth, min(n_launches, resident) * Tc - 1)
    first_chunk, total_chunks = lo // CHUNK, (n_total + CHUNK - 1) // CHUNK

    # ---- warm-up ----
    w0, w1 = timed_launches(b, preps, stream, 0, W * L)
    b.stats_allreduce(comm, tv, tq, first_chunk, total_chunks, chunk=CHUNK)  # warm-up of the statistics path too
    barrier()
    b.synchronize()

    # ---- timed region: K steps x L fused launches + the final statistics all-reduce ----
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    launches0 = b.launch_count
    gc.collect()
    gc.disable()
    barrier()  # last thing before the clock starts: any skew between the ranks here is paid for in the final all-reduce
    b.synchronize()
    t_wall0 = time.time()
    ev0, evk = timed_launches(b, preps, stream, W * L, K * L, sampler)
    enqueue_ms = timed_launches.enqueue_ms
    totals, _ = b.stats_allreduce(comm, tv, tq, first_chunk, total_chunks, chunk=CHUNK)
    end = torch.cuda.Event(enable_timing=True)
    end.record(stream)
    barrier()
    b.synchronize()
    gc.enable()
    t_wall1 = time.time()
    clocks = sampler.stop(t_wall0, t_wall1)
    launches = b.launch_count - launches0
    variant = b.last_kernel_variant
    total_ms = ev0.elapsed_time(end)
    k_ms = ev0.elapsed_time(evk) / (K * L)
    log(f"[rank {rank}] {K * L} fused launches ({N} filters x {Tc} steps each): {ev0.elapsed_time(evk):.3f} ms = {k_ms:.3f} ms per launch; host enqueue "
        f"{enqueue_ms:.3f} ms per call (first six calls, before the 8-deep launch ring paces the host); statistics + all-reduce tail {evk.elapsed_time(end):.3f} ms; total {total_ms:.3f} ms")
    total_ms = max_over_ranks(total_ms)
    value = n_total * Tc * K * L / (total_ms * 1e-3)
    summ = summarize(totals)
    stats_sha = hashlib.sha256(np.ascontiguousarray(totals).tobytes()).hexdigest()[:16]
    log(f"[rank {rank}] ensemble after {n_launches * Tc} steps: filters={summ['filters']} non_finite={summ['non_finite']} "
        f"mean NEES(9)={summ['mean_nees']:.3f} in-95%={summ['nees_in_95pct']:.3f} rms pos err={np.sqrt(np.mean(summ['rms_err'][9:12] ** 2)):.4f} m")
    if args.dump_outputs and rank == 0:
        st = [torch.empty(shape, dtype=torch.float64, device=dev) for shape in ((21, N), (4, N), (441, N), (N,))]
        b.get_state_into(*st)
        b.synchronize()
        dump_outputs(args.dump_outputs, *st, stats=totals)
        del st

    legs = {}

    def leg(name, fn, when=True):
        """Informational legs never take the headline down with them."""
        if not when or args.no_legs or (args.only_legs and name not in args.only_legs.split(",")):
            return
        try:
            t0 = time.time()
            legs[name] = fn()
            log(f"[rank {rank}] leg {name}: {time.time() - t0:.1f} s")
        except Exception as e:  # noqa: BLE001
            legs[name] = {"error": f"{type(e).__name__}: {e}"}
            log(f"[rank {rank}] leg {name} FAILED: {type(e).__name__}: {e}")
        gc.collect()
        torch.cuda.empty_cache()

    # ---- the dense kernel variant on the same launches (what a coupled ensemble would get) + bit-identity check ----
    def dense_leg():
        n_l = min(resident, 6 * L)
        with new_batch(N, dense_only=True) as bd:
            bd.set_state(wl.vec0, wl.quat0, wl.cov0)
            pd = wl.prepare(bd)
            sd = torch.cuda.ExternalStream(bd.cuda_stream, device=dev)
            timed_launches(bd, pd, sd, 0, min(W * L, n_l))
            bd.set_state(wl.vec0, wl.quat0, wl.cov0)
            bd.synchronize()
            d0, d1 = timed_launches(bd, pd, sd, 0, n_l)
            bd.synchronize()
            torch.cuda.synchronize()
            d_ms = d0.elapsed_time(d1) / n_l
            with new_batch(N) as bc:   # the headline kernels over the same launches from the same start
                bc.set_state(wl.vec0, wl.quat0, wl.cov0)
                pc = wl.prepare(bc)
                timed_launches(bc, pc, torch.cuda.ExternalStream(bc.cuda_stream, device=dev), 0, n_l)

                def dev_state(h):
                    v = torch.empty((21, N), dtype=torch.float64, device=dev)
                    c = torch.empty((441, N), dtype=torch.float64, device=dev)
                    l = torch.empty((N,), dtype=torch.float64, device=dev)
                    h.get_state_into(vec=v, cov=c, loglik=l)
                    h.synchronize()
                    return v, c, l

                same = all(bool(torch.equal(x, y)) for x, y in zip(dev_state(bc), dev_state(bd)))
            return {"value": N * Tc / (d_ms * 1e-3), "unit": UNIT, "kernel_ms": d_ms, "kernel_variant": variant_name(bd.last_kernel_variant),
                    "launches": n_l, "bit_identical_to_headline_kernels": same, "this_rank_only": True}

    leg("dense_variant", dense_leg, when=(variant & 2) != 0 and world == 1)

    # ---- e2e: host (pinned) inputs through the C ABI; one step = the headline's step (L fused launches, each with its own
    # host->device input copy) followed by the read-back of the step's statistics on the host ----
    # Reading a result keeps the calls on either side of it from overlapping, so these legs run on a handle whose calls are
    # cut into pieces of ~100 ops (rbis_batch_config_t::piece_ops): the partially filled last wave of one piece overlaps the next.
    e2e = e2e_f32 = None
    n_local = (N + CHUNK - 1) // CHUNK
    if not args.no_e2e:
        b.close()
        b = new_batch(N, dense_only=args.dense_only, piece_ops=100, snapshot_slots=2)
        stream = torch.cuda.ExternalStream(b.cuda_stream, device=dev)
        def with_snapshot(prog, slot):
            """the step's last program also leaves the ensemble in ring slot `slot`, for the side-stream statistics"""
            return np.concatenate([prog, make_ops([(capi.OP_SNAPSHOT, 0, slot, int(prog["utime"][-1]), 0.0)])])

        def host_e2e(rows_dtype):
            """rows_dtype None: the chunks as they are (float64); torch.float32: the same rows rounded to float and passed as float
            arrays (RBIS_MEM_F32_ROWS: widened exactly on the device, half the PCIe bytes)"""
            E = max(1, min(args.e2e_steps, K * L))
            ring = min(3, resident)
            host = [{k: torch.empty(v.shape, dtype=rows_dtype or v.dtype, pin_memory=True).copy_(v) for k, v in wl.chunks[c].items()} for c in range(ring)]
            torch.cuda.synchronize()
            hnp = [{k: v.numpy() for k, v in h.items()} for h in host]
            hstreams = lambda c: [MeasStream(synth.LEGODO_IDX, hnp[c]["legodo"], R_lego), MeasStream(synth.POSE_IDX, hnp[c]["pose_z"], R_pose, quat=hnp[c]["pose_q"])]
            hprep = [b.prepare_fused(wl.progs[c], imu=hnp[c]["imu"], streams=hstreams(c)) for c in range(ring)]
            hprep_last = [[b.prepare_fused(with_snapshot(wl.progs[c], s_), imu=hnp[c]["imu"], streams=hstreams(c)) for s_ in range(2)] for c in range(ring)]
            res = [torch.empty((n_local, capi.NUM_STATS), dtype=torch.float64, pin_memory=True) for _ in range(2)]
            resnp = [r.numpy() for r in res]
            b.set_state(wl.vec0, wl.quat0, wl.cov0)

            def e2e_step(i):
                for j in range(L - 1):
                    b.run_prepared(hprep[(i * L + j) % ring])
                b.run_prepared(hprep_last[(i * L + L - 1) % ring][i % 2])
                return b.stats_snapshot_enqueue(i % 2, tv, tq, resnp[i % 2], chunk=CHUNK)

            tick = None
            for i in range(2):  # warm-up (allocates the staging buffers)
                t = e2e_step(i)
                if tick is not None:
                    b.wait(tick)
                tick = t
            b.wait(tick)
            barrier()
            b.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = b.launch_count
            e0.record(stream)
            tick, acc = None, 0.0
            for i in range(E):
                t = e2e_step(i)
                if tick is not None:
                    b.wait(tick)
                    acc += float(resnp[(i - 1) % 2][0, 46])  # the launch's result is read on the host
                tick = t
            b.wait(tick)
            acc += float(resnp[(E - 1) % 2][0, 46])
            e1.record(stream)
            barrier()
            b.synchronize()
            e2e_ms = max_over_ranks(e0.elapsed_time(e1))
            assert acc == E * min(CHUNK, N)
            return {"value": n_total * Tc * L * E / (e2e_ms * 1e-3), "unit": UNIT,
                   "h2d_bytes_per_step": L * (sum(int(v.numel() * v.element_size()) for v in host[0].values()) + wl.progs[0].nbytes),
                   "d2h_bytes_per_step": n_local * capi.NUM_STATS * 8, "steps": E, "ms_per_step": e2e_ms / E,
                   "step": f"{L} fused launches ({Tc} trajectory steps of every filter each), every one with its own host->device input copy from pinned "
                           "memory; the last one snapshots the ensemble, whose statistics are computed on a side stream and read back on the host "
                           "(rbis_batch_stats_snapshot_enqueue) while the next step already runs",
                   "bound": "PCIe: per-filter input rows cross the bus", "launches_per_step": (b.launch_count - l0) / E}
        e2e = host_e2e(None)
        e2e_f32 = host_e2e(torch.float32)
        e2e_f32["what"] = ("the same steps with the sensor rows rounded to float32 and passed as float arrays (RBIS_MEM_F32_ROWS): widened exactly on "
                           "the device, half the bytes over PCIe; a different ensemble from `e2e` only in that rounding of its inputs")

    # ---- e2e_synth: the Monte-Carlo form of the call -- noise-free rows + seed from the host, noise drawn on the device ----
    e2e_synth = None
    if not args.no_e2e:
        E = max(2, min(args.e2e_steps, K * L))
        SEED = 0x5EED20261018
        specs = []
        for c in range((E + 2) * L):
            d = synth.synth_spec_inputs(wl.truth, (c % resident) * Tc, Tc)
            specs.append(SynthSpec(SEED, d["imu_mean"], d["imu_step"], d["streams"], mode=1, first_filter=lo))
        sstreams = [MeasStream(synth.LEGODO_IDX, None, R_lego), MeasStream(synth.POSE_IDX, None, R_pose, quat=True)]
        spec_bytes = sum(int(a.nbytes) for a in specs[0].keep)
        res_s = [torch.empty((n_local, capi.NUM_STATS), dtype=torch.float64, pin_memory=True).numpy() for _ in range(2)]

        def synth_step(i):
            for j in range(L - 1):
                b.run_fused_synth(wl.progs[(i * L + j) % resident], sstreams, specs[i * L + j])
            b.run_fused_synth(with_snapshot(wl.progs[(i * L + L - 1) % resident], i % 2), sstreams, specs[i * L + L - 1])
            return b.stats_snapshot_enqueue(i % 2, tv, tq, res_s[i % 2], chunk=CHUNK)

        b.set_state(wl.vec0, wl.quat0, wl.cov0)
        tick = None
        for i in range(E, E + 2):  # warm-up
            t = synth_step(i)
            if tick is not None:
                b.wait(tick)
            tick = t
        b.wait(tick)
        b.set_state(wl.vec0, wl.quat0, wl.cov0)
        barrier()
        b.synchronize()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = b.launch_count
        s0.record(stream)
        tick, acc = None, 0.0
        for i in range(E):
            t = synth_step(i)
            if tick is not None:
                b.wait(tick)
                acc += float(res_s[(i - 1) % 2][0, 46])
            tick = t
        b.wait(tick)
        acc += float(res_s[(E - 1) % 2][0, 46])
        s1.record(stream)
        barrier()
        b.synchronize()
        syn_ms = max_over_ranks(s0.elapsed_time(s1))
        e2e_synth = {"value": n_total * Tc * L * E / (syn_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": L * (spec_bytes + wl.progs[0].nbytes),
                     "d2h_bytes_per_step": n_local * capi.NUM_STATS * 8, "steps": E, "ms_per_step": syn_ms / E,
                     "launches_per_step": (b.launch_count - l0) / E, "generator": "splitmix64 counters -> Box-Muller, fast mode (rbis_synth_t::mode 1)",
                     "kernel_variant": variant_name(b.last_kernel_variant),
                     "what": f"rbis_batch_run_fused_synth, {L} calls per step + statistics read-back (of the snapshot the step's last program "
                             "leaves, on a side stream): the host sends the noise-free rows and a seed, the fused kernel draws every filter's noisy "
                             "rows itself (SYN instantiation) -- no per-filter input exists in HBM"}
        prof_s, why_s = kernel_profile(b.last_kernel_variant)
        if prof_s:
            ex_s = 2 * prof_s["dfma"] + prof_s["dmul"] + prof_s["dadd"]
            e2e_synth["roofline"] = {"bound": "fp64", "peak": dfma_tf, "unit": "TFLOP/s", "executed_flops_per_filter_step": ex_s,
                                     "achieved": e2e_synth["value"] / world * ex_s / 1e12, "frac": e2e_synth["value"] / world * ex_s / 1e12 / dfma_tf,
                                     "warp_instructions_per_32_filter_steps": prof_s.get("warp_instructions"), "executed_source": prof_s.get("source"),
                                     "note": "end-to-end rate (statistics read-back included) x executed flops of the SYN kernel instantiation"}
        else:
            e2e_synth["roofline"] = {"achieved": None, "frac": None, "executed_unavailable": why_s}
        # parity of THIS run on a slice: filters 0..63 of rank 0 replayed by the CPU oracle from the rows the device drew
        if rank == 0:
            try:
                from oracle import oracle_api
                from pronto_b200.parity import max_errors

                oracle_api.build()
                S = min(64, N)
                gv = torch.empty((21, N), dtype=torch.float64, device=dev); gq = torch.empty((4, N), dtype=torch.float64, device=dev)
                gc_ = torch.empty((441, N), dtype=torch.float64, device=dev)
                b.get_state_into(vec=gv, quat=gq, cov=gc_)
                b.synchronize()
                rv = wl.vec0[:, :S].cpu().numpy().copy(); rq = wl.quat0[:, :S].cpu().numpy().copy(); rP = wl.cov0[:, :S].cpu().numpy().copy()
                rll, ut = np.zeros(S), 0
                with new_batch(S) as bs:
                    for i in range(E * L):
                        d = synth.synth_spec_inputs(wl.truth, (i % resident) * Tc, Tc)
                        rows = bs.synthesize(SynthSpec(SEED, d["imu_mean"], d["imu_step"], d["streams"], mode=1, first_filter=lo))
                        ev = [(int(o["kind"]), int(o["stream"]), int(o["row"]), int(o["utime"]), float(o["dt"])) for o in wl.progs[i % resident]]
                        ref = oracle_api.run_ensemble(rv, rq, rP, rll, ut, q4, rows["imu"].cpu().numpy(),
                                                      [dict(idx=synth.LEGODO_IDX, z=rows["z"][0].cpu().numpy(), R=R_lego),
                                                       dict(idx=synth.POSE_IDX, z=rows["z"][1].cpu().numpy(), R=R_pose, quat=rows["quat"][1].cpu().numpy())],
                                                      ev, n_threads=os.cpu_count() or 1)
                        rv, rq, rP, rll, ut = ref["vec"], ref["quat"], ref["cov"], ref["loglik"], ev[-1][3]
                err = max_errors(gv[:, :S].cpu().numpy(), gq[:, :S].cpu().numpy(), gc_[:, :S].cpu().numpy(), rv, rq, rP)
                e2e_synth["parity_slice"] = {"filters": S, "steps": E * L * Tc, "max_err_vs_cpu_oracle": err, "gate": 1e-6,
                                             "ok": bool(max(err.values()) < 1e-6)}
                log(f"[rank 0] e2e_synth parity slice ({S} filters x {E * L * Tc} steps) vs CPU oracle: {err}")
            except Exception as e:  # noqa: BLE001
                e2e_synth["parity_slice"] = {"error": f"{type(e).__name__}: {e}"}

    # ---- parameter sweep over SHARED data (BASELINE configs[3] shape on one GPU), end to end from host buffers ----
    def sweep_leg():
        C_ = 64
        E = max(2, min(args.e2e_steps, K))
        cmap = (np.arange(N) % C_).astype(np.int32)
        g = np.repeat(np.exp(np.linspace(np.log(1 / 3), np.log(3.0), N // C_)), C_)
        hs = [{k: torch.empty(v[..., :C_].shape, dtype=v.dtype, pin_memory=True).copy_(v[..., :C_]) for k, v in wl.chunks[c].items()} for c in range(2)]
        torch.cuda.synchronize()
        hsn = [{k: v.numpy() for k, v in h.items()} for h in hs]
        r_lego = np.ascontiguousarray(np.tile(p["r_vxyz"] ** 2 * g, (3, 1)))
        with RBISBatch(N, device=local, launch_groups=args.launch_groups) as bw:
            bw.set_process_noise(np.ascontiguousarray(p["q_gyro"] * g), np.ascontiguousarray(p["q_accel"] * g[::-1]),
                                 np.full(N, p["q_gyro_bias"]), np.full(N, p["q_accel_bias"]))
            bw.set_state(wl.vec0, wl.quat0, wl.cov0)
            for w_ in (-1, 0, 1):
                bw.set_column_map(w_, cmap, C_)
            res_s = torch.empty((n_local, capi.NUM_STATS), dtype=torch.float64, pin_memory=True).numpy()
            sp = [bw.prepare_fused(wl.progs[c], imu=hsn[c]["imu"],
                                   streams=[MeasStream(synth.LEGODO_IDX, hsn[c]["legodo"], r_lego, per_filter_diag=True),
                                            MeasStream(synth.POSE_IDX, hsn[c]["pose_z"], R_pose, quat=hsn[c]["pose_q"])]) for c in range(2)]
            sw = torch.cuda.ExternalStream(bw.cuda_stream, device=dev)
            bw.run_prepared(sp[0]); bw.run_prepared(sp[1])
            bw.synchronize()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record(sw)
            for i in range(E):
                bw.run_prepared(sp[i % 2])
            bw.stats_enqueue(tv, tq, res_s, chunk=CHUNK)
            bw.wait(bw.record())
            s1.record(sw)
            bw.synchronize()
            torch.cuda.synchronize()
            ms = s0.elapsed_time(s1)
        return {"value": N * Tc * E / (ms * 1e-3), "unit": UNIT, "steps": E, "ms_per_step": ms / E, "parameter_points": N // C_, "shared_columns": C_,
                "h2d_bytes_per_step": sum(int(v.nbytes) for v in hsn[0].values()) + wl.progs[0].nbytes, "d2h_bytes_total": int(res_s.nbytes),
                "non_finite": float(res_s[:, 45].sum()),
                "what": "end to end from pinned host buffers, per-filter process noise and leg-odometry R, 64 shared input columns", "this_rank_only": True}

    leg("sweep_shared_inputs", sweep_leg, when=not args.no_e2e and N % 64 == 0 and world == 1)

    b.close()
    del preps, wl
    gc.collect()
    torch.cuda.empty_cache()

    # ---- strong scaling: TOTAL_FILTERS filters in total, contiguous shards (SURVEY.md 8e, BASELINE configs[2]) ----
    def strong_leg():
        """65,536 filters in total, split over the ranks.  Two runs: inputs resident in HBM (per-rank random rows), and the Monte-Carlo
        form with counter-based inputs (initial ensemble and rows are functions of the GLOBAL filter index), whose reduced statistics
        must hash the same for every GPU count -- and hence for every kernel mapping the shard sizes select."""
        s_lo, s_hi = shard_range(TOTAL_FILTERS, rank, world, CHUNK)
        n = s_hi - s_lo
        n_l = (W + K) * L
        out = {"unit": UNIT, "scaling": "strong", "total_filters": TOTAL_FILTERS, "filters_per_gpu": n, "n_gpus": world}
        truth_s = synth.truth_trajectory(n_l * Tc)
        t_v, t_q = synth.truth_state_at(truth_s, n_l * Tc - 1)
        if world > 1:
            ws = Workload(n, Tc, n_l, dev, 0x5EED + rank, R_lego, R_pose)
            with new_batch(n) as bs:
                bs.set_state(ws.vec0, ws.quat0, ws.cov0)
                ps = ws.prepare(bs)
                ss = torch.cuda.ExternalStream(bs.cuda_stream, device=dev)
                timed_launches(bs, ps, ss, 0, W * L)
                bs.stats_allreduce(comm, t_v, t_q, s_lo // CHUNK, TOTAL_FILTERS // CHUNK, chunk=CHUNK)
                barrier()
                bs.synchronize()
                a0, a1 = timed_launches(bs, ps, ss, W * L, K * L)
                tot, _ = bs.stats_allreduce(comm, t_v, t_q, s_lo // CHUNK, TOTAL_FILTERS // CHUNK, chunk=CHUNK)
                fin = torch.cuda.Event(enable_timing=True)
                fin.record(ss)
                barrier()
                bs.synchronize()
                ms = max_over_ranks(a0.elapsed_time(fin))
                v = bs.last_kernel_variant
                k_ms_s = a0.elapsed_time(a1) / (K * L)
            sm = summarize(tot)
            out.update({"value": TOTAL_FILTERS * Tc * K * L / (ms * 1e-3), "ms_per_step": ms / K, "kernel_ms": k_ms_s, "kernel_variant": variant_name(v),
                        "stats_sha256_16": hashlib.sha256(np.ascontiguousarray(tot).tobytes()).hexdigest()[:16],
                        "filters": sm["filters"], "non_finite": sm["non_finite"], "mean_nees9": sm["mean_nees"]})
            del ws
        # ---- counter-based ensemble through rbis_batch_run_fused_synth ----
        SEED = 0x57A0E5CA1E
        tv0 = np.zeros(21)
        tv0[9:12] = (0, 0, 0.85); tv0[15:18] = synth.NOMINAL["bg"]; tv0[18:21] = synth.NOMINAL["ba"]
        v0, q0, c0 = synth.initial_ensemble(n, tv0, truth_s["quat"][0], filters=np.arange(s_lo, s_hi), seed=SEED)
        specs = []
        for c in range(n_l):
            d = synth.synth_spec_inputs(truth_s, c * Tc, Tc)
            specs.append(SynthSpec(SEED, d["imu_mean"], d["imu_step"], d["streams"], mode=1, first_filter=s_lo))
        progs_s = [make_ops(chunk_events(Tc, c * Tc)[0]) for c in range(n_l)]
        sst = [MeasStream(synth.LEGODO_IDX, None, R_lego), MeasStream(synth.POSE_IDX, None, R_pose, quat=True)]
        with new_batch(n) as bs:
            bs.set_state(v0, q0, c0)
            ss = torch.cuda.ExternalStream(bs.cuda_stream, device=dev)
            for c in range(W * L):
                bs.run_fused_synth(progs_s[c], sst, specs[c])
            bs.stats_allreduce(comm, t_v, t_q, s_lo // CHUNK, TOTAL_FILTERS // CHUNK, chunk=CHUNK)
            barrier()
            bs.synchronize()
            a0 = torch.cuda.Event(enable_timing=True); fin = torch.cuda.Event(enable_timing=True)
            bs.record(); a0.record(ss)
            for c in range(W * L, n_l):
                bs.run_fused_synth(progs_s[c], sst, specs[c])
            tot, _ = bs.stats_allreduce(comm, t_v, t_q, s_lo // CHUNK, TOTAL_FILTERS // CHUNK, chunk=CHUNK)
            fin.record(ss)
            barrier()
            bs.synchronize()
            ms = max_over_ranks(a0.elapsed_time(fin))
            v = bs.last_kernel_variant
        sm = summarize(tot)
        out["counter_based_inputs"] = {
            "value": TOTAL_FILTERS * Tc * K * L / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / K, "kernel_variant": variant_name(v),
            "stats_sha256_16": hashlib.sha256(np.ascontiguousarray(tot).tobytes()).hexdigest()[:16],
            "filters": sm["filters"], "non_finite": sm["non_finite"], "mean_nees9": sm["mean_nees"], "nees_in_95pct": sm["nees_in_95pct"],
            "what": "the same 65,536-filter Monte-Carlo ensemble for every GPU count: initial states and sensor rows are functions of the GLOBAL filter "
                    "index (rbis_batch_run_fused_synth, rows drawn in the kernel); the SHA-256 of the reduced statistics must not depend on n_gpus"}
        return out

    leg("strong_scaling", strong_leg, when=not strong)

    # ---- configs[1]: 4,096 filters, IMU-only propagation, one GPU ----
    def config1_leg():
        n, n_l = 4096, (W + K) * L
        w1_ = Workload(n, Tc, n_l, dev, 0xC0FF1, R_lego, R_pose, imu_only=True)
        with new_batch(n) as b1:
            b1.set_state(w1_.vec0, w1_.quat0, w1_.cov0)
            p1 = w1_.prepare(b1)
            s1_ = torch.cuda.ExternalStream(b1.cuda_stream, device=dev)
            timed_launches(b1, p1, s1_, 0, W * L)
            b1.synchronize()
            a0, a1 = timed_launches(b1, p1, s1_, W * L, K * L)
            b1.synchronize()
            torch.cuda.synchronize()
            ms = a0.elapsed_time(a1) / (K * L)
            v = b1.last_kernel_variant
            gv = b1.get_state(cov=False)[0]
        prof, why = kernel_profile(f"{v}:imu_only")
        rate = n * Tc / (ms * 1e-3)
        out = {"value": rate, "unit": UNIT, "filters": n, "workload": "configs[1]: 4,096-filter ensemble, IMU-only propagation (insUpdateState / insUpdateCovariance), 1 B200",
               "kernel_ms": ms, "steps_per_launch": Tc, "launches": K * L, "kernel_variant": variant_name(v), "finite": bool(np.isfinite(gv).all()),
               "roofline": {"bound": "fp64", "peak": dfma_tf, "unit": "TFLOP/s", "algorithmic_flops_per_filter_step": F_PROP,
                            "achieved_algorithmic": rate * F_PROP / 1e12, "frac_algorithmic": rate * F_PROP / 1e12 / dfma_tf}}
        if prof:
            ex = 2 * prof["dfma"] + prof["dmul"] + prof["dadd"]
            out["roofline"].update({"achieved": rate * ex / 1e12, "frac": rate * ex / 1e12 / dfma_tf, "executed_flops_per_filter_step": ex,
                                    "executed_source": prof.get("source")})
        else:
            out["roofline"].update({"achieved": None, "frac": None, "executed_unavailable": why})
        return out

    leg("config1_imu_only_4096", config1_leg, when=world == 1)

    # ---- configs[4]: pose fixes delivered 50 steps late -- per-filter history rewind + re-propagation inside the fused program ----
    def config5_leg():
        from pronto_b200.schedule import program_from_arrivals

        n, LAT, CH = N if not strong else TOTAL_FILTERS, 50, 6
        gen = torch.Generator(device=dev); gen.manual_seed(1)
        truth = synth.truth_trajectory(CH * Tc)
        v0, q0, c0 = initial_state(n, gen, dev)
        chs = [device_chunk(truth, c * Tc, Tc, n, gen, dev) for c in range(CH)]
        cat = {k: torch.cat([c[k] for c in chs]).contiguous() for k in chs[0]}
        del chs
        ev, li, pi = [], 0, 0
        for k in range(CH * Tc):
            ut = (k + 1) * 1000
            ev.append((capi.OP_IMU, 0, k, ut, 1e-3))
            if k % 2 == 0:
                ev.append((capi.OP_MEAS, 0, li, ut, 0.0)); li += 1
            if k % 100 == 0:
                ev.append((capi.OP_MEAS, 1, pi, ut, 0.0)); pi += 1
        pose = [e for e in ev if e[0] == 1 and e[1] == 1]
        arr, pend = [], list(pose)
        for e in ev:
            if e[0] == 1 and e[1] == 1:
                continue
            arr.append(e)
            while pend and e[0] == 0 and e[3] >= pend[0][3] + LAT * 1000:
                arr.append(pend.pop(0))
        arr += pend
        out = {}
        for label, arrivals in (("in_order", ev), ("late", arr)):
            ops, cnt = program_from_arrivals(arrivals, snapshot_slots=3, snapshot_period_us=100_000, snapshot_phase_us=1000)
            with new_batch(n, snapshot_slots=3) as b5:
                sts = [MeasStream(synth.LEGODO_IDX, cat["legodo"], R_lego), MeasStream(synth.POSE_IDX, cat["pose_z"], R_pose, quat=cat["pose_q"])]
                pp = b5.prepare_fused(ops, imu=cat["imu"], streams=sts)
                s5 = torch.cuda.ExternalStream(b5.cuda_stream, device=dev)
                best = 1e30
                for rep in range(3):
                    b5.set_state(v0, q0, c0)
                    b5.synchronize()
                    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a0.record(s5)
                    b5.run_prepared(pp)
                    b5.record()
                    a1.record(s5)
                    b5.synchronize()
                    torch.cuda.synchronize()
                    best = min(best, a0.elapsed_time(a1))
                n_applied = int(np.sum((ops["kind"] == capi.OP_IMU) | (ops["kind"] == capi.OP_MEAS)))
                out[label] = {"ms": best, "value": n * CH * Tc / (best * 1e-3), "ops": int(len(ops)), "updates_applied": n_applied,
                              "planner": cnt, "kernel_variant": variant_name(b5.last_kernel_variant)}
        rate = out["late"]["value"]
        return {"value": rate, "unit": UNIT, "workload": f"configs[4]: {n} filters, pose fixes delivered {LAT} steps late (rewind to the fix's utime + replay of "
                f"{LAT} IMU + {LAT // 2} leg-odometry updates per fix), {CH * Tc} trajectory steps in ONE rbis_batch_run_fused call; replayed steps are not counted as filter-steps",
                "in_order_value": out["in_order"]["value"], "detail": out, "this_rank_only": True,
                "roofline": {"bound": "fp64", "peak": dfma_tf, "unit": "TFLOP/s", "algorithmic_flops_per_filter_step": F_CFG5,
                             "achieved_algorithmic": rate * F_CFG5 / 1e12, "frac_algorithmic": rate * F_CFG5 / 1e12 / dfma_tf,
                             "note": "executed flops per TRAJECTORY step = (updates_applied late / in order) x the headline kernel's"}}

    leg("config5_delayed_50ms", config5_leg, when=world == 1)

    # ---- configs[3]: 1,048,576-filter noise-parameter sweep sharded over the GPUs, NCCL all-reduce of the statistics ----
    def config4_leg():
        G1, G2, G3 = 128, 128, 64
        NT = G1 * G2 * G3
        n = NT // world
        c_lo = rank * n
        Kc, C_ = 10, 1
        idx = np.arange(c_lo, c_lo + n)
        ax = lambda m: np.exp(np.linspace(np.log(1 / 3), np.log(3.0), m))
        q_gyro = p["q_gyro"] * ax(G1)[idx // (G2 * G3)]
        q_accel = p["q_accel"] * ax(G2)[(idx // G3) % G2]
        r_v = np.ascontiguousarray(np.tile((p["r_vxyz"] ** 2) * ax(G3)[idx % G3], (3, 1)))
        gen = torch.Generator(device=dev); gen.manual_seed(7)  # same seed on every rank: the shared log
        truth = synth.truth_trajectory((Kc + 2) * Tc)
        v0, q0, c0 = initial_state(C_, gen, dev)
        v0, q0, c0 = (t.expand(-1, n).contiguous() for t in (v0, q0, c0))
        host, progs = [], []
        for c in range(Kc + 2):
            ch = device_chunk(truth, c * Tc, Tc, C_, gen, dev)
            host.append({k: torch.empty(v.shape, dtype=v.dtype, pin_memory=True).copy_(v).numpy() for k, v in ch.items()})
            progs.append(make_ops(chunk_events(Tc, c * Tc)[0]))
        torch.cuda.synchronize()
        t_v, t_q = synth.truth_state_at(truth, (Kc + 2) * Tc - 1)
        with RBISBatch(n, device=local, launch_groups=args.launch_groups) as b4:
            b4.set_process_noise(np.ascontiguousarray(q_gyro), np.ascontiguousarray(q_accel), np.full(n, p["q_gyro_bias"]), np.full(n, p["q_accel_bias"]))
            b4.set_state(v0, q0, c0)
            cmap = np.zeros(n, dtype=np.int32)
            for w_ in (-1, 0, 1):
                b4.set_column_map(w_, cmap, C_)
            pr = [b4.prepare_fused(progs[c], imu=host[c]["imu"], streams=[MeasStream(synth.LEGODO_IDX, host[c]["legodo"], r_v, per_filter_diag=True),
                                                                            MeasStream(synth.POSE_IDX, host[c]["pose_z"], R_pose, quat=host[c]["pose_q"])])
                  for c in range(Kc + 2)]
            s4 = torch.cuda.ExternalStream(b4.cuda_stream, device=dev)
            b4.run_prepared(pr[0]); b4.run_prepared(pr[1])
            b4.stats_allreduce(comm, t_v, t_q, c_lo // CHUNK, NT // CHUNK, chunk=CHUNK)
            barrier()
            b4.synchronize()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record(s4)
            for c in range(2, Kc + 2):
                b4.run_prepared(pr[c])
            tot, _ = b4.stats_allreduce(comm, t_v, t_q, c_lo // CHUNK, NT // CHUNK, chunk=CHUNK)
            a1.record(s4)
            barrier()
            b4.synchronize()
            ms = max_over_ranks(a0.elapsed_time(a1))
            v = b4.last_kernel_variant
        sm = summarize(tot)
        rate = NT * Kc * Tc / (ms * 1e-3)
        return {"value": rate, "unit": UNIT, "workload": f"configs[3]: {NT}-filter Monte-Carlo noise-parameter sweep ({G1} x {G2} x {G3} grid of q_gyro, q_accel, leg-odometry R; "
                f"every grid point replays one shared log), {n} filters per GPU on {world} GPUs, inputs from pinned host buffers, NCCL all-reduce of the statistics inside the timed region",
                "launches": Kc, "steps_per_launch": Tc, "ms_total": ms, "kernel_variant": variant_name(v), "filters": sm["filters"], "non_finite": sm["non_finite"],
                "mean_nees9": sm["mean_nees"], "stats_sha256_16": hashlib.sha256(np.ascontiguousarray(tot).tobytes()).hexdigest()[:16],
                "roofline": {"bound": "fp64", "peak": dfma_tf * world, "unit": "TFLOP/s", "algorithmic_flops_per_filter_step": F_CFG3,
                             "achieved_algorithmic": rate * F_CFG3 / 1e12, "frac_algorithmic": rate * F_CFG3 / 1e12 / (dfma_tf * world)}}

    leg("config4_sweep_1M", config4_leg, when=world in (4, 8))

    # ---- the "next" rows of SURVEY.md 8f on this GPU (rank 0, N=1 only) ----
    def next_rows_leg():
        from pronto_b200 import smoother

        out = {}
        hbm_peak, hbm_src = 6544.7, "fallback: copy bandwidth of this pool's MEASURED_PEAKS.json at the time of writing"
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                hbm_peak, hbm_src = float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
        except Exception:
            pass
        n = 65_536
        gen = torch.Generator(device=dev); gen.manual_seed(3)
        truth = synth.truth_trajectory(Tc)
        ch = device_chunk(truth, 0, Tc, n, gen, dev)
        v0, q0, c0 = initial_state(n, gen, dev)
        with new_batch(n) as bn:
            sn = torch.cuda.ExternalStream(bn.cuda_stream, device=dev)
            buf = ch["imu"].clone()
            bn.notch_configure(85.0, 1000.0, 3)
            bn.notch_filter(buf)
            bn.synchronize()
            n0, n1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n0.record(sn)
            for _ in range(10):
                bn.notch_filter(buf)
            n1.record(sn)
            bn.synchronize()
            torch.cuda.synchronize()
            n_ms = n0.elapsed_time(n1) / 10
        n_bytes = Tc * 3 * n * 8 * 2
        out["notch_cascade"] = {"kernel": "notch_kernel", "ms_per_call": n_ms, "rows": Tc, "columns": n,
                                "roofline": {"bound": "hbm", "achieved": n_bytes / (n_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                             "frac": n_bytes / (n_ms * 1e-3) / 1e9 / hbm_peak, "peak_source": hbm_src,
                                             "algorithmic_bytes": "24 B read + 24 B written per row and column (3 accelerometer channels)"},
                                "value": Tc * n / (n_ms * 1e-3), "unit": "column-samples/s"}
        del buf
        Ns, Ts = 4096, 100
        ev_s, _, _ = chunk_events(Ts, 0)
        ops_s, is_ins, slot = smoother.forward_program(ev_s)
        sub = lambda t, rows: t[:rows, ..., :Ns].contiguous()
        n_lego_s, n_pose_s = sum(1 for e in ev_s if e[0] == 1 and e[1] == 0), sum(1 for e in ev_s if e[0] == 1 and e[1] == 1)
        with new_batch(Ns, snapshot_slots=len(is_ins)) as bs:
            st_s = [MeasStream(synth.LEGODO_IDX, sub(ch["legodo"], n_lego_s), R_lego),
                    MeasStream(synth.POSE_IDX, sub(ch["pose_z"], n_pose_s), R_pose, quat=sub(ch["pose_q"], n_pose_s))]
            imu_s = sub(ch["imu"], Ts)
            np_slot, n_slot, steps_s, alias = smoother.plan(is_ins, slot)
            best_f, best_b = 1e30, 1e30
            for rep in range(2):
                bs.set_state(v0[:, :Ns].contiguous(), q0[:, :Ns].contiguous(), c0[:, :Ns].contiguous())
                bs.synchronize()
                t0 = time.perf_counter()
                bs.run_fused(ops_s, imu=imu_s, streams=st_s)
                bs.synchronize()
                t1 = time.perf_counter()
                bs.smooth_backward(np_slot, n_slot, steps_s, 1e-3)
                bs.synchronize()
                t2 = time.perf_counter()
                best_f, best_b = min(best_f, t1 - t0), min(best_b, t2 - t1)
        out["ekf_smoother"] = {"kernel": "rbis_smooth_kernel", "filters": Ns, "smoothing_steps": int(len(steps_s)), "backward_ms": best_b * 1e3,
                               "value": Ns * len(steps_s) / best_b, "unit": "smoothing steps/s", "forward_with_snapshots_ms": best_f * 1e3,
                               "timing": "host wall clock around synchronised calls"}
        return out

    leg("next_rows", next_rows_leg, when=rank == 0 and world == 1 and not args.no_e2e)

    # ---- CPU baseline (rank 0, N=1 only) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        rate, times, _ = cpu_oracle_rate(args.cpu_sample_steps, REF_FILTERS, threads)
        rate1, t1 = cpu_config1_rate()
        cpu = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port", "per_thread_value": rate / threads,
               "sample": f"{REF_FILTERS} filters x {args.cpu_sample_steps} steps of the same schedule, {threads} threads, {times[0]:.2f} s wall",
               "config1_single_filter": {"value": rate1, "unit": UNIT, "cores": 1, "seconds": t1,
                                         "what": "BASELINE.md 3: ONE filter, 60,000 IMU steps (60 s at 1 kHz) + 30,000 leg-odometry updates through the reference's "
                                                 "time-ordered multimap history, one thread -- the reference's actual execution model"},
               "note": "Eigen-free C++ restatement of the reference (g++ -O3, no fast-math); the reference itself cannot be built here"}

    if rank == 0:
        flops_chunk = flops_per_chunk(Tc, Tc // 2, Tc // 100) * N
        alg = flops_chunk / (k_ms * 1e-3) / 1e12
        prof, why = kernel_profile(variant)
        roof = {"bound": "fp64", "peak": dfma_tf, "unit": "TFLOP/s", "kernel": "rbis_fused_kernel" if not (variant >> 4) else "rbis_group_kernel", "kernel_ms": k_ms,
                "kernel_ms_how": "CUDA events on the library stream around the K x L back-to-back fused launches (the stream joins the launch-group streams before "
                                 "the closing event), divided by their number: launches overlap by design (launch groups), so a per-launch event pair would not bracket one launch",
                "algorithmic_flops_per_filter_step": flops_chunk / (N * Tc), "achieved_algorithmic": alg, "frac_algorithmic": alg / dfma_tf,
                "peak_source": "DFMA microbenchmark in this run (MEASURED_PEAKS.json has no FP64 entry)", "nominal_peak": NOMINAL_FP64_TFLOPS,
                "dmma_peak_measured": dmma_tf, "hbm_stream_gbs": BYTES_PER_STEP * N * Tc / (k_ms * 1e-3) / 1e9,
                "traffic_unit": "bytes per launch (ncu dram read+write)",
                "note": "achieved / frac count the FP64 flops the kernel EXECUTES (ncu instruction counts: 2 x DFMA + DMUL + DADD per filter-step); the kernel skips the "
                        "structural zeros of Ad, uses the symmetry of P and (decoupled variant) drops the exactly-zero omega / a couplings, so the dense algorithmic "
                        "count of SURVEY.md 8d (achieved_algorithmic / frac_algorithmic) is ~16x larger and not a utilisation figure"}
        if prof:
            ex = 2 * prof["dfma"] + prof["dmul"] + prof["dadd"]
            sm_clk = (clocks.get("sm_mhz") or 1965.0) * 1e6
            n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
            roof.update({"achieved": ex * N * Tc / (k_ms * 1e-3) / 1e12, "frac": ex * N * Tc / (k_ms * 1e-3) / 1e12 / dfma_tf,
                         "executed_flops_per_filter_step": ex, "executed_source": prof.get("source"),
                         "fp64_pipe_busy_frac": (prof["dfma"] + prof["dmul"] + prof["dadd"]) * 2 * N * Tc / 32 / (k_ms * 1e-3) / (n_sm * 4 * sm_clk),
                         "traffic": prof.get("dram_bytes") if (prof.get("filters"), prof.get("chunk_steps")) == (N, Tc) else None})
        else:
            roof.update({"achieved": None, "frac": None, "traffic": None, "executed_unavailable": why})
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": ("configs[2]: 65,536-filter ensemble per GPU" if not strong else f"configs[2]: {n_total}-filter ensemble split over {world} GPU(s)")
                                   + ", IMU 1 kHz + leg-odometry 500 Hz (m=3) + pose fix 10 Hz (m=6), fused kernel",
                       "filters_per_gpu": N, "total_filters": n_total, "chunk_steps": Tc, "launches_per_step": L, "filter_steps_per_step": n_total * Tc * L,
                       "kernel_variant": variant_name(variant), "kernel_source_sha": kernel_source_sha(),
                       "host_enqueue_ms_per_call": enqueue_ms,
                       "l2_policy": f"every launch reads a fresh {BYTES_PER_STEP * N * Tc / 1e6:.0f} MB input chunk (L2 is 126 MB); {resident} of {n_launches} chunks resident in HBM"
                                    + ("" if resident == n_launches else " (cycled)"),
                       "stats_allreduce": ("rbis_batch_stats_allreduce over ncclComm_t, inside the timed region" if world > 1 else "single GPU, inside the timed region")},
            "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "e2e_f32_rows": e2e_f32, "e2e_synth": e2e_synth, "gpu_launches": launches, "clocks": clocks,
            "ensemble": {"mean_nees9": summ["mean_nees"], "nees_in_95pct": summ["nees_in_95pct"], "non_finite": summ["non_finite"], "stats_sha256_16": stats_sha},
        }
        line.update(legs)
        emit(line)
    if comm is not None:
        comm.close()
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line goes to the process's real stdout; everything else that lands on fd 1 (NCCL prints its
    version banner there, torchrun its OMP note) was redirected to stderr by main()."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    args = parse()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
