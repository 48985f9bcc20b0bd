#!/usr/bin/env python
"""bench.py - ICP iterations/s (whole-job) and Mpoints/s of the J^T J / J^T r reduction on B200.

Contract (see the task statement): `python bench.py --gpus N --steps K --warmup W [--impl reference]`
prints ONE JSON line on rank 0.  A "step" is one full registration of the C2 workload (synthetic
100k-point cylinder pair, 50 fixed ICP iterations: correspondences + K1 + K2 every iteration).

  value      ICP iterations/s, source + target resident in HBM when the timed region starts
  e2e        same metric through the public C-ABI call with HOST buffers: every step uploads the
             scan from pinned host memory and reads back pose + per-iteration log
  roofline   K1 (fused residual/weight/Jacobian/27-sum reduction) at C4 size (10M slots, frozen
             float4 planes, 32 B/slot), CUDA-event timed on the launching stream, vs MEASURED_PEAKS
  cpu_baseline  the CPU oracle (port of the reference loop) timed on this box's host cores on a
             bounded sample of the same workload
N > 1: replicas (one independent scan pair per GPU, no data-path collective, "weak"); the sharded
10M-slot reduction with its 32-double ncclAllReduce is reported under "sharded".
`--impl reference` times the reference's own CPU algorithm (oracle port; the reference binary cannot
be built here: Eigen/PCL/yaml-cpp absent and its "Ours" stage is a stub) on the same config.
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

C2_POINTS = 100_000
C2_ITERS = 50
C4_SLOTS = 10_000_000
C4_RADIUS = 0.05
C4_ICP_ITERS = 10                # fixed iterations of the sharded 10 M-point corridor registration
C5_TRIALS = 5000                 # perturbation Monte-Carlo (BASELINE.json configs[4]), split over the ranks
ALG_BYTES_PER_SLOT = 32          # float4 point + float4 plane (SURVEY.md §8d)
K1_NCU_TRAFFIC_BYTES = 320.07e6 + 3.54e6   # dram read + write of one 10 M-slot K1 launch (ncu --set full, profiles/k1_r2_ncu_summary.txt)


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.path = tempfile.mktemp(suffix=".csv")
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.index)],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None
        atexit.register(self.stop)                         # a run that fails mid-way must not leave nvidia-smi polling

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.proc = None
        sm, mx, reasons = [], [], set()
        try:
            for ln in open(self.path):
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), samples=len(sm))
        out["reasons"] = sorted(reasons)
        return out


def c2_params(default_params):
    # "Ours" = [SCHUR_CONDITION_NUMBER, PRECONDITIONED_CG] (icp_pk01.yaml:106), kappa_th = kappa_tg = 10 (icp.yaml),
    # USE_WEIGHT_DERIVATIVE = false (the released default, icp_test_runner.cpp:1691; with the derivative term the
    # Gauss-Newton iteration DIVERGES on this 100k scene - checked with the CPU oracle - so it is not a sane
    # benchmark workload), init = the published cylinder perturbation, 50 fixed iterations (BASELINE.json configs[1])
    return default_params(search_radius=1.0, max_iterations=C2_ITERS, fixed_iterations=1, kappa_target=10.0,
                          cond_thresh=10.0, use_weight_derivative=0, detection="SCHUR_CONDITION_NUMBER",
                          handling="PRECONDITIONED_CG")


def result_arrays(prefix, r):
    """What one ICP call handed back (an IcpResult) as arrays named <prefix>_<what>: the pose, iteration count and
    flags, and every per-iteration log field stacked over the iterations.  The log's wall-clock iter_time_ms and the
    reserved padding are left out: they are not results and would differ between identical runs."""
    from dcreg_b200.api import Analysis, IterLog
    out = {f"{prefix}_pose": r.T, f"{prefix}_iterations": r.iterations, f"{prefix}_converged": r.converged,
           f"{prefix}_status": r.status}
    for struct, part in ((IterLog, lambda L: L), (Analysis, lambda L: L.analysis)):
        for name, _ in struct._fields_:
            if r.logs and name not in ("analysis", "iter_time_ms", "reserved1"):
                out[f"{prefix}_log_{name}"] = [np.array(getattr(part(L), name)) for L in r.logs]
    return out


def write_outputs(directory, arrays):
    """--dump-outputs: DIR/<name>.npy, float64, one file per array."""
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), np.asarray(a, dtype=np.float64))


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port on host cores
# ------------------------------------------------------------------------------------------------
def workload_config(world):
    """The `config` object both arms print (the reference arm runs "your arm's config")."""
    return {"workload": f"C2 synthetic cylinder pair {C2_POINTS} pts x {C2_ITERS} fixed ICP iterations per step from the published "
                        "perturbation, method Ours (Schur detection + PCG), search_radius 1.0, weight derivative off (released default)",
            "parallelism": "replicas (one scan pair per GPU)" if world > 1 else "1 GPU",
            "l2": "K1 roofline inputs 320 MB > 126 MB L2; no flush needed",
            "roofline_workload": f"C4 synthetic corridor {C4_SLOTS} slots, frozen float4 planes"}


_BUDGET = None


def host_cpu_budget():
    """CPUs this process may really use: the affinity mask, capped by the cgroup CPU quota when there is one.
    Returns (usable, affinity, quota or None).  Evaluated once, BEFORE libgomp exists in the process: with
    OMP_PROC_BIND set libgomp pins the initial thread to its first place and the mask would read 2."""
    global _BUDGET
    if _BUDGET is not None:
        return _BUDGET
    aff = len(os.sched_getaffinity(0))
    quota = None
    try:                                               # cgroup v2
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        pass
    if quota is None:
        try:                                           # cgroup v1
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0 and per > 0:
                quota = q / per
        except Exception:
            pass
    usable = aff if quota is None else max(1, min(aff, int(quota + 0.5)))
    _BUDGET = (usable, aff, quota)
    return _BUDGET


def pin_openmp_env(threads):
    """Explicit OpenMP settings for the CPU arm, BEFORE libgomp is loaded: torchrun exports OMP_NUM_THREADS=1, and an
    unset thread count makes libgomp spawn one spinning thread per visible CPU, which on a shared / quota-limited host
    ran the same code anywhere between 2 and 700 iterations/s (VERDICT round 1)."""
    os.environ["OMP_NUM_THREADS"] = str(threads)
    os.environ["OMP_DYNAMIC"] = "false"
    os.environ["OMP_PROC_BIND"] = "close"
    os.environ["OMP_PLACES"] = "cores"
    os.environ["OMP_WAIT_POLICY"] = "passive"          # a descheduled team member must not be spun on


class CpuArm:
    """The C/OpenMP oracle (CPU port of the reference loop; the reference binary cannot be built here: Eigen, PCL,
    yaml-cpp, Ceres, TBB, Open3D absent and its "Ours" stage is a stub) on the C2 workload.  A step is the SAME step
    the GPU arm runs: 50 fixed ICP iterations from the published perturbation; the kd-tree build is excluded as in
    the reference's own timing (icp_test_runner.cpp:408-461)."""

    def __init__(self, seed=42):
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        self.usable, self.aff, self.quota = host_cpu_budget()
        pin_openmp_env(self.usable)
        import dcreg_oracle_c as oc
        from dcreg_b200.scenes import make_cylinder, g2_initial_pose
        self.oc = oc
        self.T0 = g2_initial_pose()
        pts = make_cylinder(C2_POINTS, seed=seed)
        self.scene = oc.Scene(pts, pts)
        self.threads = None
        self.calibration = []

    def run(self, iters, threads, thread_mode=1):
        prm = self.oc.make_params(max_iterations=iters, fixed_iterations=True, kappa_target=10.0,
                                  use_weight_derivative=False, thread_mode=thread_mode, n_threads=threads)
        t0 = time.perf_counter()
        st, conv, n_it, T, _ = self.scene.icp_run(prm, self.T0, want_log=False)
        dt = time.perf_counter() - t0
        assert st == 0 and n_it == iters
        return dt, T

    def calibrate(self):
        """Pick the OpenMP team size that is actually fastest on this host (one short sample per candidate, after a
        cold-start sample): a visible-CPU count says nothing about SMT siblings, quotas or noisy neighbours."""
        cands = sorted({c for c in (4, 8, 16, 24, 32, 48, 64, 96, 128, self.usable // 2, self.usable) if 1 <= c <= self.usable})
        self.run(3, min(8, self.usable))                                   # first touch: page in the tree, spawn the pool
        best = None
        for c in cands:
            self.run(2, c)
            dt, _ = self.run(6, c)
            rate = 6 / dt
            self.calibration.append({"threads": c, "it_per_s": round(rate, 1)})
            if best is None or rate > best[1]:
                best = (c, rate)
        self.threads = best[0]
        return self.threads

    def steps(self, n_steps, warmup):
        for _ in range(max(1, warmup)):                                    # at least one full untimed step
            self.run(C2_ITERS, self.threads)
        times, T = [], None
        for _ in range(max(1, n_steps)):
            dt, T = self.run(C2_ITERS, self.threads)
            times.append(dt)
        return np.array(times), T

    def faithful(self, n_steps=3):
        """Reference-faithful threading: omp num_threads(8) on the correspondence loop only, serial Jacobian build and
        serial A^T A (icp_test_runner.cpp:1714, 1863-1915)."""
        th = min(8, self.usable)
        self.run(5, th, thread_mode=0)
        ts = [self.run(C2_ITERS, th, thread_mode=0)[0] for _ in range(n_steps)]
        return {"value": C2_ITERS / float(np.median(ts)), "cores": th, "sample": f"median of {n_steps} steps of {C2_ITERS} iterations",
                "note": "omp num_threads(8) on correspondences only, serial J build and A^T A (icp_test_runner.cpp:1714,1863-1915)"}

    def describe(self, times):
        med = float(np.median(times))
        return {"value": C2_ITERS / med, "unit": "ICP iterations/s", "cores": int(self.threads), "kind": "port",
                "sample": f"median of {len(times)} steps, each {C2_ITERS} fixed ICP iterations of the C2 workload from the initial pose "
                          "(the GPU arm's step; kd-tree build excluded as in the reference)",
                "step_s": {"median": med, "min": float(times.min()), "max": float(times.max()), "mean": float(times.mean())},
                "host": {"affinity_cpus": self.aff, "cgroup_quota_cpus": self.quota, "usable_cpus": self.usable,
                         "omp": {k: os.environ.get(k) for k in ("OMP_PROC_BIND", "OMP_PLACES", "OMP_WAIT_POLICY")}},
                "thread_calibration": self.calibration}


def cpu_worker(args):
    """`bench.py --cpu-worker`: everything the GPU arm wants from the host cores, in a CLEAN process (no torch, no CUDA
    threads, same OpenMP set-up as `--impl reference`): the C2 cpu_baseline with the oracle's final pose (parity of the
    benchmarked step), and for C5 the oracle's results of the first 16 trials plus an all-cores trials/s sample."""
    arm = CpuArm(seed=42)
    arm.calibrate()
    times, T_cpu = arm.steps(args.steps, 1)
    cpu = arm.describe(times)
    cpu["reference_faithful_8_threads"] = arm.faithful()
    from dcreg_b200.scenes import load_pcd_xyz, trial_poses
    cyl = load_pcd_xyz(os.path.join(ROOT, "tests", "golden", "cylinder_7562.pcd"))
    poses = trial_poses(C5_TRIALS, seed=45)
    sc = arm.oc.Scene(cyl, cyl)
    prm5 = arm.oc.make_params(max_iterations=30, kappa_target=10.0, n_threads=min(8, arm.usable))
    ref5 = []
    for k in range(16):
        st5, conv5, it5, T5, _ = sc.icp_run(prm5, poses[k], want_log=False)
        ref5.append({"status": int(st5), "converged": bool(conv5), "iterations": int(it5), "T": T5.reshape(-1).tolist()})
    c5_cpu = None
    if args.cpu_trials:
        # independent trials: one single-threaded oracle registration per worker thread, all usable CPUs busy.  The
        # workers drop the core binding the initial thread got from OMP_PROC_BIND.
        from concurrent.futures import ThreadPoolExecutor
        workers = int(arm.usable)
        everything = set(range(os.cpu_count() or 1))
        n5 = int(min(C5_TRIALS, max(4 * workers, 64)))
        prm51 = arm.oc.make_params(max_iterations=30, kappa_target=10.0, n_threads=1)
        scenes5 = [arm.oc.Scene(cyl, cyl) for _ in range(workers)]

        def one(k):
            try:
                os.sched_setaffinity(0, everything)
            except OSError:
                pass
            return scenes5[k % workers].icp_run(prm51, poses[k], want_log=False)[2]
        with ThreadPoolExecutor(workers) as ex:
            list(ex.map(one, range(workers)))                                # spin up
            t5 = time.perf_counter()
            list(ex.map(one, range(n5)))
            t5 = time.perf_counter() - t5
        pool_rate = n5 / t5
        # ... or one registration at a time with the OpenMP team inside it (the reference's own arrangement)
        prm5t = arm.oc.make_params(max_iterations=30, kappa_target=10.0, n_threads=arm.threads)
        sc.icp_run(prm5t, poses[0], want_log=False)
        n5s = 48
        t5s = time.perf_counter()
        for k in range(n5s):
            sc.icp_run(prm5t, poses[k], want_log=False)
        t5s = time.perf_counter() - t5s
        seq_rate = n5s / t5s
        c5_cpu = {"trials_per_s": max(pool_rate, seq_rate), "workers": workers,
                  "modes": {"one_single_threaded_registration_per_worker": pool_rate, "sequential_registrations_openmp_inside": seq_rate},
                  "sample": f"{n5} (pool) / {n5s} (sequential, {arm.threads} OpenMP threads) of the {C5_TRIALS} trials; the faster arrangement is quoted"}
    print(json.dumps({"cpu_baseline": cpu, "c2_pose": T_cpu.reshape(-1).tolist(), "c5_ref": ref5, "c5_cpu": c5_cpu}))


def run_reference(args, rank, world):
    """The reference's own CPU algorithm (oracle port) on the host cores; rank 0 only (the other ranks exit 0)."""
    if rank != 0:
        return
    arm = CpuArm(seed=42)
    arm.calibrate()
    times, T = arm.steps(args.steps, args.warmup)
    if args.dump_outputs:
        write_outputs(args.dump_outputs, {"c2_pose": T})
    cpu = arm.describe(times)
    cpu["reference_faithful_8_threads"] = arm.faithful()
    value = cpu["value"]
    line = {
        "impl": "reference", "metric": "icp_iterations_per_s", "value": value, "unit": "ICP iterations/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * cpu["step_s"]["median"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(world),
        "timing": "value = 50 iterations / MEDIAN step time (host CPUs are shared with other tenants; min/max/mean in cpu_baseline.step_s)",
        "cpu_baseline": cpu,
        "e2e": {"value": value, "unit": "ICP iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_ours(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    torch.set_num_threads(1)
    from dcreg_b200 import Context, default_params
    from dcreg_b200.scenes import make_cylinder, make_corridor, g2_initial_pose

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - dcreg_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    ctx = Context(local_rank)
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)

    # ---------------- C2: full ICP iterations/s (replicas at N > 1) ----------------
    pts = make_cylinder(C2_POINTS, seed=42 + rank)
    pinned = torch.from_numpy(pts).pin_memory()
    pts_pinned = pinned.numpy()
    T0 = g2_initial_pose()
    prm = c2_params(default_params)
    ctx.set_target(pts, 1.0)                 # cell = radius (measured fastest; finer grids are exact too but slower): index build: setup, outside the reference's timed region too
    ctx.set_source(pts_pinned)
    for _ in range(max(args.warmup, 3)):
        res = ctx.icp_run(prm, T0, want_log=False)
    assert res.iterations == C2_ITERS

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)                                   # let nvidia-smi finish starting up before anything is timed
    barrier()
    l0 = ctx.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        ctx.icp_enqueue(prm, T0)                         # inputs resident in HBM; the device never waits for the host:
    e1.record(stream)                                    # the K runs are queued back to back (dcreg_icp_enqueue)
    e1.synchronize()
    res = ctx.icp_fetch()
    assert res.iterations == C2_ITERS
    outputs = result_arrays("c2", res)
    barrier()
    dev_ms = max_over_ranks(e0.elapsed_time(e1))
    launches = ctx.launch_count - l0
    value = world * args.steps * C2_ITERS / (dev_ms * 1e-3)

    # how much correspondence work the loop reused in one step (untimed extra run, counters on)
    ctx.iteration_counters(True)
    ctx.icp_run(prm, T0, want_log=False)
    searched, fitted = ctx.iteration_counters(False)

    # e2e: host buffers in, pose + log out, every step
    ctx.set_source(pts_pinned)
    res = ctx.icp_run(prm, T0, want_log=True)            # untimed: this run shape's first use (graph capture)
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    step_wall = []
    w0 = time.perf_counter()
    e2.record(stream)
    for _ in range(args.steps):
        ws = time.perf_counter()
        ctx.set_source(pts_pinned)                        # H2D of this step's scan (pinned)
        res = ctx.icp_run(prm, T0, want_log=True)         # D2H of pose + per-iteration records
        step_wall.append(time.perf_counter() - ws)
    e3.record(stream)
    e3.synchronize()
    wall = time.perf_counter() - w0
    outputs.update(result_arrays("e2e", res))
    barrier()
    e2e_ms = max_over_ranks(max(e2.elapsed_time(e3), wall * 1e3))
    clocks = sampler.stop() if rank == 0 else None
    e2e_value = world * args.steps * C2_ITERS / (e2e_ms * 1e-3)
    from dcreg_b200.api import IterLog
    import ctypes
    h2d = int(pts.shape[0] * 3 * 4 + 16 * 8)
    d2h = int(ctypes.sizeof(IterLog) * C2_ITERS + 472)

    # ---------------- C4: K1 reduction roofline (sharded at N > 1) ----------------
    from dcreg_b200.parallel import init_sharded, shard_range
    n_total = C4_SLOTS
    scene = make_corridor(n_total, seed=44, noise=0.002)
    lo, hi = shard_range(n_total, rank, world)
    Tc = np.eye(4); Tc[:3, 3] = [0.004, 0.003, -0.002]
    ctx.set_target(scene, C4_RADIUS)
    ctx.set_source(scene[lo:hi])
    ctx.find_planes(Tc, C4_RADIUS, want_planes=False)     # correspondences once; planes stay on the device
    ctx.freeze_planes_f32()
    if world > 1:
        init_sharded(ctx, dist, n_total, device=dev)      # NCCL comm inside the C library; id via torch.distributed
    else:
        ctx.set_global_source_count(n_total)
    out27, stats = ctx.reduce_device(False, Tc, False)    # warm-up + sanity
    for wd in (False, True):
        for f64 in (False, True):
            ctx.time_reduce(f64, Tc, wd, 3, False)
    barrier()
    reps = 20

    def k1_time(f64, wd):
        """median over 5 batches of `reps` back-to-back launches (CUDA events on the context's stream around each batch,
        max over ranks per batch): one batch right after an idle gap reads ~1 us high while the clocks ramp"""
        ts = [max_over_ranks(ctx.time_reduce(f64, Tc, wd, reps, False)) for _ in range(5)]
        return float(np.median(ts)), ts
    k1_ms, k1_batches = k1_time(False, False)                                   # inputs (320 MB) > L2 (126 MB)
    k1_ms_f64, _ = k1_time(True, False)
    k1_ms_wd, _ = k1_time(False, True)
    barrier()
    peak, peak_src = measured_peak_gbs()
    n_local = hi - lo
    achieved = ALG_BYTES_PER_SLOT * n_local / (k1_ms * 1e-3) / 1e9             # per GPU
    mpts = n_total / (k1_ms * 1e-3) / 1e6                                       # whole job

    # ---------------- C4 end to end: the point-sharded 10 M-point corridor REGISTRATION (row N1) ----------------
    # every rank holds a contiguous block of source slots and the whole target; one sum over ranks per iteration
    # (inside the iteration kernel over peer memory when dcreg_comm_mode == 2), the solve step redundantly everywhere
    prm4 = default_params(search_radius=C4_RADIUS, max_iterations=C4_ICP_ITERS, fixed_iterations=1, kappa_target=10.0)
    res4 = ctx.icp_run(prm4, Tc, want_log=True)                              # warm-up (allocations, graph capture)
    c4_runs = 3
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record(stream)
    for _ in range(c4_runs):
        res4 = ctx.icp_run(prm4, Tc, want_log=True)
    f1.record(stream)
    f1.synchronize()
    barrier()
    c4_ms = max_over_ranks(f0.elapsed_time(f1)) / c4_runs
    outputs.update(result_arrays("c4", res4))
    comm_mode = ctx.comm_mode
    sharded_ok, sharded_dT = None, None
    ctx2 = Context(local_rank)                                               # plain context: no communicator
    if world > 1:
        # parity of the sharded run, on every rank: the same registration unsharded on this GPU alone
        ctx2.set_target(scene, C4_RADIUS)
        ctx2.set_source(scene)
        ref4 = ctx2.icp_run(prm4, Tc, want_log=True)
        sharded_dT = float(np.abs(res4.T - ref4.T).max())
        ok = (res4.iterations == ref4.iterations and sharded_dT < 1e-9 and
              all(a.n_effective == b.n_effective and a.n_corr_pt == b.n_corr_pt and abs(a.fitness - b.fitness) < 1e-12
                  for a, b in zip(res4.logs, ref4.logs)))
        t_ok = torch.tensor([1.0 if ok else 0.0], dtype=torch.float64, device=dev)
        t_dT = torch.tensor([sharded_dT], dtype=torch.float64, device=dev)
        dist.all_reduce(t_ok, op=dist.ReduceOp.MIN)
        dist.all_reduce(t_dT, op=dist.ReduceOp.MAX)
        # all ranks must hold the same pose bit for bit (the sums are formed in rank order everywhere)
        t_pose = torch.from_numpy(res4.T.copy()).to(dev)
        t_lo, t_hi = t_pose.clone(), t_pose.clone()
        dist.all_reduce(t_lo, op=dist.ReduceOp.MIN); dist.all_reduce(t_hi, op=dist.ReduceOp.MAX)
        same_bits = bool(torch.equal(t_lo, t_hi))
        sharded_ok, sharded_dT = bool(t_ok.item() == 1.0) and (same_bits or comm_mode != 2), float(t_dT.item())
        if not sharded_ok:
            raise SystemExit(f"bench.py: sharded C4 registration does not match the single-GPU run (max |dT| {sharded_dT:.3e}, "
                             f"identical over ranks: {same_bits})")
    c4 = {"it_per_s": C4_ICP_ITERS / (c4_ms * 1e-3), "ms_per_iteration": c4_ms / C4_ICP_ITERS, "points": n_total,
          "iterations_per_run": C4_ICP_ITERS, "runs_timed": c4_runs, "scaling": "strong",
          "n_effective_last": int(res4.logs[-1].n_effective),
          "collective": {0: None, 1: "ncclAllReduce of 32 doubles behind the iteration kernel + separate solve kernel (fallback)",
                         2: "in-kernel: peer-memory mailboxes over NVLink in the iteration kernel's last block, solve step folded in"}[comm_mode],
          "parity_vs_single_gpu": None if world == 1 else {"ok": sharded_ok, "max_abs_dT": sharded_dT,
                                                           "what": "same 10 M-point registration unsharded on every rank: iteration counts, N_eff, N_pt, fitness identical, |dT| < 1e-9, pose bit-identical across ranks"}}

    # ---------------- C5: perturbation Monte-Carlo, trials batched and split over the ranks (row N2) ----------------
    from dcreg_b200.scenes import load_pcd_xyz, trial_poses
    cyl = load_pcd_xyz(os.path.join(ROOT, "tests", "golden", "cylinder_7562.pcd"))     # the reference's shipped cloud
    poses = trial_poses(C5_TRIALS, seed=45)
    tlo, thi = shard_range(C5_TRIALS, rank, world)
    prm5 = default_params(kappa_target=10.0)                                  # icp.yaml defaults: radius 1.0, 30 iterations
    ctx2.set_target(cyl, 1.0)
    ctx2.set_source(cyl)
    ctx2.icp_run_batch(prm5, poses[tlo:thi])                                  # warm-up
    stream2 = torch.cuda.ExternalStream(ctx2.stream, device=dev)
    barrier()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w5 = time.perf_counter()
    g0.record(stream2)
    trials = ctx2.icp_run_batch(prm5, poses[tlo:thi])                         # H2D of the poses, D2H of the results inside
    g1.record(stream2)
    g1.synchronize()
    w5 = time.perf_counter() - w5
    barrier()
    c5_ms = max_over_ranks(max(g0.elapsed_time(g1), w5 * 1e3))
    per_trial = [result_arrays("c5", t) for t in trials]
    outputs.update({k: [p[k] for p in per_trial] for k in per_trial[0]})
    n_conv = torch.tensor([float(sum(t.converged for t in trials)), float(sum(t.iterations for t in trials))],
                          dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(n_conv)
    c5 = {"trials": C5_TRIALS, "trials_per_s": C5_TRIALS / (c5_ms * 1e-3), "ms": c5_ms, "scaling": "strong",
          "trials_per_gpu": thi - tlo, "converged": int(n_conv[0].item()), "mean_iterations": float(n_conv[1].item()) / C5_TRIALS,
          "workload": "shipped 7 562-point cylinder, t ~ U[-1,1]^3 m, rpy ~ U[-3,3]^3 deg (seed 45), icp.yaml defaults, method Ours; "
                      "one dcreg_icp_run_batch call per rank (host poses in, host results out)"}
    ctx2.close()

    # ---------------- parity of the benchmarked configuration + CPU baseline (rank 0) ----------------
    # the host side runs in a clean subprocess (see cpu_worker), after every GPU-timed region
    cpu, parity = None, None
    if rank == 0 and not args.no_cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import dcreg_oracle as onp                                           # se3 log distance (NumPy twin), checker only
        env = {k: v for k, v in os.environ.items() if not k.startswith("OMP_") and k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")}
        cmd = [sys.executable, os.path.abspath(__file__), "--cpu-worker", "--steps", "8" if world == 1 else "1"]
        if world == 1:
            cmd.append("--cpu-trials")
        out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
        if out.returncode != 0:
            raise SystemExit("bench.py: the CPU worker failed:\n" + out.stderr[-2000:])
        host = json.loads(out.stdout.strip().splitlines()[-1])
        pose_err = float(onp.se3_log_distance(np.array(host["c2_pose"]).reshape(4, 4), res.T))
        parity = {"parity_checked": True, "pose_err": pose_err, "tolerance": 1e-6,
                  "what": "|log(T_oracle^-1 T_gpu)| after the 50 fixed iterations of the timed C2 step, C/OpenMP oracle vs the e2e GPU result"}
        if not pose_err < 1e-6:
            raise SystemExit(f"bench.py: C2 parity FAILED, pose error {pose_err:.3e} vs the CPU oracle")
        worst5 = 0.0
        for k, r5 in enumerate(host["c5_ref"]):
            if r5["status"] != trials[k].status or r5["iterations"] != trials[k].iterations or r5["converged"] != trials[k].converged:
                raise SystemExit(f"bench.py: C5 trial {k} differs from the CPU oracle (status/iterations/converged)")
            worst5 = max(worst5, float(onp.se3_log_distance(np.array(r5["T"]).reshape(4, 4), trials[k].T)))
        if not worst5 < 1e-6:
            raise SystemExit(f"bench.py: C5 parity FAILED, pose error {worst5:.3e}")
        c5["parity"] = {"trials_checked": len(host["c5_ref"]), "max_pose_err": worst5, "tolerance": 1e-6}
        if world == 1:
            cpu = host["cpu_baseline"]
            c5["cpu_port"] = host["c5_cpu"]

    if rank == 0 and args.dump_outputs:
        write_outputs(args.dump_outputs, outputs)
    if rank == 0:
        line = {
            "metric": "icp_iterations_per_s", "value": value, "unit": "ICP iterations/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(world),
            "e2e": {"value": e2e_value, "unit": "ICP iterations/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / args.steps,
                    "step_wall_ms": {"min": 1e3 * min(step_wall), "median": 1e3 * float(np.median(step_wall)), "max": 1e3 * max(step_wall)}},
            "gpu_launches": int(launches),
            "launches_per_step": {"kernels": int(launches) // max(args.steps, 1), "host_calls": "1 graph launch (the 50 loop iterations, one kernel each: "
                                  "correspondences + rows + reduction + solve step) + 7 set-up kernels (state, source sort)"},
            "loop": {"slot_iterations_per_step": C2_POINTS * C2_ITERS, "searched": int(searched), "plane_fits": int(fitted),
                     "note": "every iteration recomputes every correspondence; a slot whose 7 stored neighbours provably still "
                             "contain its 5 nearest (gap certificate) skips the cell search, a slot whose 5 neighbours are the same "
                             "ordered list reuses its plane - results identical to searching and fitting every time (tests/test_gpu_parity.py)"},
            "roofline": {"kernel": "k1s::reduce_stream_kernel<float4, wd=false> (K1)", "bound": "hbm", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak,
                         "traffic": K1_NCU_TRAFFIC_BYTES * n_local / C4_SLOTS, "traffic_source": "ncu --set full dram__bytes_read+write per 10 M-slot launch, profiles/k1_r2_ncu_summary.txt",
                         "peak_source": peak_src,
                         "ms_per_launch": k1_ms, "slots_per_launch": n_local, "bytes_per_slot": ALG_BYTES_PER_SLOT,
                         "timing": f"median of 5 batches of {reps} back-to-back launches, CUDA events on the launching stream", "batch_ms": k1_batches},
            "reduction": {"mpoints_per_s": mpts, "slots_total": n_total, "ms": k1_ms,
                          "weight_derivative_variant_ms": k1_ms_wd,
                          "weight_derivative_variant_gbs": ALG_BYTES_PER_SLOT * n_local / (k1_ms_wd * 1e-3) / 1e9,
                          "f64_plane_variant_ms": k1_ms_f64,
                          "f64_plane_variant_gbs": 48 * n_local / (k1_ms_f64 * 1e-3) / 1e9,
                          "n_effective": int(stats[1]),
                          "collective": None if world == 1 else ("sum over ranks inside K1's last block over peer memory (in the timed region)" if comm_mode == 2 else "ncclAllReduce 32 doubles per launch (inside the timed region)"),
                          "sharding": f"{world} contiguous point blocks of {n_local} slots" if world > 1 else None},
            "sharded_icp": c4,
            "trials": c5,
            "cpu_baseline": cpu,
            "parity_checked": bool(parity), "pose_err": parity["pose_err"] if parity else None, "parity": parity,
            "clocks": clocks,
        }
        print(json.dumps(line))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the run, write what the timed calls returned in their last step as DIR/<name>.npy "
                         "(float64; rank 0): c2_* the flagship step, e2e_* the host-buffer step, c4_* the corridor "
                         "registration, c5_* the Monte-Carlo trials; the reference arm writes c2_pose")
    ap.add_argument("--cpu-worker", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--cpu-trials", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank, local_rank, world = env_int("RANK", 0), env_int("LOCAL_RANK", 0), env_int("WORLD_SIZE", 1)
    if args.cpu_worker:
        pin_openmp_env(host_cpu_budget()[0])
        cpu_worker(args)
        return
    if args.impl == "reference":
        pin_openmp_env(host_cpu_budget()[0])   # before anything loads libgomp: see pin_openmp_env
        run_reference(args, rank, world)
    else:
        # the GPU arm needs no host parallelism: keep torch's libgomp from parking one spinning thread per visible CPU
        # (128 of them against a 16-CPU cgroup quota get the launching thread throttled for milliseconds at a time)
        host_cpu_budget()
        os.environ["OMP_NUM_THREADS"] = "1"
        os.environ["OMP_WAIT_POLICY"] = "passive"
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
