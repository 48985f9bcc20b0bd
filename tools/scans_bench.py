"""Scan-to-map throughput: one dcreg_icp_run_scans call against the same scans one at a time (set_source + icp_run).

Workload (BASELINE config C3 as a sequence): make_parking_sequence - 500 k-point map, --scans frames of 3-8 k points,
radius 0.5, at most 30 iterations, ROT 1e-5 / TRANS 1e-3, kappa_target 10, "Ours".  Both rates are host wall clock
around calls that end in a stream synchronisation, upload and source sort included.  The two ways must agree: identical
iteration counts and statuses, poses within 1e-8 on the SE(3) log.  Prints the GPU name and power limit it ran on,
min / median over --reps repeats after a warm-up, and one JSON line.

    python tools/scans_bench.py [--scans 1000] [--reps 3] [--timeline]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

from dcreg_b200 import Context, default_params  # noqa: E402
from dcreg_b200.scenes import make_parking_sequence  # noqa: E402


def gpu_identity():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # pragma: no cover
        out = f"nvidia-smi unavailable ({e})"
    return out


def se3_log_distance(A, B):
    import dcreg_oracle as o
    return o.se3_log_distance(A, B)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scans", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--timeline", action="store_true", help="also time the parts of one batched call")
    args = ap.parse_args()
    if args.reps < 3:
        ap.error("--reps must be >= 3")

    t0 = time.perf_counter()
    scans, tgt, _, T_init = make_parking_sequence(args.scans)
    n_pts = [len(s) for s in scans]
    print(f"workload: {len(scans)} scans, {sum(n_pts)} points ({min(n_pts)}..{max(n_pts)} per scan), "
          f"{len(tgt)}-point map, built in {time.perf_counter() - t0:.1f} s")
    print(f"gpu: {gpu_identity()}")
    gp = default_params(search_radius=0.5, max_iterations=30, conv_thresh_rot=1e-5, conv_thresh_trans=1e-3,
                        kappa_target=10.0, detection="SCHUR_CONDITION_NUMBER", handling="PRECONDITIONED_CG")

    with Context(0) as ctx:
        ctx.set_target(tgt, 0.5)

        def batched():
            t = time.perf_counter()
            res = ctx.icp_run_scans(gp, scans, T_init)
            return time.perf_counter() - t, res

        def one_at_a_time():
            t = time.perf_counter()
            res = []
            for s, T0 in zip(scans, T_init):
                ctx.set_source(s)
                res.append(ctx.icp_run(gp, T0, want_log=False))
            return time.perf_counter() - t, res

        batched(); one_at_a_time()                                         # warm-up: allocations, graphs, module load
        tb, ts = [], []
        for _ in range(args.reps):                                         # alternate the two ways
            dt, rb = batched(); tb.append(dt)
            dt, rs = one_at_a_time(); ts.append(dt)

        same_counts = all(a.iterations == b.iterations and a.status == b.status and a.converged == b.converged
                          for a, b in zip(rb, rs))
        worst = max(se3_log_distance(b.T, a.T) for a, b in zip(rb, rs))
        n = len(scans)
        out = {
            "scans": n, "points": int(sum(n_pts)), "reps": args.reps,
            "batched_s": {"min": min(tb), "median": float(np.median(tb))},
            "one_at_a_time_s": {"min": min(ts), "median": float(np.median(ts))},
            "batched_scans_per_s": {"max": n / min(tb), "median": n / float(np.median(tb))},
            "one_at_a_time_scans_per_s": {"max": n / min(ts), "median": n / float(np.median(ts))},
            "agree": {"iterations_and_status_identical": same_counts, "max_pose_se3_log": worst,
                      "ok": bool(same_counts and worst <= 1e-8)},
            "converged": int(sum(r.converged for r in rb)), "mean_iterations": float(np.mean([r.iterations for r in rb])),
            "gpu": gpu_identity(),
        }
        print(f"batched       : {out['batched_scans_per_s']['max']:9.1f} scans/s best, "
              f"{out['batched_scans_per_s']['median']:9.1f} median  ({min(tb) * 1e3:.1f} / {np.median(tb) * 1e3:.1f} ms per call)")
        print(f"one at a time : {out['one_at_a_time_scans_per_s']['max']:9.1f} scans/s best, "
              f"{out['one_at_a_time_scans_per_s']['median']:9.1f} median  ({min(ts) * 1e3:.1f} / {np.median(ts) * 1e3:.1f} ms in all)")
        print(f"agreement     : iterations/status identical = {same_counts}, worst pose difference {worst:.2e} "
              f"({out['converged']} / {n} converged, {out['mean_iterations']:.1f} iterations on average)")

        if args.timeline:
            # where the time of one batched call goes: upload + sort + first iteration chunk vs the rest (torch profiler)
            import torch
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                ctx.icp_run_scans(gp, scans, T_init)
                torch.cuda.synchronize()
            rows = {}
            for e in prof.events():
                if e.device_type.name == "CUDA":
                    r = rows.setdefault(e.name[:60], [0, 0.0])
                    r[0] += 1; r[1] += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
            print("device time of one batched call by kernel / copy (us):")
            for name, (cnt, us) in sorted(rows.items(), key=lambda kv: -kv[1][1])[:12]:
                print(f"  {us:10.1f}  x{cnt:<5d} {name}")
            out["timeline_us"] = {k: v[1] for k, v in rows.items()}
        print(json.dumps(out))
        if not out["agree"]["ok"]:
            sys.exit(1)


if __name__ == "__main__":
    main()
