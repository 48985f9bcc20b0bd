"""Point-to-point metrics for many poses: N dcreg_point_to_point_metrics calls against one
dcreg_point_to_point_metrics_batch call, in the same process, alternating.

Workloads: the shipped 7 562-point cylinder (threshold 0.2, cell 1.0) at 1, 50 and 5000 poses (scenes.trial_poses), and
the C2 100 k cylinder at 50 poses.  Times are host wall clock around calls that end in a stream synchronisation, min /
median over --reps repeats after a warm-up of both ways.  The two ways must agree bit for bit.  Then the CLI end to end
on an icp_iter.yaml-shaped config of the shipped cloud (5 SO(3) methods, 5000 iterations each with convergence
thresholds ~0, so 25 000 iteration rows whose metrics the batched call evaluates, one call per method).  Prints the GPU
name and power limit it ran on, and one JSON line.

    python tools/p2p_batch_bench.py [--reps 3] [--skip-cli]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from dcreg_b200 import Context  # noqa: E402
from dcreg_b200.scenes import load_pcd_xyz, make_cylinder, trial_poses  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def gpu_identity():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # pragma: no cover
        out = f"nvidia-smi unavailable ({e})"
    return out


def compare(ctx, pts, n_poses, reps, thr=0.2, cell=1.0):
    ctx.set_source(pts)
    ctx.set_target(pts, cell)
    T = trial_poses(n_poses)

    def singles():
        t = time.perf_counter()
        out = np.empty((n_poses, 4))
        for i in range(n_poses):
            m = ctx.point_to_point_metrics(T[i], thr)
            out[i] = (m["rmse"], m["fitness"], m["chamfer"], m["n_valid"])
        return time.perf_counter() - t, out

    def batch():
        t = time.perf_counter()
        m = ctx.point_to_point_metrics_batch(T, thr)
        dt = time.perf_counter() - t
        return dt, np.stack([m["rmse"], m["fitness"], m["chamfer"], m["n_valid"].astype(np.float64)], axis=1)

    singles(); batch()                                         # warm-up: module load, source grid, buffers
    ts, tb = [], []
    for _ in range(reps):
        dt, a = singles(); ts.append(dt)
        dt, b = batch(); tb.append(dt)
    same = bool(np.array_equal(a, b))
    r = {"points": len(pts), "poses": n_poses, "reps": reps,
         "singles_ms": {"min": 1e3 * min(ts), "median": 1e3 * float(np.median(ts))},
         "batch_ms": {"min": 1e3 * min(tb), "median": 1e3 * float(np.median(tb))},
         "speedup_min": min(ts) / min(tb), "bit_identical": same}
    print(f"{len(pts):7d} pts x {n_poses:5d} poses: singles {r['singles_ms']['min']:9.2f} / {r['singles_ms']['median']:9.2f} ms, "
          f"batch {r['batch_ms']['min']:8.2f} / {r['batch_ms']['median']:8.2f} ms (min / median), "
          f"x{r['speedup_min']:.1f}, bit-identical {same}")
    return r


def cli_run(reps):
    """icp_iter.yaml-shaped run of the CLI on the shipped cloud: 5 methods, 5000 iterations each."""
    import json as js
    from dcreg_b200 import build as b
    from test_cli_runner import METHODS, write_config
    with open(os.path.join(GOLD, "golden.json")) as f:
        setup = js.load(f)["G3"]["setup"]
    runner = b.build_runner()
    times = []
    with tempfile.TemporaryDirectory() as d:
        cfg = os.path.join(d, "icp_iter.yaml")
        write_config(cfg, os.path.join(d, "out"), setup, sorted(METHODS))
        for _ in range(reps + 1):
            t = time.perf_counter()
            res = subprocess.run([runner, cfg], capture_output=True, text=True, timeout=1800)
            times.append(time.perf_counter() - t)
            if res.returncode != 0:
                raise RuntimeError(res.stdout[-2000:] + res.stderr[-2000:])
        with open(os.path.join(d, "out", "iteration_details_with_dx.csv")) as f:
            rows = sum(1 for _ in f) - 1
    times = times[1:]
    r = {"methods": len(METHODS), "max_iterations": setup["max_iterations"], "csv_rows": rows,
         "wall_s": {"min": min(times), "median": float(np.median(times))}}
    print(f"CLI, {len(METHODS)} methods x {setup['max_iterations']} iterations ({rows} CSV rows): "
          f"{r['wall_s']['min']:.2f} / {r['wall_s']['median']:.2f} s wall (min / median)")
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--skip-cli", action="store_true")
    args = ap.parse_args()
    if args.reps < 1:
        ap.error("--reps must be >= 1")
    gpu = gpu_identity()
    print(f"gpu: {gpu}")
    shipped = load_pcd_xyz(os.path.join(GOLD, "cylinder_7562.pcd"))
    out = {"gpu": gpu, "runs": []}
    with Context(0) as ctx:
        for n in (1, 50, 5000):
            out["runs"].append(compare(ctx, shipped, n, args.reps))
        out["runs"].append(compare(ctx, make_cylinder(100_000), 50, args.reps))
    if not args.skip_cli:
        out["cli"] = cli_run(args.reps)
        single = next(r for r in out["runs"] if r["points"] == len(shipped) and r["poses"] == 5000)
        per_call_ms = single["singles_ms"]["min"] / single["poses"]
        out["cli"]["single_call_ms"] = per_call_ms
        print(f"  (the same {out['cli']['csv_rows']} rows one single call each: {out['cli']['csv_rows'] * per_call_ms / 1e3:.1f} s "
              f"at the {per_call_ms:.3f} ms per call measured above)")
    out["gpu_after"] = gpu_identity()
    print(json.dumps(out))
    if not all(r["bit_identical"] for r in out["runs"]):
        sys.exit(1)


if __name__ == "__main__":
    main()
