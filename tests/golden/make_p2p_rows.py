#!/usr/bin/env python
"""Extract the reference's shipped per-iteration point-to-point metrics into tests/golden/p2p_rows.npz.

Needs a checkout of the reference project (JokerJohn/DCReg with its shipped results); the tests only read the npz
this writes:
    python tests/golden/make_p2p_rows.py <reference checkout> [--check]

Every row of the reference's iteration_details_with_dx.csv carries P2P_RMSE and Chamfer_Distance (calculatePointToPoint-
Error, error threshold 0.2, on the shipped cylinder cloud tests/golden/cylinder_7562.pcd) next to the pose it was
evaluated at, all printed with 8 decimals.  Rows kept:
  results/simulation/table3_fig9_fig10/  all 120 rows                (source 0)
  results/simulation/fig8_5000iters/     every 10th of 25 000 rows    (source 1)
= 2620 poses.  Arrays: method (str), source, run, iteration (int32), T (n, 4, 4) as printed, p2p_rmse, chamfer.

--check evaluates oracle/dcreg_oracle.py:point_to_point_metrics at every kept pose.  First run, all 2620 rows: worst
|P2P_RMSE - oracle| = 9.1e-8 and worst |Chamfer_Distance - oracle| = 1.0e-7 (the 8-decimal printing of the CSV and
of the poses).
Only numeric rows are extracted; no reference source code is copied.
"""
import csv
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = (("results/simulation/table3_fig9_fig10/iteration_details_with_dx.csv", 1),
           ("results/simulation/fig8_5000iters/iteration_details_with_dx.csv", 10))


def extract(ref):
    cols = {k: [] for k in ("method", "source", "run", "iteration", "T", "p2p_rmse", "chamfer")}
    for s, (rel, every) in enumerate(SOURCES):
        with open(os.path.join(ref, rel)) as f:
            for i, r in enumerate(csv.DictReader(f)):
                if i % every:
                    continue
                cols["method"].append(r["Method"]); cols["source"].append(s)
                cols["run"].append(int(r["Run"])); cols["iteration"].append(int(r["Iteration"]))
                cols["T"].append([float(r[f"T_{a}{b}"]) for a in range(4) for b in range(4)])
                cols["p2p_rmse"].append(float(r["P2P_RMSE"])); cols["chamfer"].append(float(r["Chamfer_Distance"]))
    return {"method": np.array(cols["method"]), "source": np.array(cols["source"], np.int32),
            "run": np.array(cols["run"], np.int32), "iteration": np.array(cols["iteration"], np.int32),
            "T": np.array(cols["T"]).reshape(-1, 4, 4), "p2p_rmse": np.array(cols["p2p_rmse"]),
            "chamfer": np.array(cols["chamfer"])}


def oracle_worst(rows, idx=None):
    """Worst |shipped - oracle| of P2P_RMSE and Chamfer_Distance over rows idx (default: all)."""
    sys.path.insert(0, os.path.join(HERE, "..", "..", "oracle"))
    import dcreg_oracle as o
    pts = o.read_pcd_xyz(os.path.join(HERE, "cylinder_7562.pcd"))
    tree = o.build_tree(pts)
    worst = [0.0, 0.0]
    for i in range(len(rows["T"])) if idx is None else idx:
        m = o.point_to_point_metrics(pts, pts, rows["T"][i], 0.2, tree_tgt=tree)
        worst[0] = max(worst[0], abs(m["rmse"] - rows["p2p_rmse"][i]))
        worst[1] = max(worst[1], abs(m["chamfer"] - rows["chamfer"][i]))
    return worst


def main():
    if len(sys.argv) < 2:
        sys.exit(__doc__)
    rows = extract(sys.argv[1])
    np.savez_compressed(os.path.join(HERE, "p2p_rows.npz"), **rows)
    print(f"{len(rows['T'])} rows -> {os.path.join(HERE, 'p2p_rows.npz')}")
    if "--check" in sys.argv[2:]:
        print("worst |P2P_RMSE - oracle| = %.2g, worst |Chamfer_Distance - oracle| = %.2g" % tuple(oracle_worst(rows)))


if __name__ == "__main__":
    main()
