#!/usr/bin/env python
"""Extract the reference's shipped golden vectors into tests/golden/golden.json.

Needs a checkout of the reference project (JokerJohn/DCReg with its shipped results); the tests only read the
golden.json this writes:
    python tests/golden/make_golden.py <reference checkout>

Sources (SURVEY.md §8c), all relative to the reference checkout:
  G1  DCReg/dataset/icp_results/            released code, init t=(0.01,0.01,0.01), WD off
  G2  results/simulation/table3_fig9_fig10/ full code incl. "Ours", init (0.2,0.8,0.5 m;
                                            0.1,0.1,2 deg), weight derivative ON
  G3  results/simulation/fig8_5000iters/    same as G2, 5000 iterations, thresholds ~ 0
The input cloud (byte-identical in G1 and G2) is committed as tests/golden/cylinder_7562.pcd.
Only numeric rows are extracted; no reference source code is copied.
"""
import csv
import json
import os
import re
import sys

HERE = os.path.dirname(os.path.abspath(__file__))

DX = ["dx_wx", "dx_wy", "dx_wz", "dx_x", "dx_y", "dx_z"]
GRAD = ["grad_wx", "grad_wy", "grad_wz", "grad_x", "grad_y", "grad_z"]


def rows_of(path, methods, keep=None):
    out = {}
    with open(path) as f:
        for r in csv.DictReader(f):
            m = r["Method"]
            if m not in methods:
                continue
            it = int(r["Iteration"])
            if keep is not None and it not in keep:
                continue
            out.setdefault(m, []).append({
                "iteration": it,
                "rmse": float(r["RMSE"]), "fitness": float(r["Fitness"]),
                "time_ms": float(r["Time_ms"]),
                "dx": [float(r[k]) for k in DX],
                "grad": [float(r[k]) for k in GRAD],
                "objective": float(r["objective_value"]),
                "T": [float(r["T_%d%d" % (a, b)]) for a in range(4) for b in range(4)],
                "cond_schur_rot": float(r["Cond_Schur_Rot"]),
                "cond_schur_trans": float(r["Cond_Schur_Trans"]),
                "cond_sub_rot": float(r["Cond_Sub_Rot"]),
                "cond_sub_trans": float(r["Cond_Sub_Trans"]),
                "cond_full_svd": float(r["Cond_Full_SVD"]),
                "mask": [int(r["Degenerate_%d" % i]) for i in range(6)],
                "is_degenerate": int(r["Is_Degenerate"]),
            })
    return out


def first_iter_blocks(path):
    """Parse degeneracy_analysis_first_iter.txt into {method: {...}}."""
    txt = open(path).read()
    out = {}
    for blk in re.split(r"\n(?=Method: )", txt):
        m = re.match(r"Method: (\S+)", blk)
        if not m:
            continue
        d = {}
        e = re.search(r"Eigenvalues \(Full\): ([^\n]+)", blk)
        if e:
            d["eigenvalues_full"] = [float(x) for x in e.group(1).split()]
        k = re.search(r"Degenerate Mask[^:]*: ([^\n]+)", blk)
        if k:
            d["mask"] = [int(x) for x in k.group(1).split()]
        for key, pat in (("cond_full_svd", r"Full SVD: (\S+)"), ("cond_schur_rot", r"Schur Rot: (\S+)"),
                         ("cond_schur_trans", r"Schur Trans: (\S+)"), ("cond_diag_rot", r"\n\s+Diag Rot: (\S+)"),
                         ("cond_diag_trans", r"\n\s+Diag Trans: (\S+)")):
            q = re.search(pat, blk)
            if q and q.group(1) != "nan":
                d[key] = float(q.group(1))
        p = re.search(r"Preconditioner Matrix P:\n((?:\s+[-0-9. ]+\n){6})", blk)
        if p:
            d["P_logged"] = [[float(x) for x in ln.split()] for ln in p.group(1).strip().split("\n")]
        al = re.findall(r"\[(\d)\]~(\w) \(orig_idx=(\d)\): λ=([-0-9.]+), Angle=([-0-9.]+)°", blk)
        if al:
            d["alignment"] = [{"slot": int(a), "axis": b, "orig_idx": int(c), "lambda": float(x), "angle_deg": float(y)}
                              for a, b, c, x, y in al]
        out[m.group(1)] = d
    return out


def main(ref):
    g = {"_source": "JokerJohn/DCReg @ 0519bdb shipped result dumps; see make_golden.py"}
    so3 = {"Ours", "ME-SR", "ME-TSVD", "ME-TReg", "FCN-SR"}
    g1 = os.path.join(ref, "DCReg/dataset/icp_results")
    g["G1"] = {
        "setup": {"init_xyz": [0.01, 0.01, 0.01], "init_rpy_deg": [0, 0, 0], "use_weight_derivative": False,
                  "search_radius": 1.0, "conv_rot": 1e-4, "conv_trans": 1e-3, "std_reg_gamma": 100.0,
                  "eig_thresh": 120.0, "cond_thresh": 10.0, "kappa_target": 10.0, "max_iterations": 30},
        "iterations": rows_of(os.path.join(g1, "iteration_details_with_dx.csv"), so3),
        "first_iter": first_iter_blocks(os.path.join(g1, "degeneracy_analysis_first_iter.txt")),
    }
    g2 = os.path.join(ref, "results/simulation/table3_fig9_fig10")
    g["G2"] = {
        "setup": {"init_xyz": [0.2, 0.8, 0.5], "init_rpy_deg": [0.1, 0.1, 2.0], "use_weight_derivative": True,
                  "search_radius": 1.0, "conv_rot": 1e-5, "conv_trans": 1e-3, "std_reg_gamma": 100.0,
                  "eig_thresh": 120.0, "cond_thresh": 10.0, "kappa_target": 10.0, "max_iterations": 30},
        "iterations": rows_of(os.path.join(g2, "iteration_details_with_dx.csv"), so3),
        "first_iter": first_iter_blocks(os.path.join(g2, "degeneracy_analysis_first_iter.txt")),
        "schur_lambda_rot": [422.505477, 1447.735216, 2999.323349],
        "schur_lambda_trans": [0.629416, 5.601848, 16.871859],
    }
    g3 = os.path.join(ref, "results/simulation/fig8_5000iters")
    keep = set(range(0, 40)) | {99, 999, 4999}
    g["G3"] = {
        "setup": dict(g["G2"]["setup"], conv_rot=1e-14, conv_trans=1e-12, max_iterations=5000),
        "iterations": rows_of(os.path.join(g3, "iteration_details_with_dx.csv"), {"Ours", "ME-TReg"}, keep),
    }
    with open(os.path.join(HERE, "golden.json"), "w") as f:
        json.dump(g, f, indent=0, separators=(",", ":"))
    print("wrote golden.json", os.path.getsize(os.path.join(HERE, "golden.json")), "bytes")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
