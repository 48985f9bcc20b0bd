"""Point-to-point metrics for many poses in one call (dcreg_point_to_point_metrics_batch), through the C ABI.

Row i of a batched call equals dcreg_point_to_point_metrics at pose i bit for bit (np.array_equal on the (n, 4) result)
on the shipped cylinder, a 100 k cylinder, a ~200 k corridor turned by 90 / 180 degrees and a parking scan against its
map; all 2620 shipped per-iteration poses of the reference go through in one call and land within 2e-7 of its printed
P2P_RMSE / Chamfer_Distance; the pose order and the internal chunking do not change results; the cached source grid
follows set_source / set_target; bad arguments are refused.  The CLI's iteration CSV and Monte-Carlo CSV carry the
single call's values.
"""
import csv
import math
import os
import subprocess

import numpy as np
import pytest

import dcreg_oracle as o

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def ctx():
    from dcreg_b200 import Context
    c = Context(0)
    yield c
    c.close()


def singles(ctx, T, thr):
    out = np.empty((len(T), 4))
    for i, Ti in enumerate(T):
        m = ctx.point_to_point_metrics(Ti, thr)
        out[i] = (m["rmse"], m["fitness"], m["chamfer"], m["n_valid"])
    return out


def batched(ctx, T, thr):
    m = ctx.point_to_point_metrics_batch(T, thr)
    assert m["rmse"].dtype == np.float64 and m["n_valid"].dtype.kind == "i"
    return np.stack([m["rmse"], m["fitness"], m["chamfer"], m["n_valid"].astype(np.float64)], axis=1)


def about(c, yaw_deg, t=(0.0, 0.0, 0.0)):
    """yaw about the point c, then a translation"""
    th = math.radians(yaw_deg)
    T = np.eye(4)
    T[:2, :2] = [[math.cos(th), -math.sin(th)], [math.sin(th), math.cos(th)]]
    T[:3, 3] = np.asarray(c) - T[:3, :3] @ np.asarray(c) + np.asarray(t)
    return T


def test_shipped_cylinder_equals_single_calls(ctx, cylinder):
    from dcreg_b200.scenes import g2_initial_pose, trial_poses
    ctx.set_source(cylinder)
    ctx.set_target(cylinder, 1.0)
    T = np.concatenate([np.eye(4)[None], g2_initial_pose()[None], trial_poses(64)])
    assert np.array_equal(batched(ctx, T, 0.2), singles(ctx, T, 0.2))
    one = batched(ctx, T[1:2], 0.2)                         # a one-pose call
    assert np.array_equal(one, singles(ctx, T[1:2], 0.2))


def test_cylinder_100k_equals_single_calls(ctx):
    from dcreg_b200.scenes import make_cylinder, trial_poses
    pts = make_cylinder(100_000)
    ctx.set_source(pts)
    ctx.set_target(pts, 1.0)
    T = trial_poses(8, seed=9)
    assert np.array_equal(batched(ctx, T, 0.2), singles(ctx, T, 0.2))


def test_corridor_turned_equals_single_calls(ctx):
    """yaw 90 / 180 degrees about the corridor's centre: the aligned bounding box is not the source's"""
    from dcreg_b200.scenes import make_corridor
    pts = make_corridor(200_000)
    ctx.set_source(pts)
    ctx.set_target(pts, 1.0)
    c = (100.0, 0.0, 1.5)
    T = np.array([about(c, 90.0), about(c, 180.0), about(c, 180.0, (0.3, -0.1, 0.05)), about(c, -90.0, (2.0, 0.5, 0.0)),
                  about(c, 1.0)])
    assert np.array_equal(batched(ctx, T, 0.2), singles(ctx, T, 0.2))


def test_parking_pair_equals_single_calls(ctx):
    from dcreg_b200.scenes import make_parking, trial_poses
    scan, tgt = make_parking(n_map=100_000, n_scan=6_000)
    ctx.set_source(scan)
    ctx.set_target(tgt, 0.5)
    T = trial_poses(12, seed=5)
    assert np.array_equal(batched(ctx, T, 0.5), singles(ctx, T, 0.5))


def test_shipped_rows_in_one_call(ctx, cylinder):
    f = np.load(os.path.join(GOLD, "p2p_rows.npz"))
    ctx.set_source(cylinder)
    ctx.set_target(cylinder, 1.0)
    out = batched(ctx, f["T"], 0.2)
    assert out.shape == (2620, 4)
    assert np.abs(out[:, 0] - f["p2p_rmse"]).max() < 2e-7
    assert np.abs(out[:, 2] - f["chamfer"]).max() < 2e-7
    sub = np.arange(0, 2620, 131)
    assert np.array_equal(out[sub], singles(ctx, f["T"][sub], 0.2))


def test_permutation_and_chunks(ctx, cylinder, monkeypatch):
    from dcreg_b200.scenes import trial_poses
    ctx.set_source(cylinder)
    ctx.set_target(cylinder, 1.0)
    T = trial_poses(200, seed=21)
    ref = batched(ctx, T, 0.2)
    perm = np.random.default_rng(0).permutation(len(T))
    assert np.array_equal(batched(ctx, T[perm], 0.2), ref[perm])
    monkeypatch.setenv("DCREG_P2P_CHUNK", "7")                # 29 chunks of at most 7 poses
    assert np.array_equal(batched(ctx, T, 0.2), ref)
    monkeypatch.delenv("DCREG_P2P_CHUNK")
    sub = [0, 6, 7, 8, 13, 14, 99, 195, 196, 199]
    assert np.array_equal(ref[sub], singles(ctx, T[sub], 0.2))


def test_cache_follows_set_source_and_set_target(ctx, cylinder):
    from dcreg_b200.scenes import make_cylinder, trial_poses
    T = trial_poses(16, seed=33)
    ctx.set_source(cylinder)
    ctx.set_target(cylinder, 1.0)
    assert np.array_equal(batched(ctx, T, 0.2), singles(ctx, T, 0.2))
    other = make_cylinder(20_000, seed=8, noise=0.01)
    ctx.set_source(other)                                      # another source: its own grid
    assert np.array_equal(batched(ctx, T, 0.2), singles(ctx, T, 0.2))
    ctx.set_target(cylinder, 0.4)                              # another cell size: the source grid is rebuilt with it
    assert np.array_equal(batched(ctx, T, 0.2), singles(ctx, T, 0.2))
    ctx.set_target(cylinder, 2.5)
    assert np.array_equal(batched(ctx, T, 0.2), singles(ctx, T, 0.2))


def test_bad_arguments_are_refused(ctx, cylinder):
    from dcreg_b200 import Context
    from dcreg_b200.api import BAD_ARG, DcregError, _dptr
    T = np.eye(4)[None]
    out = np.empty(4)
    lib = ctx.lib
    with Context(0) as fresh:                                  # no source / target yet
        assert lib.dcreg_point_to_point_metrics_batch(fresh._h, 1, _dptr(T), 0.2, _dptr(out)) == BAD_ARG
        assert "set source and target" in lib.dcreg_last_error(fresh._h).decode()
        fresh.set_source(cylinder)
        assert lib.dcreg_point_to_point_metrics_batch(fresh._h, 1, _dptr(T), 0.2, _dptr(out)) == BAD_ARG
    ctx.set_source(cylinder)
    ctx.set_target(cylinder, 1.0)
    assert lib.dcreg_point_to_point_metrics_batch(ctx._h, 0, _dptr(T), 0.2, _dptr(out)) == BAD_ARG
    assert "n_poses" in lib.dcreg_last_error(ctx._h).decode()
    assert lib.dcreg_point_to_point_metrics_batch(ctx._h, -3, _dptr(T), 0.2, _dptr(out)) == BAD_ARG
    assert lib.dcreg_point_to_point_metrics_batch(ctx._h, 1, None, 0.2, _dptr(out)) == BAD_ARG
    assert lib.dcreg_point_to_point_metrics_batch(ctx._h, 1, _dptr(T), 0.2, None) == BAD_ARG
    assert "null pointer" in lib.dcreg_last_error(ctx._h).decode()
    assert lib.dcreg_point_to_point_metrics_batch(None, 1, _dptr(T), 0.2, _dptr(out)) == BAD_ARG
    with pytest.raises(DcregError):
        ctx.point_to_point_metrics_batch(np.empty((0, 4, 4)), 0.2)
    # a hash-grid target: bounding box too large for a dense grid at this cell size
    far = np.concatenate([cylinder, np.array([[6000.0, 6000.0, 3000.0]], np.float32)])
    ctx.set_target(far, 0.5)
    assert lib.dcreg_point_to_point_metrics_batch(ctx._h, 1, _dptr(T), 0.2, _dptr(out)) == BAD_ARG
    assert "dense grid" in lib.dcreg_last_error(ctx._h).decode()
    # a source too large for a dense grid of its own, against a dense target
    ctx.set_target(cylinder, 0.5)
    ctx.set_source(np.concatenate([cylinder, np.array([[5000.0, 5000.0, 2500.0]], np.float32)]))
    assert lib.dcreg_point_to_point_metrics_batch(ctx._h, 1, _dptr(T), 0.2, _dptr(out)) == BAD_ARG
    assert "over the source" in lib.dcreg_last_error(ctx._h).decode()
    ctx.set_source(cylinder)                                   # and the context still works afterwards
    ctx.set_target(cylinder, 1.0)
    assert np.array_equal(batched(ctx, T, 0.2), singles(ctx, T, 0.2))


# ---- CLI -------------------------------------------------------------------------------------------------------------
METHODS = {
    "ME-SR": ("FULL_EVD_MIN_EIGENVALUE", "SOLUTION_REMAPPING"),
    "ME-TSVD": ("FULL_EVD_MIN_EIGENVALUE", "TRUNCATED_SVD"),
    "ME-TReg": ("FULL_EVD_MIN_EIGENVALUE", "STANDARD_REGULARIZATION"),
    "FCN-SR": ("FULL_SVD_CONDITION", "SOLUTION_REMAPPING"),
    "Ours": ("SCHUR_CONDITION_NUMBER", "PRECONDITIONED_CG"),
}


def g2_config(path, out_dir, s, methods, extra=""):
    x, y, z = s["init_xyz"]
    r, p, w = s["init_rpy_deg"]
    lines = "\n".join(f'  "{m}": [ "{METHODS[m][0]}", "{METHODS[m][1]}" ]' for m in methods)
    path.write_text(f"""
test:
  num_runs: 1
  save_pcd: false
  save_error_pcd: false
  visualize: false
output:
  save_csv: true
paths:
  folder_path: "{GOLD}/"
  output_folder: "{out_dir}/"
  source_pcd: "cylinder_7562.pcd"
  target_pcd: "cylinder_7562.pcd"
icp:
  search_radius: {s['search_radius']}
  max_iterations: {s['max_iterations']}
  error_threshold: 0.2
  CONVERGENCE_THRESH_TRANS: {s['conv_trans']}
  CONVERGENCE_THRESH_ROT: {s['conv_rot']}
  normal_nn: 5
  use_weight_derivative: {'true' if s['use_weight_derivative'] else 'false'}
initial_noise:
  x: {x}
  y: {y}
  z: {z}
  roll_deg: {r}
  pitch_deg: {p}
  yaw_deg: {w}
gt_pose:
  x: 0.0
  y: 0.0
  z: 0.0
  roll_deg: 0.0
  pitch_deg: 0.0
  yaw_deg: 0.
degeneracy:
  condition_threshold: {s['cond_thresh']}
  eigenvalue_threshold: {s['eig_thresh']}
method_params:
  standard_reg:
    gamma: {s['std_reg_gamma']}
  pcg:
    kappa_target: {s['kappa_target']}
    tolerance: 1e-6
    max_iter: 10
test_methods:
{lines}
{extra}
""")


def params(s, m):
    from dcreg_b200 import default_params
    return default_params(search_radius=s["search_radius"], max_iterations=s["max_iterations"], detection=METHODS[m][0],
                          handling=METHODS[m][1], use_weight_derivative=int(s["use_weight_derivative"]),
                          conv_thresh_rot=s["conv_rot"], conv_thresh_trans=s["conv_trans"], cond_thresh=s["cond_thresh"],
                          eig_thresh=s["eig_thresh"], kappa_target=s["kappa_target"], std_reg_gamma=s["std_reg_gamma"])


def read_csv(path):
    with open(path) as f:
        return list(csv.DictReader(f))


def test_cli_p2p_columns_equal_single_calls(golden, cylinder, tmp_path):
    from dcreg_b200 import api
    from dcreg_b200 import build as b
    runner = b.build_runner()
    g = golden["G2"]
    s = g["setup"]
    methods = ["FCN-SR", "Ours"]
    cfg = tmp_path / "icp.yaml"
    out_dir = tmp_path / "out"
    g2_config(cfg, out_dir, s, methods, extra="monte_carlo:\n  trials: 40\n  seed: 5\n  max_trans_m: 0.6\n  max_rot_deg: 2.0\n")
    res = subprocess.run([runner, str(cfg)], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    rows = read_csv(out_dir / "iteration_details_with_dx.csv")
    d = math.pi / 180
    T0 = o.pose6d_to_matrix(*s["init_xyz"], *(v * d for v in s["init_rpy_deg"]))
    with api.Context() as ctx:
        ctx.set_source(cylinder)
        ctx.set_target(cylinder, s["search_radius"])
        for m in methods:
            mine = [r for r in rows if r["Method"] == m]
            run = ctx.icp_run(params(s, m), T0, want_log=True)
            assert len(mine) == len(run.logs) > 0, m
            for r, lg in zip(mine, run.logs):
                sm = ctx.point_to_point_metrics(np.array(lg.T).reshape(4, 4), 0.2)
                assert r["P2P_RMSE"] == "%.8f" % sm["rmse"] and r["Chamfer_Distance"] == "%.8f" % sm["chamfer"], (m, r["Iteration"])
            mc = read_csv(out_dir / f"monte_carlo_{m}.csv")
            assert len(mc) == 40 and list(mc[0].keys())[-3:] == ["P2P_RMSE", "P2P_Fitness", "Chamfer_Distance"]
            for r in mc:
                T = np.eye(4)
                T[:3] = np.array([float(r[f"T{k // 4}{k % 4}"]) for k in range(12)]).reshape(3, 4)
                sm = ctx.point_to_point_metrics(T, 0.2)
                assert (float(r["P2P_RMSE"]), float(r["P2P_Fitness"]), float(r["Chamfer_Distance"])) == \
                       (sm["rmse"], sm["fitness"], sm["chamfer"]), (m, r["Trial"])
