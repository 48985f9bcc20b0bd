"""CPU test of the Chamfer search of dcreg_point_to_point_metrics_batch (corr::nn1_search_posed), independent of CUDA.

The batched call finds the nearest ALIGNED source point a = fl32(T p) of every target point y through one grid over the
source in its own frame: rings of cells of growing Chebyshev radius around q' = R^T (y - t), a ring skipped when
(L - margin)^2 * shrink > best with L = (r - 1) * cell * 0.99999 and (margin, shrink) from p2p_bound.hpp.  This test
compiles p2p_bound.hpp for the host, restates the search in NumPy (FP64 transform with a float32 store, float32 squared
distances in corr::dist2's order) and requires the minimum float d2 to equal brute force over fl32(T p) for every query:
random clouds, exact lattices with ties and duplicated points, rotations up to 180 degrees, poses rounded to 8
decimals (not orthonormal), coordinates offset by up to 4096 m and cell sizes from 0.1 to 2 m.  It also checks the
bound point by point: no source point is closer (in float d2) than its source-frame lower bound allows.
"""
import ctypes as C
import math
import os
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F = np.float32

SHIM = r"""
#include "%s"
extern "C" void bound(const double* T, double pmax, double ymax, double* out) {
    const p2p_bound::Bound b = p2p_bound::backward_bound(T, pmax, ymax);
    out[0] = b.margin; out[1] = b.shrink;
}
"""


@pytest.fixture(scope="module")
def bound(tmp_path_factory):
    gxx = shutil.which("g++")
    if not gxx:
        pytest.skip("g++ not available")
    d = tmp_path_factory.mktemp("p2p_bound")
    src = d / "shim.cpp"
    src.write_text(SHIM % os.path.join(ROOT, "dcreg_b200", "csrc", "p2p_bound.hpp"))
    so = d / "libshim.so"
    subprocess.run([gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-o", str(so), str(src)], check=True,
                   capture_output=True)
    lib = C.CDLL(str(so))
    dp = C.POINTER(C.c_double)
    lib.bound.argtypes = [dp, C.c_double, C.c_double, dp]

    def f(T, pmax, ymax):
        T = np.ascontiguousarray(T, dtype=np.float64)
        out = np.zeros(2)
        lib.bound(T.ctypes.data_as(dp), float(pmax), float(ymax), out.ctypes.data_as(dp))
        return out[0], out[1]
    return f


def aligned(src, T):
    """fl32(T p): FP64 transform, float32 store (transform_points_kernel)."""
    return (src.astype(np.float64) @ T[:3, :3].T + T[:3, 3]).astype(F)


def dist2(y, a):
    """corr::dist2: float32 differences, products and sums, x then y then z."""
    e = (y[None, :] - a).astype(F)
    return ((e[:, 0] * e[:, 0]).astype(F) + (e[:, 1] * e[:, 1]).astype(F)).astype(F) + (e[:, 2] * e[:, 2]).astype(F)


def cells(x, inv_cell):
    return np.floor(x.astype(np.float64) * inv_cell).astype(np.int64)


def search(src, src_cells, a, y, T, cell, margin, shrink):
    """nn1_search_posed for one query: returns (min float d2, number of points visited)."""
    inv = 1.0 / cell
    q = T[:3, :3].T @ (y.astype(np.float64) - T[:3, 3])
    qc = np.clip(np.floor(q * inv), -2.0 ** 30, 2.0 ** 30).astype(np.int64)
    ring = np.abs(src_cells - qc).max(axis=1)
    best = F(3.0e38)
    visited = 0
    for r in np.unique(ring):                 # the device also walks empty rings; the bound only grows with r
        if r > 0:
            l = (r - 1) * (1.0 / inv) * 0.99999 - margin
            if l > 0.0 and l * l * shrink > float(best):
                break
        sel = ring == r
        visited += int(sel.sum())
        best = min(best, dist2(y, a[sel]).min())
    return best, visited


def rot(axis, deg):
    axis = np.asarray(axis, np.float64) / np.linalg.norm(axis)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    th = math.radians(deg)
    return np.eye(3) + math.sin(th) * K + (1 - math.cos(th)) * K @ K


def pose(R, t, decimals=None):
    T = np.eye(4)
    T[:3, :3] = R; T[:3, 3] = t
    return np.round(T, decimals) if decimals is not None else T


def cases():
    rng = np.random.default_rng(7)
    rnd = rng.uniform(-4, 4, (1500, 3)).astype(F)
    g = np.arange(-3, 3, 0.5, dtype=F)
    X, Y, Z = np.meshgrid(g, g, g[:4])
    lat = np.stack([X.ravel(), Y.ravel(), Z.ravel()], axis=1).astype(F)
    latdup = np.concatenate([lat, lat[::3], lat[::5]]).astype(F)
    surf = rng.uniform(-6, 6, (1500, 3)).astype(F)
    surf[:, 2] = (0.3 * np.sin(surf[:, 0])).astype(F)
    poses = [
        ("identity", np.eye(4)),
        ("yaw90", pose(rot([0, 0, 1], 90), [0.5, -0.25, 0.0])),
        ("yaw180", pose(rot([0, 0, 1], 180), [0.0, 0.0, 0.0])),
        ("x180", pose(rot([1, 0, 0], 180), [1.0, 0.5, -0.5])),
        ("random", pose(rot(rng.normal(size=3), rng.uniform(0, 180)), rng.uniform(-1, 1, 3))),
        ("small", pose(rot(rng.normal(size=3), 2.0), [0.2, 0.8, 0.5])),
        ("8 decimals", pose(rot(rng.normal(size=3), 37.0), rng.uniform(-1, 1, 3), decimals=8)),
    ]
    for cname, cloud in (("random", rnd), ("lattice", lat), ("lattice+duplicates", latdup), ("surface", surf)):
        for off in (0.0, 4096.0):
            src = (cloud + F(off)).astype(F)
            for pname, T in poses:
                T = T.copy()
                if off:   # keep the aligned cloud at the offset too: rotate about it
                    c = np.full(3, off)
                    T[:3, 3] += c - T[:3, :3] @ c
                for cell in (0.1, 0.35, 1.0, 2.0):
                    yield f"{cname}/off{off:g}/{pname}/cell{cell}", src, T, cell


def queries(src, T, rng):
    """Target points: near aligned points, exactly on aligned points, inside the cloud's box and outside it."""
    a = aligned(src, T)
    k = min(120, len(src))
    pick = rng.choice(len(src), k, replace=False)
    near = (a[pick] + rng.normal(scale=0.02, size=(k, 3))).astype(F)
    exact = a[pick[:30]]
    lo, hi = a.min(axis=0).astype(np.float64), a.max(axis=0).astype(np.float64)
    box = rng.uniform(lo, hi, (40, 3)).astype(F)
    far = (hi + rng.uniform(0.5, 6.0, (10, 3))).astype(F)
    return np.concatenate([near, exact, box, far]).astype(F)


def test_posed_search_equals_brute_force(bound):
    rng = np.random.default_rng(3)
    n_cases = pruned = 0
    for name, src, T, cell in cases():
        a = aligned(src, T)
        y = queries(src, T, rng)
        pmax = float(np.linalg.norm(src.astype(np.float64), axis=1).max())
        ymax = float(np.linalg.norm(y.astype(np.float64), axis=1).max())
        margin, shrink = bound(T, pmax, ymax)
        assert 0 < margin < 1e-2 and 0.999 < shrink < 1, (name, margin, shrink)
        sc = cells(src, 1.0 / cell)
        for j in range(len(y)):
            got, visited = search(src, sc, a, y[j], T, cell, margin, shrink)
            want = dist2(y[j], a).min()
            assert got == want, (name, j, got, want)
            pruned += visited < len(src)
        n_cases += 1
    assert n_cases == 4 * 2 * 7 * 4
    assert pruned > 0.5 * n_cases * 200          # the bound does prune: most queries skip rings


def test_bound_holds_point_by_point(bound):
    """(|p - q'| - margin)^2 * shrink <= float d2(y, fl32(T p)) for every source point: the inequality the skip rule
    rests on, with the exact source-frame distance instead of the ring bound."""
    rng = np.random.default_rng(5)
    for name, src, T, cell in cases():
        if cell != 1.0:
            continue
        a = aligned(src, T)
        y = queries(src, T, rng)[::4]
        pmax = float(np.linalg.norm(src.astype(np.float64), axis=1).max())
        ymax = float(np.linalg.norm(y.astype(np.float64), axis=1).max())
        margin, shrink = bound(T, pmax, ymax)
        for j in range(len(y)):
            q = T[:3, :3].T @ (y[j].astype(np.float64) - T[:3, 3])
            L = np.linalg.norm(src.astype(np.float64) - q, axis=1)
            l = np.maximum(L - margin, 0.0)
            assert np.all(l * l * shrink <= dist2(y[j], a).astype(np.float64)), name


def test_bound_of_a_non_rotation_disables_pruning(bound):
    T = np.eye(4); T[0, 0] = 2.0
    margin, shrink = bound(T, 10.0, 10.0)
    assert shrink == 0.0 and margin == math.inf
    T = np.eye(4); T[0, 1] = np.nan
    assert bound(T, 10.0, 10.0)[1] == 0.0


def test_p2p_fixture_matches_the_oracle():
    """tests/golden/p2p_rows.npz (make_p2p_rows.py): shape and provenance, and a subset against the CPU oracle."""
    import dcreg_oracle as o
    f = np.load(os.path.join(ROOT, "tests", "golden", "p2p_rows.npz"))
    assert f["T"].shape == (2620, 4, 4) and f["p2p_rmse"].shape == (2620,) and f["chamfer"].shape == (2620,)
    assert int((f["source"] == 0).sum()) == 120 and int((f["source"] == 1).sum()) == 2500
    assert {"FCN-SR", "ME-SR", "ME-TReg", "ME-TSVD", "Ours"} <= set(f["method"].tolist())
    pts = o.read_pcd_xyz(os.path.join(ROOT, "tests", "golden", "cylinder_7562.pcd"))
    tree = o.build_tree(pts)
    for i in list(range(0, 120, 7)) + list(range(120, 2620, 97)):
        m = o.point_to_point_metrics(pts, pts, f["T"][i], 0.2, tree_tgt=tree)
        assert abs(m["rmse"] - f["p2p_rmse"][i]) < 2e-7 and abs(m["chamfer"] - f["chamfer"][i]) < 2e-7, i
