"""Synthetic scan pairs for the BASELINE.json configs (SURVEY.md §8d).  NumPy only; seeds fixed.

C2  make_cylinder : the shipped cylinder's geometry (wall R = 40 m, z in [0, 20] + floor disc z = 0) at any size
C3  make_parking  : ground-dominated local map + sparse verticals, LiDAR-like frame (stand-in, pair not shipped)
    make_parking_sequence : a sequence of ragged frames along a path over the same map (scan-to-map batches)
C4  make_corridor : two parallel walls + floor + ceiling, rank-deficient along x
C5  trial_poses   : seeded perturbations t ~ U[-1, 1]^3 m, rpy ~ U[-3, 3]^3 deg for the Monte-Carlo (SURVEY.md §8d)
    load_pcd_xyz  : PCD v0.7 `DATA binary` with float32 fields (the shipped clouds, SURVEY.md Appendix B.3)
"""
from __future__ import annotations

import math

import numpy as np


def pose6d_to_matrix(x, y, z, roll, pitch, yaw):
    """T = Trans * Rz * Ry * Rx (radians) - the reference's Pose6D2Matrix convention (utils.hpp:452-460)."""
    cr, sr, cp, sp, cy, sy = math.cos(roll), math.sin(roll), math.cos(pitch), math.sin(pitch), math.cos(yaw), math.sin(yaw)
    Rx = np.array([[1, 0, 0], [0, cr, -sr], [0, sr, cr]], dtype=np.float64)
    Ry = np.array([[cp, 0, sp], [0, 1, 0], [-sp, 0, cp]], dtype=np.float64)
    Rz = np.array([[cy, -sy, 0], [sy, cy, 0], [0, 0, 1]], dtype=np.float64)
    T = np.eye(4)
    T[:3, :3] = Rz @ Ry @ Rx
    T[:3, 3] = [x, y, z]
    return T


def g2_initial_pose():
    """The perturbation of the reference's published cylinder run (0.2, 0.8, 0.5 m; 0.1, 0.1, 2 deg)."""
    d = math.pi / 180.0
    return pose6d_to_matrix(0.2, 0.8, 0.5, 0.1 * d, 0.1 * d, 2.0 * d)


def make_cylinder(n, seed=42, radius=40.0, height=20.0, noise=0.0):
    rng = np.random.default_rng(seed)
    nw = n // 2
    nf = n - nw
    th = rng.uniform(0, 2 * np.pi, nw); z = rng.uniform(0, height, nw)
    wall = np.stack([radius * np.cos(th), radius * np.sin(th), z], axis=1)
    rr = radius * np.sqrt(rng.uniform(0, 1, nf)); th2 = rng.uniform(0, 2 * np.pi, nf)
    floor = np.stack([rr * np.cos(th2), rr * np.sin(th2), np.zeros(nf)], axis=1)
    pts = np.concatenate([wall, floor], axis=0)
    if noise > 0:
        pts = pts + rng.normal(0, noise, pts.shape)
    return np.ascontiguousarray(pts, dtype=np.float32)


def make_corridor(n, seed=44, length=200.0, half_width=2.0, height=3.0, noise=0.0):
    rng = np.random.default_rng(seed)
    k = n // 4
    parts = []
    for ysign in (1.0, -1.0):
        x = rng.uniform(0, length, k); z = rng.uniform(0, height, k)
        parts.append(np.stack([x, np.full(k, ysign * half_width), z], axis=1))
    x = rng.uniform(0, length, k); y = rng.uniform(-half_width, half_width, k)
    parts.append(np.stack([x, y, np.zeros(k)], axis=1))
    m = n - 3 * k
    x = rng.uniform(0, length, m); y = rng.uniform(-half_width, half_width, m)
    parts.append(np.stack([x, y, np.full(m, height)], axis=1))
    pts = np.concatenate(parts, axis=0)
    if noise > 0:
        pts = pts + rng.normal(0, noise, pts.shape)
    return np.ascontiguousarray(pts, dtype=np.float32)


def make_parking(n_map=500_000, n_scan=6_000, seed=43, extent=60.0, max_range=30.0):
    """Ground plane (z = -1.8 + 1 cm noise) with a few pillars/walls; the scan is a range-limited subsample of
    the map seen from the origin.  Planar degeneracy: x, y, yaw weakly constrained."""
    rng = np.random.default_rng(seed)
    ng = int(n_map * 0.9)
    g = np.stack([rng.uniform(-extent, extent, ng), rng.uniform(-extent, extent, ng),
                  -1.8 + rng.normal(0, 0.01, ng)], axis=1)
    nv = n_map - ng
    npil = 12
    centers = rng.uniform(-extent * 0.8, extent * 0.8, (npil, 2))
    which = rng.integers(0, npil, nv)
    ang = rng.uniform(0, 2 * np.pi, nv)
    v = np.stack([centers[which, 0] + 0.4 * np.cos(ang), centers[which, 1] + 0.4 * np.sin(ang),
                  rng.uniform(-1.8, 1.5, nv)], axis=1)
    tgt = np.concatenate([g, v], axis=0).astype(np.float32)
    rngs = np.linalg.norm(tgt[:, :2], axis=1)
    cand = np.nonzero(rngs < max_range)[0]
    pick = rng.choice(cand, size=min(n_scan, cand.size), replace=False)
    scan = (tgt[pick].astype(np.float64) + rng.normal(0, 0.005, (pick.size, 3))).astype(np.float32)
    return np.ascontiguousarray(scan), np.ascontiguousarray(tgt)


def make_parking_sequence(n_scans, seed=46, n_map=500_000, path_radius=20.0, max_range=30.0, min_points=3_000,
                          max_points=8_000, noise=0.005):
    """A recorded sequence over make_parking's map: returns (scans, map, T_gt, T_init).

    The vehicle drives one lap of a circle of radius path_radius around the map's centre, heading along the path;
    scan s is a subsample of the map points within max_range (horizontally) of its position, between min_points and
    max_points of them (ragged), plus `noise` m of Gaussian noise, in the vehicle's body frame: T_gt[s] @ scan lies on
    the map.  T_init[s] = T_gt[s] @ dT with dT of the size of icp_pk01.yaml's initial offset (0.15 / 0.12 / 0.13 m,
    0.015 / 1.31 / 2.17 deg), each component scaled by a seeded U[-1, 1]."""
    _, tgt = make_parking(n_map=n_map, seed=43)
    rng = np.random.default_rng(seed)
    d = math.pi / 180.0
    size = np.array([0.15, 0.12, 0.13, 0.015 * d, 1.31 * d, 2.17 * d])
    mx, my = tgt[:, 0].astype(np.float64), tgt[:, 1].astype(np.float64)
    scans, T_gt, T_init = [], [], []
    for s in range(n_scans):
        th = 2.0 * math.pi * s / n_scans
        T = pose6d_to_matrix(path_radius * math.cos(th), path_radius * math.sin(th), 0.0, 0.0, 0.0, th + math.pi / 2)
        cand = np.nonzero((mx - T[0, 3]) ** 2 + (my - T[1, 3]) ** 2 < max_range * max_range)[0]
        k = min(int(rng.integers(min_points, max_points + 1)), cand.size)
        pick = np.sort(rng.choice(cand, size=k, replace=False))
        world = tgt[pick].astype(np.float64) + rng.normal(0, noise, (k, 3))
        scans.append(np.ascontiguousarray(((world - T[:3, 3]) @ T[:3, :3]).astype(np.float32)))
        dT = pose6d_to_matrix(*(size * rng.uniform(-1.0, 1.0, 6)))
        T_gt.append(T)
        T_init.append(T @ dT)
    return scans, tgt, np.array(T_gt), np.array(T_init)


def trial_poses(n, seed=45, max_trans=1.0, max_rot_deg=3.0):
    """(n, 4, 4) initial poses of a perturbation Monte-Carlo (BASELINE.json configs[4])."""
    rng = np.random.default_rng(seed)
    t = rng.uniform(-max_trans, max_trans, (n, 3))
    rpy = np.deg2rad(rng.uniform(-max_rot_deg, max_rot_deg, (n, 3)))
    return np.array([pose6d_to_matrix(t[i, 0], t[i, 1], t[i, 2], rpy[i, 0], rpy[i, 1], rpy[i, 2]) for i in range(n)])


def load_pcd_xyz(path):
    """x, y, z columns of a PCD v0.7 file with `DATA binary` and 4-byte float fields (pcl::PointXYZI on disk)."""
    with open(path, "rb") as f:
        raw = f.read()
    head_end = raw.index(b"DATA binary") + len(b"DATA binary")
    head_end = raw.index(b"\n", head_end - 1) + 1
    hdr = {}
    for ln in raw[:head_end].decode("ascii", "replace").splitlines():
        tok = ln.split()
        if tok and not tok[0].startswith("#"):
            hdr[tok[0]] = tok[1:]
    if any(s != "4" for s in hdr["SIZE"]) or any(t != "F" for t in hdr["TYPE"]):
        raise ValueError("only 4-byte float fields are supported")
    nf, npts = len(hdr["FIELDS"]), int(hdr["POINTS"][0])
    a = np.frombuffer(raw, dtype="<f4", count=npts * nf, offset=head_end).reshape(npts, nf)
    cols = [hdr["FIELDS"].index(c) for c in ("x", "y", "z")]
    return np.ascontiguousarray(a[:, cols], dtype=np.float32)
