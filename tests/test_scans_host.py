"""Host side of scan-to-map batches (dcreg_icp_run_scans): the sequence scene and the list -> (xyz, offsets) packing.
No GPU needed."""
import numpy as np
import pytest
from scipy.spatial import cKDTree

from dcreg_b200.api import pack_scans
from dcreg_b200.scenes import make_parking, make_parking_sequence


@pytest.fixture(scope="module")
def seq():
    return make_parking_sequence(5)


def test_sequence_is_seeded_and_deterministic(seq):
    scans, tgt, T_gt, T_init = seq
    again = make_parking_sequence(5)
    assert all(np.array_equal(a, b) for a, b in zip(scans, again[0]))
    assert np.array_equal(tgt, again[1]) and np.array_equal(T_gt, again[2]) and np.array_equal(T_init, again[3])
    other = make_parking_sequence(5, seed=47)
    assert not np.array_equal(other[3], T_init)
    assert np.array_equal(tgt, make_parking(n_map=500_000, seed=43)[1])            # the map is make_parking's map


def test_sequence_shapes_and_perturbations(seq):
    scans, tgt, T_gt, T_init = seq
    assert len(scans) == 5 and T_gt.shape == T_init.shape == (5, 4, 4)
    sizes = [len(s) for s in scans]
    assert all(3_000 <= n <= 8_000 for n in sizes) and len(set(sizes)) == 5         # ragged
    assert all(s.dtype == np.float32 and s.shape[1] == 3 for s in scans)
    for Tg, Ti in zip(T_gt, T_init):
        dT = np.linalg.inv(Tg) @ Ti
        assert np.all(np.abs(dT[:3, 3]) <= [0.15, 0.12, 0.13])
        assert 0.0 < np.linalg.norm(dT[:3, 3]) and np.allclose(dT[:3, :3] @ dT[:3, :3].T, np.eye(3), atol=1e-12)
    assert len({tuple(np.round(T[:2, 3], 3)) for T in T_gt}) == 5                   # the vehicle moves


def test_scans_lie_on_the_map_in_the_true_pose(seq):
    scans, tgt, T_gt, _ = seq
    tree = cKDTree(tgt)
    for s, T in zip(scans, T_gt):
        world = s.astype(np.float64) @ T[:3, :3].T + T[:3, 3]
        d, _ = tree.query(world)
        assert np.median(d) < 0.015 and d.max() < 0.05                              # 5 mm noise per axis
        assert np.linalg.norm(s[:, :2], axis=1).max() < 30.0 + 0.05                 # range-limited, body frame


def test_pack_scans_layout():
    rng = np.random.default_rng(0)
    scans = [rng.normal(size=(n, 3)).astype(np.float32) for n in (1, 31, 32, 33, 257)]
    scans.append(rng.normal(size=(4, 4)))                                           # xyzi, float64: cast, 4th column dropped
    xyz, off = pack_scans(scans)
    assert xyz.dtype == np.float32 and xyz.shape == (1 + 31 + 32 + 33 + 257 + 4, 3) and xyz.flags.c_contiguous
    assert off.dtype == np.int64 and off.tolist() == [0, 1, 32, 64, 97, 354, 358]
    for s, lo, hi in zip(scans, off[:-1], off[1:]):
        assert np.array_equal(xyz[lo:hi], np.asarray(s, dtype=np.float32)[:, :3])
    with pytest.raises(ValueError):
        pack_scans([])
    with pytest.raises(ValueError):
        pack_scans([np.zeros((5, 2), np.float32)])
    _, off = pack_scans([np.zeros((3, 3)), np.zeros((0, 3)), np.zeros((2, 3))])   # an empty scan packs; the C ABI refuses it
    assert off.tolist() == [0, 3, 3, 5]
