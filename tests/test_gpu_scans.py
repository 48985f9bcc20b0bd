"""Many different scans against one map in one call (dcreg_icp_run_scans), through the C ABI.

Every scan of a batch runs the kernels a dcreg_icp_run of that scan alone runs: statuses, flags, iteration counts and
per-iteration counts / masks identical, poses equal to the grouping of the FP64 sums (1e-8 on the SE(3) log).  A one-scan
call is a dcreg_icp_run bit for bit; scans do not see each other (permuting them permutes the results bit for bit).
"""
import ctypes as C
import math

import numpy as np
import pytest

import dcreg_oracle as o

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from dcreg_b200 import Context
    c = Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def seq():
    from dcreg_b200.scenes import make_parking_sequence
    return make_parking_sequence(6)


METHODS = {"Ours": ("SCHUR_CONDITION_NUMBER", "PRECONDITIONED_CG"), "ME-TSVD": ("FULL_EVD_MIN_EIGENVALUE", "TRUNCATED_SVD"),
           "FCN-SR": ("FULL_SVD_CONDITION", "STANDARD_REGULARIZATION")}


def pk01_params(method="Ours", **over):
    """icp_pk01.yaml: radius 0.5, 30 iterations, ROT 1e-5 / TRANS 1e-3; kappa_target 10."""
    from dcreg_b200 import default_params
    det, hand = METHODS[method]
    kw = dict(search_radius=0.5, max_iterations=30, conv_thresh_rot=1e-5, conv_thresh_trans=1e-3, kappa_target=10.0,
              detection=det, handling=hand)
    kw.update(over)
    return default_params(**kw)


def log_bytes(rec):
    """An iteration record without its wall-clock field."""
    from dcreg_b200.api import IterLog
    c = IterLog.from_buffer_copy(rec)
    c.iter_time_ms = 0.0
    return bytes(c)


def single(ctx, gp, scan, T0, want_log=True):
    ctx.set_source(scan)
    return ctx.icp_run(gp, T0, want_log=want_log)


def assert_same_run(b, s, tol=1e-8):
    assert b.status == s.status and b.converged == s.converged and b.iterations == s.iterations
    assert o.se3_log_distance(s.T, b.T) < tol
    assert len(b.logs) == len(s.logs)
    for x, y in zip(b.logs, s.logs):
        assert x.n_effective == y.n_effective and x.n_corr_pt == y.n_corr_pt
        assert list(x.analysis.degenerate_mask) == list(y.analysis.degenerate_mask)
        assert x.analysis.pcg_iterations == y.analysis.pcg_iterations


def assert_bitwise(a, b):
    assert a.status == b.status and a.converged == b.converged and a.iterations == b.iterations
    assert np.array_equal(a.T, b.T)
    assert [log_bytes(x) for x in a.logs] == [log_bytes(y) for y in b.logs]


@pytest.mark.parametrize("method,use_wd", [("Ours", 0), ("Ours", 1), ("ME-TSVD", 0), ("FCN-SR", 0)])
def test_each_scan_equals_a_single_run(ctx, seq, method, use_wd):
    """Ours folds the solve step into the iteration kernel; the baseline methods take the separate solve kernel, which
    reads the per-scan lever arm too."""
    scans, tgt, _, T_init = seq
    gp = pk01_params(method, use_weight_derivative=use_wd)
    ctx.set_target(tgt, 0.5)
    batch = ctx.icp_run_scans(gp, scans, T_init, want_log=True)
    assert len(batch) == len(scans)
    for b, scan, T0 in zip(batch, scans, T_init):
        assert_same_run(b, single(ctx, gp, scan, T0))
        assert all(abs(L.fitness * len(scan) - L.n_corr_pt) < 1e-6 * len(scan) for L in b.logs)   # over its own count
    assert sum(b.converged for b in batch) >= len(scans) // 2


def test_one_scan_call_is_a_single_run(ctx, seq):
    scans, tgt, _, T_init = seq
    gp = pk01_params()
    ctx.set_target(tgt, 0.5)
    for k in (0, 3):
        b, = ctx.icp_run_scans(gp, [scans[k]], T_init[k:k + 1], want_log=True)
        assert_bitwise(b, single(ctx, gp, scans[k], T_init[k]))


def test_scans_match_the_c_oracle(ctx, seq):
    """Four frames of the sequence against the C oracle, as the C3 test does for one pair."""
    import dcreg_oracle_c as oc
    scans, tgt, _, T_init = seq
    gp = pk01_params()
    ctx.set_target(tgt, 0.5)
    batch = ctx.icp_run_scans(gp, scans[:4], T_init[:4], want_log=True)
    cp = oc.make_params(search_radius=0.5, max_iterations=30, conv_rot=1e-5, conv_trans=1e-3, kappa_target=10.0)
    for b, scan, T0 in zip(batch, scans[:4], T_init[:4]):
        sc = oc.Scene(scan, tgt)
        st, conv, n_it, Tc, clogs = sc.icp_run(cp, T0)
        sc.close()
        assert b.status == st and b.converged == conv and b.iterations == n_it
        for C_, G in zip(clogs, b.logs):
            assert G.n_effective == C_.n_eff and G.n_corr_pt == C_.n_pt
            assert list(G.analysis.degenerate_mask) == list(C_.mask)
            assert np.allclose(G.analysis.np("lambda_schur_rot"), C_.lam_schur_rot, rtol=1e-8)
            assert np.allclose(G.analysis.np("lambda_schur_trans"), C_.lam_schur_trans, rtol=1e-8)
        assert o.se3_log_distance(Tc, b.T) < 1e-6


def test_permuting_scans_permutes_results_and_calls_reproduce(ctx, seq):
    scans, tgt, _, T_init = seq
    gp = pk01_params()
    ctx.set_target(tgt, 0.5)
    base = ctx.icp_run_scans(gp, scans, T_init, want_log=True)
    again = ctx.icp_run_scans(gp, scans, T_init, want_log=True)
    for a, b in zip(base, again):
        assert_bitwise(a, b)
    perm = [4, 0, 5, 2, 1, 3]
    moved = ctx.icp_run_scans(gp, [scans[p] for p in perm], T_init[perm], want_log=True)
    for j, p in enumerate(perm):
        assert_bitwise(moved[j], base[p])


def test_ragged_sizes_and_a_scan_too_small_to_register(ctx):
    """Scans of 1, 31, 32, 33, 257 and 20 000 points (more than 64 full tiles) in one batch.  The one-point scan aborts
    with NOT_ENOUGH_POINTS on its own; the others are exactly what they are without it."""
    from dcreg_b200.api import NOT_ENOUGH_POINTS
    from dcreg_b200.scenes import make_parking_sequence
    scans, tgt, _, T_init = make_parking_sequence(6, seed=48, min_points=20_000, max_points=20_000)
    rng = np.random.default_rng(3)
    sizes = [1, 31, 32, 33, 257, 20_000]
    batch_scans = [scans[k][np.sort(rng.choice(len(scans[k]), n, replace=False))] for k, n in enumerate(sizes)]
    gp = pk01_params()
    ctx.set_target(tgt, 0.5)
    batch = ctx.icp_run_scans(gp, batch_scans, T_init, want_log=True)
    assert batch[0].status == NOT_ENOUGH_POINTS and not batch[0].converged
    assert batch[-1].status == 0 and batch[-1].converged
    for b, scan, T0 in zip(batch, batch_scans, T_init):
        assert_same_run(b, single(ctx, gp, scan, T0))
    without = ctx.icp_run_scans(gp, batch_scans[1:], T_init[1:], want_log=True)
    for a, b in zip(without, batch[1:]):
        assert_bitwise(a, b)
    ctx.icp_run_scans(gp, batch_scans, T_init)
    assert np.array_equal(ctx.last_covariances(len(sizes))[0], 1e6 * np.eye(6))        # not converged: 1e6 * I


def test_context_source_is_untouched(ctx, seq):
    scans, tgt, _, T_init = seq
    gp = pk01_params()
    ctx.set_target(tgt, 0.5)
    before = single(ctx, gp, scans[2], T_init[2])
    ctx.icp_run_scans(gp, scans, T_init, want_log=True)
    after = ctx.icp_run(gp, T_init[2], want_log=True)
    assert_bitwise(after, before)


def test_covariances(ctx, seq, cylinder):
    scans, tgt, _, T_init = seq
    gp = pk01_params()
    ctx.set_target(tgt, 0.5)
    res = ctx.icp_run_scans(gp, scans, T_init)
    covs = ctx.last_covariances(len(scans))
    assert covs.shape == (len(scans), 6, 6)
    assert any(r.converged for r in res)
    for r, cov, scan, T0 in zip(res, covs, scans, T_init):
        s = single(ctx, gp, scan, T0, want_log=False)
        ref = ctx.last_covariance()
        assert s.converged == r.converged
        assert np.max(np.abs(cov - ref)) <= 1e-6 * np.max(np.abs(ref))
    # after a single run: trial 0, bit for bit; more than one trial is refused
    assert np.array_equal(ctx.last_covariances(1)[0], ctx.last_covariance())
    from dcreg_b200.api import DcregError
    with pytest.raises(DcregError):
        ctx.last_covariances(2)
    # after a batch of trials: one matrix per trial
    from dcreg_b200 import default_params
    from dcreg_b200.scenes import trial_poses
    ctx.set_target(cylinder, 1.0)
    ctx.set_source(cylinder)
    Ts = trial_poses(5, seed=46, max_trans=0.3, max_rot_deg=1.0)
    bres = ctx.icp_run_batch(default_params(kappa_target=10.0), Ts)
    bcov = ctx.last_covariances(5)
    assert bcov.shape == (5, 6, 6) and np.array_equal(bcov[0], ctx.last_covariance())
    for r, c in zip(bres, bcov):
        assert r.converged == (not np.array_equal(c, 1e6 * np.eye(6)))
    with pytest.raises(DcregError):
        ctx.last_covariances(6)


def _raw_call(ctx, gp, n_scans, xyz, stride, off, T, T_out=True):
    T_out_arr = np.empty((max(n_scans, 1), 4, 4)) if T_out else None
    dp = C.POINTER(C.c_double)
    return ctx.lib.dcreg_icp_run_scans(
        ctx._h, C.byref(gp) if gp is not None else None, n_scans,
        xyz.ctypes.data_as(C.POINTER(C.c_float)) if xyz is not None else None, stride,
        off.ctypes.data_as(C.POINTER(C.c_int64)) if off is not None else None,
        T.ctypes.data_as(dp) if T is not None else None,
        T_out_arr.ctypes.data_as(dp) if T_out else None, None, None, None, None, 0)


def test_bad_arguments(ctx, seq):
    from dcreg_b200 import Context
    from dcreg_b200.api import BAD_ARG, DcregError
    scans, tgt, _, T_init = seq
    gp = pk01_params()
    ctx.set_target(tgt, 0.5)
    xyz = np.ascontiguousarray(scans[0][:100]); off = np.array([0, 60, 100], dtype=np.int64); T2 = np.ascontiguousarray(T_init[:2])

    def refused(rc, what):
        assert rc == BAD_ARG and what in ctx.lib.dcreg_last_error(ctx._h).decode()

    assert _raw_call(ctx, gp, 2, xyz, 3, off, T2) == 0                                   # the well-formed call runs
    refused(_raw_call(ctx, None, 2, xyz, 3, off, T2), "null pointer")
    refused(_raw_call(ctx, gp, 2, None, 3, off, T2), "null pointer")
    refused(_raw_call(ctx, gp, 2, xyz, 3, None, T2), "null pointer")
    refused(_raw_call(ctx, gp, 2, xyz, 3, off, None), "null pointer")
    refused(_raw_call(ctx, gp, 2, xyz, 3, off, T2, T_out=False), "null pointer")
    refused(_raw_call(ctx, gp, 0, xyz, 3, off, T2), "n_scans")
    refused(_raw_call(ctx, gp, 65536, xyz, 3, off, T2), "n_scans")
    refused(_raw_call(ctx, gp, 2, xyz, 2, off, T2), "stride")
    refused(_raw_call(ctx, gp, 2, xyz, 3, np.array([1, 60, 100], dtype=np.int64), T2), "scan_offsets[0]")
    refused(_raw_call(ctx, gp, 2, xyz, 3, np.array([0, 60, 60], dtype=np.int64), T2), "empty")
    refused(_raw_call(ctx, gp, 2, xyz, 3, np.array([0, 70, 60], dtype=np.int64), T2), "empty")
    refused(_raw_call(ctx, gp, 1, xyz, 3, np.array([0, 0x20000000], dtype=np.int64), T2), "0x1fffffff")
    refused(_raw_call(ctx, pk01_params(weight_gate=1.5), 2, xyz, 3, off, T2), "weight_gate")
    with pytest.raises(DcregError):                                                     # through the binding
        ctx.icp_run_scans(gp, [scans[0], np.zeros((0, 3), np.float32)], T_init[:2])
    with pytest.raises(ValueError):
        ctx.icp_run_scans(gp, scans[:2], T_init[:3])
    # no target / a hash-grid target
    with Context(0) as c2:
        refused_c2 = c2.lib.dcreg_icp_run_scans(c2._h, C.byref(gp), 2, xyz.ctypes.data_as(C.POINTER(C.c_float)), 3,
                                                off.ctypes.data_as(C.POINTER(C.c_int64)), T2.ctypes.data_as(C.POINTER(C.c_double)),
                                                np.empty((2, 4, 4)).ctypes.data_as(C.POINTER(C.c_double)),
                                                None, None, None, None, 0)
        assert refused_c2 == BAD_ARG and "Target" in c2.lib.dcreg_last_error(c2._h).decode()
        far = np.array([[0, 0, 0], [3000, 3000, 3000], [1, 0, 0]], dtype=np.float32)       # > 2^27 cells: hash grid
        c2.set_target(far, 1.0)
        with pytest.raises(DcregError, match="dense target grid"):
            c2.icp_run_scans(gp, [far, far], np.stack([np.eye(4)] * 2))


def test_sharded_context_refuses_scans(seq):
    """Scans are independent registrations: the caller distributes them over ranks (here: a one-rank communicator)."""
    from dcreg_b200 import Context
    from dcreg_b200.api import DcregError
    scans, tgt, _, T_init = seq
    with Context(0) as c:
        c.set_target(tgt, 0.5)
        try:
            c.comm_init(c.comm_unique_id(), 0, 1)
        except DcregError as e:
            pytest.skip(f"no NCCL communicator on this machine: {e}")
        with pytest.raises(DcregError, match="distribute them over ranks"):
            c.icp_run_scans(pk01_params(), scans[:2], T_init[:2])
        c.comm_destroy()


def test_scans_cut_from_the_shipped_cylinder(ctx, cylinder):
    """Scans cut from the shipped cylinder (cell 1.0, the G2 setup) with a log: counts identical to single runs; the
    tiny scans do not disturb the large one."""
    from dcreg_b200 import default_params
    from dcreg_b200.scenes import g2_initial_pose
    gp = default_params(kappa_target=10.0, max_iterations=30)
    ctx.set_target(cylinder, 1.0)
    rng = np.random.default_rng(9)
    scans = [cylinder, cylinder[rng.choice(len(cylinder), 5, replace=False)], cylinder[::3]]
    T0 = g2_initial_pose()
    Ts = np.stack([T0, T0, o.pose6d_to_matrix(0.1, -0.2, 0.1, 0.0, math.radians(0.5), math.radians(-1.0))])
    batch = ctx.icp_run_scans(gp, scans, Ts, want_log=True)
    for b, s, T in zip(batch, scans, Ts):
        assert_same_run(b, single(ctx, gp, s, T))
    assert batch[1].status == 1 and batch[0].converged and batch[2].converged
