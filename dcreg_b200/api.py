"""ctypes host binding of include/dcreg_b200.h.

Mirrors the reference's operator interface for the hot path (names, argument meaning, error
behaviour) so the parity tests read like the reference's own call sites:

  reference (C++)                                            here
  ---------------------------------------------------------  ----------------------------------
  ICPContext::setTargetCloud          utils.hpp:393-424       Context.set_target
  TestRunner::Point2PlaneICP_SO3_OpenMP  icp_test_runner.h:92  Context.Point2PlaneICP_SO3 / icp_run
  DCReg::analyzeDegeneracy + solveDegenerateSystem
                                      dcreg.hpp:45-264        Context.analyze_and_solve
  DCReg::solvePCG                     dcreg.hpp:279-283       Context.solve_pcg
  SymmetricHessianComputer            hessian_computer.h:62   Context.reduce_normal_equations

There is NO CPU fallback: if the CUDA library is missing or no GPU is visible the calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libdcreg_b200.so")

# ---- enums (DCReg/include/utils.hpp:106-121) ----
DET = {"NONE_DETE": 0, "SCHUR_CONDITION_NUMBER": 1, "FULL_EVD_MIN_EIGENVALUE": 2,
       "EVD_SUB_CONDITION": 3, "FULL_SVD_CONDITION": 4}
HAND = {"NONE_HAND": 0, "STANDARD_REGULARIZATION": 1, "ADAPTIVE_REGULARIZATION": 2,
        "PRECONDITIONED_CG": 3, "SOLUTION_REMAPPING": 4, "TRUNCATED_SVD": 5}
STATUS = {0: "OK", 1: "NOT_ENOUGH_POINTS", 2: "NONFINITE_UPDATE", 3: "SINGULAR_BLOCK", 4: "CUDA_ERROR",
          5: "NCCL_ERROR", 6: "BAD_ARG", 7: "NO_DEVICE"}
OK, NOT_ENOUGH_POINTS, NONFINITE_UPDATE, SINGULAR_BLOCK, CUDA_ERROR, NCCL_ERROR, BAD_ARG, NO_DEVICE = range(8)


class IcpParams(C.Structure):
    _fields_ = [
        ("search_radius", C.c_double), ("max_iterations", C.c_int32), ("detection", C.c_int32),
        ("handling", C.c_int32), ("use_weight_derivative", C.c_int32),
        ("conv_thresh_rot", C.c_double), ("conv_thresh_trans", C.c_double),
        ("cond_thresh", C.c_double), ("eig_thresh", C.c_double), ("kappa_target", C.c_double),
        ("pcg_tol", C.c_double), ("pcg_max_iter", C.c_int32), ("reserved0", C.c_int32),
        ("std_reg_gamma", C.c_double), ("plane_thickness", C.c_double), ("weight_slope", C.c_double),
        ("weight_gate", C.c_double), ("min_normal_norm", C.c_double),
        ("min_effective_points", C.c_int32), ("fixed_iterations", C.c_int32),
    ]


class Analysis(C.Structure):
    _fields_ = [
        ("is_degenerate", C.c_int32), ("degenerate_mask", C.c_int32 * 6), ("pcg_iterations", C.c_int32),
        ("cond_schur_rot", C.c_double), ("cond_schur_trans", C.c_double),
        ("cond_diag_rot", C.c_double), ("cond_diag_trans", C.c_double), ("cond_full", C.c_double),
        ("cond_full_sub_rot", C.c_double), ("cond_full_sub_trans", C.c_double),
        ("eigenvalues_full", C.c_double * 6), ("singular_values", C.c_double * 6),
        ("lambda_schur_rot", C.c_double * 3), ("lambda_schur_trans", C.c_double * 3),
        ("lambda_sub_rot", C.c_double * 3), ("lambda_sub_trans", C.c_double * 3),
        ("schur_V_rot", C.c_double * 9), ("schur_V_trans", C.c_double * 9),
        ("aligned_V_rot", C.c_double * 9), ("aligned_V_trans", C.c_double * 9),
        ("rot_indices", C.c_int32 * 3), ("trans_indices", C.c_int32 * 3), ("schur_singular", C.c_int32),
        ("reserved1", C.c_int32), ("P_preconditioner", C.c_double * 36), ("W_adaptive", C.c_double * 36),
        ("pcg_residual", C.c_double),
    ]

    def np(self, name):
        return np.array(getattr(self, name))


class IterLog(C.Structure):
    _fields_ = [
        ("iter", C.c_int32), ("status", C.c_int32), ("n_effective", C.c_int32), ("n_corr_pt", C.c_int32),
        ("rmse", C.c_double), ("fitness", C.c_double), ("objective", C.c_double), ("iter_time_ms", C.c_double),
        ("gradient", C.c_double * 6), ("H27", C.c_double * 27), ("dx", C.c_double * 6), ("T", C.c_double * 16),
        ("analysis", Analysis),
    ]


PLANE_CALLBACK = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double),
                             C.POINTER(C.c_int64))

_lib = None

# every symbol include/dcreg_b200.h declares (checked by tests/test_abi.py)
EXPORTS = [
    "dcreg_abi_version", "dcreg_create", "dcreg_destroy", "dcreg_last_error", "dcreg_default_params",
    "dcreg_stream", "dcreg_set_source", "dcreg_set_target", "dcreg_find_planes",
    "dcreg_reduce_normal_equations", "dcreg_reduce_normal_equations_f64plane",
    "dcreg_reduce_normal_equations_host", "dcreg_analyze_and_solve", "dcreg_solve_pcg", "dcreg_icp_run",
    "dcreg_icp_run_batch", "dcreg_icp_run_scans", "dcreg_icp_enqueue", "dcreg_icp_fetch", "dcreg_icp_run_host_planes", "dcreg_comm_mode", "dcreg_last_covariance", "dcreg_last_covariances", "dcreg_point_to_point_metrics", "dcreg_point_to_point_metrics_batch", "dcreg_comm_unique_id", "dcreg_comm_init",
    "dcreg_comm_destroy", "dcreg_set_global_source_count", "dcreg_launch_count", "dcreg_device_source",
    "dcreg_device_planes_f64", "dcreg_device_planes_f32", "dcreg_freeze_planes_f32", "dcreg_time_reduce", "dcreg_time_iteration", "dcreg_iteration_counters", "dcreg_iteration_timeline",
]


def load_library():
    """dlopen the in-tree CUDA library.  Raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m dcreg_b200.build` "
            "(__graft_entry__.build()).  dcreg_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    dp, vp, i64, ci = C.POINTER(C.c_double), C.c_void_p, C.c_int64, C.c_int
    lib.dcreg_abi_version.restype = ci
    lib.dcreg_create.argtypes = [ci, C.POINTER(vp)]
    lib.dcreg_destroy.argtypes = [vp]
    lib.dcreg_last_error.argtypes = [vp]; lib.dcreg_last_error.restype = C.c_char_p
    lib.dcreg_default_params.argtypes = [C.POINTER(IcpParams)]; lib.dcreg_default_params.restype = None
    lib.dcreg_stream.argtypes = [vp]; lib.dcreg_stream.restype = vp
    lib.dcreg_set_source.argtypes = [vp, C.POINTER(C.c_float), i64, ci]
    lib.dcreg_set_target.argtypes = [vp, C.POINTER(C.c_float), i64, ci, C.c_double]
    lib.dcreg_find_planes.argtypes = [vp, dp, C.c_double, dp, C.POINTER(i64)]
    lib.dcreg_reduce_normal_equations.argtypes = [vp, vp, vp, i64, dp, ci, dp, dp]
    lib.dcreg_reduce_normal_equations_f64plane.argtypes = [vp, vp, vp, i64, dp, ci, dp, dp]
    lib.dcreg_reduce_normal_equations_host.argtypes = [vp, C.POINTER(C.c_float), vp, ci, i64, dp, ci, dp, dp]
    lib.dcreg_analyze_and_solve.argtypes = [vp, dp, C.POINTER(IcpParams), C.POINTER(Analysis), dp]
    lib.dcreg_solve_pcg.argtypes = [vp, dp, dp, dp, ci, C.c_double, dp, C.POINTER(ci)]
    lib.dcreg_icp_run.argtypes = [vp, C.POINTER(IcpParams), dp, dp, C.POINTER(IterLog), ci, C.POINTER(ci),
                                  C.POINTER(ci)]
    lib.dcreg_icp_run_batch.argtypes = [vp, C.POINTER(IcpParams), ci, dp, dp, C.POINTER(ci), C.POINTER(ci), C.POINTER(ci),
                                        C.POINTER(IterLog), ci]
    lib.dcreg_icp_run_scans.argtypes = [vp, C.POINTER(IcpParams), ci, C.POINTER(C.c_float), ci, C.POINTER(i64), dp, dp,
                                        C.POINTER(ci), C.POINTER(ci), C.POINTER(ci), C.POINTER(IterLog), ci]
    lib.dcreg_comm_mode.argtypes = [vp]
    lib.dcreg_icp_enqueue.argtypes = [vp, C.POINTER(IcpParams), dp]
    lib.dcreg_icp_fetch.argtypes = [vp, dp, C.POINTER(ci), C.POINTER(ci)]
    lib.dcreg_icp_run_host_planes.argtypes = [vp, C.POINTER(IcpParams), dp, PLANE_CALLBACK, vp, dp,
                                              C.POINTER(IterLog), ci, C.POINTER(ci), C.POINTER(ci)]
    lib.dcreg_last_covariance.argtypes = [vp, dp]
    lib.dcreg_last_covariances.argtypes = [vp, ci, dp]
    lib.dcreg_point_to_point_metrics.argtypes = [vp, dp, C.c_double, dp]
    lib.dcreg_point_to_point_metrics_batch.argtypes = [vp, ci, dp, C.c_double, dp]
    lib.dcreg_comm_unique_id.argtypes = [vp, C.POINTER(C.c_uint8)]
    lib.dcreg_comm_init.argtypes = [vp, C.POINTER(C.c_uint8), ci, ci]
    lib.dcreg_comm_destroy.argtypes = [vp]
    lib.dcreg_set_global_source_count.argtypes = [vp, i64]
    lib.dcreg_launch_count.argtypes = [vp]; lib.dcreg_launch_count.restype = i64
    for nm in ("dcreg_device_source", "dcreg_device_planes_f64", "dcreg_device_planes_f32"):
        getattr(lib, nm).argtypes = [vp]; getattr(lib, nm).restype = vp
    lib.dcreg_freeze_planes_f32.argtypes = [vp]
    lib.dcreg_time_reduce.argtypes = [vp, ci, dp, ci, ci, ci, C.POINTER(C.c_float)]
    lib.dcreg_time_iteration.argtypes = [vp, C.POINTER(IcpParams), dp, ci, ci, C.POINTER(C.c_float)]
    lib.dcreg_iteration_counters.argtypes = [vp, ci, C.POINTER(C.c_uint64)]
    lib.dcreg_iteration_timeline.argtypes = [vp, C.POINTER(IcpParams), dp, ci, C.POINTER(C.c_uint64), ci, C.POINTER(ci)]
    _lib = lib
    return lib


def default_params(**overrides) -> IcpParams:
    p = IcpParams()
    load_library().dcreg_default_params(C.byref(p))
    for k, v in overrides.items():
        if k == "detection" and isinstance(v, str):
            v = DET[v]
        if k == "handling" and isinstance(v, str):
            v = HAND[v]
        if not hasattr(p, k):
            raise AttributeError(k)
        setattr(p, k, v)
    return p


class DcregError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__(f"dcreg status {status} ({STATUS.get(status, '?')}): {msg}")
        self.status = status


def _dptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _as_points(xyz):
    a = np.ascontiguousarray(xyz, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] < 3:
        raise ValueError("points must be (N, >=3)")
    return a


def pose_Rt(T):
    T = np.asarray(T, dtype=np.float64)
    return np.ascontiguousarray(np.concatenate([T[:3, :3].reshape(-1), T[:3, 3]]))


def pack_scans(scans):
    """A list of (N_i, >=3) point arrays -> (xyz (sum N_i, 3) float32, offsets (n + 1,) int64): scan i is
    xyz[offsets[i]:offsets[i + 1]], the layout dcreg_icp_run_scans takes.  Columns past the third are dropped."""
    parts = [_as_points(s)[:, :3] for s in scans]
    if not parts:
        raise ValueError("no scans")
    offsets = np.zeros(len(parts) + 1, dtype=np.int64)
    offsets[1:] = np.cumsum([p.shape[0] for p in parts])
    return np.ascontiguousarray(np.concatenate(parts, axis=0), dtype=np.float32), offsets


def _batch_results(B, T_out, n_it, conv, st, logs, cap):
    out = []
    for b in range(B):
        recs = []
        if logs is not None:
            nrec = min(n_it[b], cap)
            if st[b] == NONFINITE_UPDATE and n_it[b] < cap:
                nrec = n_it[b] + 1
            recs = [logs[b * cap + i] for i in range(nrec)]
        out.append(IcpResult(int(st[b]), bool(conv[b]), int(n_it[b]), T_out[b], recs))
    return out


class IcpResult:
    def __init__(self, status, converged, iterations, T, logs):
        self.status, self.converged, self.iterations, self.T, self.logs = status, converged, iterations, T, logs


class Context:
    """One engine context per GPU (owns the stream, device buffers and the optional NCCL comm)."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        self._h = C.c_void_p()
        rc = self.lib.dcreg_create(device, C.byref(self._h))
        if rc != OK:
            msg = self.lib.dcreg_last_error(self._h).decode() if self._h else "no CUDA device"
            if self._h:
                self.lib.dcreg_destroy(self._h)
            self._h = None
            raise DcregError(rc, msg)
        self.n_source = 0

    # -- lifetime --
    def close(self):
        if getattr(self, "_h", None):
            self.lib.dcreg_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc, allow=()):
        if rc != OK and rc not in allow:
            raise DcregError(rc, self.lib.dcreg_last_error(self._h).decode())
        return rc

    @property
    def stream(self) -> int:
        return int(self.lib.dcreg_stream(self._h) or 0)

    @property
    def launch_count(self) -> int:
        return int(self.lib.dcreg_launch_count(self._h))

    # -- clouds --
    def set_source(self, xyz):
        a = _as_points(xyz)
        self._check(self.lib.dcreg_set_source(self._h, a.ctypes.data_as(C.POINTER(C.c_float)), a.shape[0], a.shape[1]))
        self.n_source = a.shape[0]

    def set_target(self, xyz, cell_size: float):
        a = _as_points(xyz)
        self._check(self.lib.dcreg_set_target(self._h, a.ctypes.data_as(C.POINTER(C.c_float)), a.shape[0], a.shape[1],
                                              float(cell_size)))

    # -- seams --
    def find_planes(self, T, search_radius: float, want_planes: bool = True):
        T = np.ascontiguousarray(T, dtype=np.float64)
        planes = np.empty((self.n_source, 4), dtype=np.float64) if want_planes else None
        npt = C.c_int64(0)
        self._check(self.lib.dcreg_find_planes(self._h, _dptr(T), float(search_radius),
                                               _dptr(planes) if want_planes else None, C.byref(npt)))
        return planes, int(npt.value)

    def reduce_normal_equations(self, src4, plane4, T, use_weight_derivative: bool):
        """Host arrays in, (out27, stats) out.  plane4 dtype float32 -> 32 B/slot, float64 -> 48 B/slot."""
        src4 = np.ascontiguousarray(src4, dtype=np.float32)
        assert src4.ndim == 2 and src4.shape[1] == 4
        plane4 = np.ascontiguousarray(plane4)
        is64 = plane4.dtype == np.float64
        if not is64:
            plane4 = plane4.astype(np.float32, copy=False)
        out = np.empty(27); stats = np.empty(3)
        prt = pose_Rt(T)
        self._check(self.lib.dcreg_reduce_normal_equations_host(
            self._h, src4.ctypes.data_as(C.POINTER(C.c_float)), plane4.ctypes.data_as(C.c_void_p), int(is64),
            src4.shape[0], _dptr(prt), int(bool(use_weight_derivative)), _dptr(out), _dptr(stats)))
        self.n_source = src4.shape[0]
        return out, stats

    def reduce_device(self, plane_is_f64: bool, T, use_weight_derivative: bool):
        """K1 over the ctx-resident source + planes (after find_planes / freeze_planes_f32)."""
        out = np.empty(27); stats = np.empty(3)
        prt = pose_Rt(T)
        fn = self.lib.dcreg_reduce_normal_equations_f64plane if plane_is_f64 else self.lib.dcreg_reduce_normal_equations
        planes = self.lib.dcreg_device_planes_f64(self._h) if plane_is_f64 else self.lib.dcreg_device_planes_f32(self._h)
        self._check(fn(self._h, self.lib.dcreg_device_source(self._h), planes, self.n_source, _dptr(prt),
                       int(bool(use_weight_derivative)), _dptr(out), _dptr(stats)))
        return out, stats

    def freeze_planes_f32(self):
        self._check(self.lib.dcreg_freeze_planes_f32(self._h))

    def time_reduce(self, plane_is_f64: bool, T, use_weight_derivative: bool, reps: int, flush_l2: bool) -> float:
        ms = C.c_float(0)
        prt = pose_Rt(T)
        self._check(self.lib.dcreg_time_reduce(self._h, int(plane_is_f64), _dptr(prt), int(bool(use_weight_derivative)),
                                               reps, int(flush_l2), C.byref(ms)))
        return float(ms.value)

    def time_iteration(self, params: IcpParams, T, what: int, reps: int) -> float:
        ms = C.c_float(0)
        T = np.ascontiguousarray(T, dtype=np.float64)
        self._check(self.lib.dcreg_time_iteration(self._h, C.byref(params), _dptr(T), int(what), int(reps), C.byref(ms)))
        return float(ms.value)

    def iteration_timeline(self, params: IcpParams, T, iters: int):
        """Phase time stamps (ns) of the last of `iters` real iterations from pose T: (blocks (n, 16), solve (16,))."""
        T = np.ascontiguousarray(T, dtype=np.float64)
        cap = 4096
        out = np.zeros((cap, 16), dtype=np.uint64)
        nb = C.c_int(0)
        self._check(self.lib.dcreg_iteration_timeline(self._h, C.byref(params), _dptr(T), int(iters),
                                                      out.ctypes.data_as(C.POINTER(C.c_uint64)), cap, C.byref(nb)))
        return out[:nb.value].astype(np.int64), out[nb.value].astype(np.int64)

    def iteration_counters(self, enable: bool = True):
        out = (C.c_uint64 * 2)()
        self._check(self.lib.dcreg_iteration_counters(self._h, int(enable), out))
        return int(out[0]), int(out[1])

    def analyze_and_solve(self, H27, params: IcpParams):
        """DCReg::analyzeDegeneracy + solveDegenerateSystem on the device.  Returns (Analysis, dx, status)."""
        H27 = np.ascontiguousarray(H27, dtype=np.float64)
        a = Analysis(); dx = np.empty(6)
        rc = self._check(self.lib.dcreg_analyze_and_solve(self._h, _dptr(H27), C.byref(params), C.byref(a), _dptr(dx)),
                         allow=(NONFINITE_UPDATE,))
        return a, dx, rc

    def solve_pcg(self, A, b, P, max_iterations: int, tolerance: float):
        A = np.ascontiguousarray(A, dtype=np.float64); b = np.ascontiguousarray(b, dtype=np.float64)
        P = np.ascontiguousarray(P, dtype=np.float64)
        x = np.empty(6); it = C.c_int(0)
        self._check(self.lib.dcreg_solve_pcg(self._h, _dptr(A), _dptr(b), _dptr(P), max_iterations, tolerance,
                                             _dptr(x), C.byref(it)))
        return x, int(it.value)

    # -- outer loop --
    def icp_run(self, params: IcpParams, T_init, want_log: bool = True) -> IcpResult:
        """TestRunner::Point2PlaneICP_SO3_OpenMP (icp_test_runner.cpp:1611-2060), device correspondences."""
        T_init = np.ascontiguousarray(T_init, dtype=np.float64)
        T_out = np.empty((4, 4))
        cap = int(params.max_iterations) if want_log else 0
        logs = (IterLog * max(cap, 1))()
        n_it = C.c_int(0); conv = C.c_int(0)
        rc = self._check(self.lib.dcreg_icp_run(self._h, C.byref(params), _dptr(T_init), _dptr(T_out),
                                                logs if want_log else None, cap, C.byref(n_it), C.byref(conv)),
                         allow=(NOT_ENOUGH_POINTS, NONFINITE_UPDATE))
        nrec = min(n_it.value, cap)
        return IcpResult(rc, bool(conv.value), n_it.value, T_out, [logs[i] for i in range(nrec)])

    Point2PlaneICP_SO3 = icp_run

    def icp_enqueue(self, params: IcpParams, T_init):
        """Put a whole run on the context's stream without any host synchronisation (see icp_fetch)."""
        T_init = np.ascontiguousarray(T_init, dtype=np.float64)
        self._check(self.lib.dcreg_icp_enqueue(self._h, C.byref(params), _dptr(T_init)))

    def icp_fetch(self) -> IcpResult:
        """Wait for the stream; pose / iteration count / flags of the last enqueued run."""
        T_out = np.empty((4, 4)); n_it = C.c_int(0); conv = C.c_int(0)
        rc = self._check(self.lib.dcreg_icp_fetch(self._h, _dptr(T_out), C.byref(n_it), C.byref(conv)),
                         allow=(NOT_ENOUGH_POINTS, NONFINITE_UPDATE))
        return IcpResult(rc, bool(conv.value), n_it.value, T_out, [])

    def icp_run_batch(self, params: IcpParams, T_init, want_log: bool = False):
        """`num_runs` registrations side by side (icp_test_runner.cpp:331-345): T_init (B, 4, 4).
        Returns a list of IcpResult, one per trial (logs only when want_log)."""
        T_init = np.ascontiguousarray(T_init, dtype=np.float64).reshape(-1, 4, 4)
        B = T_init.shape[0]
        T_out = np.empty((B, 4, 4))
        n_it = (C.c_int * B)(); conv = (C.c_int * B)(); st = (C.c_int * B)()
        cap = int(params.max_iterations) if want_log else 0
        logs = (IterLog * max(cap * B, 1))() if want_log else None
        self._check(self.lib.dcreg_icp_run_batch(self._h, C.byref(params), B, _dptr(T_init), _dptr(T_out), n_it, conv, st,
                                                 logs, cap))
        return _batch_results(B, T_out, n_it, conv, st, logs, cap)

    def icp_run_scans(self, params: IcpParams, scans, T_init, want_log: bool = False):
        """Many different scans against the context's target, side by side: scans = list of (N_i, >=3) arrays,
        T_init (n, 4, 4), one initial pose per scan.  Returns a list of IcpResult, one per scan (logs only when
        want_log).  The context's source (set_source) is left as it was."""
        xyz, offsets = pack_scans(scans)
        B = offsets.size - 1
        T_init = np.ascontiguousarray(T_init, dtype=np.float64).reshape(-1, 4, 4)
        if T_init.shape[0] != B:
            raise ValueError(f"{B} scans but {T_init.shape[0]} initial poses")
        T_out = np.empty((B, 4, 4))
        n_it = (C.c_int * B)(); conv = (C.c_int * B)(); st = (C.c_int * B)()
        cap = int(params.max_iterations) if want_log else 0
        logs = (IterLog * max(cap * B, 1))() if want_log else None
        self._check(self.lib.dcreg_icp_run_scans(self._h, C.byref(params), B, xyz.ctypes.data_as(C.POINTER(C.c_float)),
                                                 xyz.shape[1], offsets.ctypes.data_as(C.POINTER(C.c_int64)),
                                                 _dptr(T_init), _dptr(T_out), n_it, conv, st, logs, cap))
        return _batch_results(B, T_out, n_it, conv, st, logs, cap)

    def icp_run_host_planes(self, params: IcpParams, T_init, plane_fn, want_log: bool = True) -> IcpResult:
        """Same loop with caller-supplied correspondences: plane_fn(T 4x4) -> (planes (N,4) f64, n_corr_pt)."""
        T_init = np.ascontiguousarray(T_init, dtype=np.float64)
        T_out = np.empty((4, 4))
        cap = int(params.max_iterations) if want_log else 0
        logs = (IterLog * max(cap, 1))()
        n = self.n_source
        err = []

        def _cb(user, Tp, planes_p, npt_p):
            try:
                T = np.ctypeslib.as_array(Tp, shape=(16,)).reshape(4, 4).copy()
                planes, npt = plane_fn(T)
                dst = np.ctypeslib.as_array(planes_p, shape=(n * 4,))
                dst[:] = np.ascontiguousarray(planes, dtype=np.float64).reshape(-1)
                npt_p[0] = int(npt)
                return 0
            except Exception as e:  # pragma: no cover
                err.append(e)
                return 1

        cb = PLANE_CALLBACK(_cb)
        n_it = C.c_int(0); conv = C.c_int(0)
        rc = self.lib.dcreg_icp_run_host_planes(self._h, C.byref(params), _dptr(T_init), cb, None, _dptr(T_out),
                                                logs if want_log else None, cap, C.byref(n_it), C.byref(conv))
        if err:
            raise err[0]
        self._check(rc, allow=(NOT_ENOUGH_POINTS, NONFINITE_UPDATE))
        nrec = min(n_it.value, cap)
        return IcpResult(rc, bool(conv.value), n_it.value, T_out, [logs[i] for i in range(nrec)])

    def last_covariance(self):
        cov = np.empty((6, 6))
        self._check(self.lib.dcreg_last_covariance(self._h, _dptr(cov)))
        return cov

    def last_covariances(self, n: int):
        """Covariance of each of the first n trials of the last run (icp_run: 1; icp_run_batch / icp_run_scans: their
        count), shape (n, 6, 6)."""
        cov = np.empty((int(n), 6, 6))
        self._check(self.lib.dcreg_last_covariances(self._h, int(n), _dptr(cov)))
        return cov

    def point_to_point_metrics(self, T, error_threshold: float):
        """calculatePointToPointError on the device: returns dict(rmse, fitness, chamfer, n_valid)."""
        T = np.ascontiguousarray(T, dtype=np.float64)
        out = np.empty(4)
        self._check(self.lib.dcreg_point_to_point_metrics(self._h, _dptr(T), float(error_threshold), _dptr(out)))
        return {"rmse": out[0], "fitness": out[1], "chamfer": out[2], "n_valid": int(out[3])}

    def point_to_point_metrics_batch(self, T, error_threshold: float):
        """point_to_point_metrics for many poses in one call: T (n, 4, 4).  Returns dict of arrays rmse, fitness,
        chamfer (float64) and n_valid (int64), each (n,); row i equals point_to_point_metrics(T[i]) bit for bit."""
        T = np.ascontiguousarray(T, dtype=np.float64).reshape(-1, 4, 4)
        out = np.empty((T.shape[0], 4))
        self._check(self.lib.dcreg_point_to_point_metrics_batch(self._h, T.shape[0], _dptr(T), float(error_threshold),
                                                                _dptr(out)))
        return {"rmse": out[:, 0].copy(), "fitness": out[:, 1].copy(), "chamfer": out[:, 2].copy(),
                "n_valid": out[:, 3].astype(np.int64)}

    # -- multi-GPU --
    def comm_unique_id(self) -> bytes:
        buf = (C.c_uint8 * 128)()
        self._check(self.lib.dcreg_comm_unique_id(self._h, buf))
        return bytes(buf)

    def comm_init(self, unique_id: bytes, rank: int, nranks: int):
        buf = (C.c_uint8 * 128).from_buffer_copy(unique_id)
        self._check(self.lib.dcreg_comm_init(self._h, buf, rank, nranks))

    @property
    def comm_mode(self) -> int:
        """0 no communicator, 1 ncclAllReduce fallback, 2 in-kernel peer-memory all-reduce."""
        return int(self.lib.dcreg_comm_mode(self._h))

    def comm_destroy(self):
        self._check(self.lib.dcreg_comm_destroy(self._h))

    def set_global_source_count(self, n_total: int):
        self._check(self.lib.dcreg_set_global_source_count(self._h, int(n_total)))
