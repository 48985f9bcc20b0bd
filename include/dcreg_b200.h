/*
 * dcreg_b200.h - C ABI of the B200-native point-to-plane ICP + Schur-decoupled degeneracy engine.
 *
 * This is the drop-in boundary for ONE hot path of JokerJohn/DCReg (SURVEY.md §8b).  The
 * reference has no FFI layer; each entry point below names the C++ member / code block of the
 * reference it replaces (paths relative to the reference checkout).  Plain pointers and sizes
 * only: no torch, Eigen or PCL types cross this boundary.  Nothing here ever throws; every
 * function returns a dcreg_status and dcreg_last_error() holds the text.
 *
 * State-vector order everywhere: [wx wy wz | x y z] (rotation first, right perturbation),
 * as on the reference's SO(3) path (DCReg/src/icp_test_runner.cpp:1611-2060).
 * 4x4 / 3x3 / 6x6 matrices are ROW-major doubles.
 */
#ifndef DCREG_B200_H
#define DCREG_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DCREG_ABI_VERSION 2

/* -------------------------------------------------------------------------------------------
 * Status codes.  Reference convention: bool return + std::cerr text
 * (icp_test_runner.cpp:1635-1646, 1847-1854, 1942-1950; dcreg.hpp:259-262).
 * ----------------------------------------------------------------------------------------- */
typedef enum dcreg_status {
    DCREG_OK = 0,
    DCREG_NOT_ENOUGH_POINTS = 1,   /* < 10 effective correspondences (icp_test_runner.cpp:1847) */
    DCREG_NONFINITE_UPDATE = 2,    /* solver returned non-finite dx (icp_test_runner.cpp:1942)  */
    DCREG_SINGULAR_BLOCK = 3,      /* never RETURNED: the reference only warns when H_RR or H_tt is not invertible
                                      (icp_test_runner.cpp:2464) and carries on with cond = inf; the warning is
                                      surfaced per iteration as dcreg_analysis.schur_singular.  Value kept reserved. */
    DCREG_CUDA_ERROR = 4,
    DCREG_NCCL_ERROR = 5,
    DCREG_BAD_ARG = 6,
    DCREG_NO_DEVICE = 7            /* no CUDA device: the product has no CPU fallback            */
} dcreg_status;

/* DetectionMethod / HandlingMethod, DCReg/include/utils.hpp:106-121 (same order, same names). */
typedef enum dcreg_detection {
    DCREG_DET_NONE_DETE = 0,
    DCREG_DET_SCHUR_CONDITION_NUMBER = 1,
    DCREG_DET_FULL_EVD_MIN_EIGENVALUE = 2,
    DCREG_DET_EVD_SUB_CONDITION = 3,
    DCREG_DET_FULL_SVD_CONDITION = 4
} dcreg_detection;

typedef enum dcreg_handling {
    DCREG_HAND_NONE_HAND = 0,
    DCREG_HAND_STANDARD_REGULARIZATION = 1,
    DCREG_HAND_ADAPTIVE_REGULARIZATION = 2, /* parsed by the reference, no handler: plain QR */
    DCREG_HAND_PRECONDITIONED_CG = 3,
    DCREG_HAND_SOLUTION_REMAPPING = 4,
    DCREG_HAND_TRUNCATED_SVD = 5
} dcreg_handling;

/* -------------------------------------------------------------------------------------------
 * Parameters: POD mirror of ICPRunner::Config + ICPParameters
 * (DCReg/include/utils.hpp:82-103, 132-171), passed by pointer, no global state
 * (the reference re-sets them every iteration through DCReg::setConfig, dcreg.hpp:36-38).
 * dcreg_default_params() fills the reference defaults.
 * ----------------------------------------------------------------------------------------- */
typedef struct dcreg_icp_params {
    double search_radius;          /* icp.search_radius                       (1.0)   */
    int32_t max_iterations;        /* icp.max_iterations                      (30)    */
    int32_t detection;             /* dcreg_detection                                  */
    int32_t handling;              /* dcreg_handling                                   */
    int32_t use_weight_derivative; /* USE_WEIGHT_DERIVATIVE, icp_test_runner.cpp:1691 (0) */
    double conv_thresh_rot;        /* CONVERGENCE_THRESH_ROT                  (1e-5)  */
    double conv_thresh_trans;      /* CONVERGENCE_THRESH_TRANS                (1e-3)  */
    double cond_thresh;            /* DEGENERACY_THRES_COND                   (10)    */
    double eig_thresh;             /* DEGENERACY_THRES_EIG                    (120)   */
    double kappa_target;           /* KAPPA_TARGET                            (1)     */
    double pcg_tol;                /* PCG_TOLERANCE                           (1e-6)  */
    int32_t pcg_max_iter;          /* PCG_MAX_ITER                            (10)    */
    int32_t reserved0;
    double std_reg_gamma;          /* STD_REG_GAMMA                           (0.01)  */
    /* compile-time constants of the reference, exposed with the reference values */
    double plane_thickness;        /* 0.2   icp_test_runner.cpp:1772 */
    double weight_slope;           /* 0.9   icp_test_runner.cpp:1776: s = 1 - weight_slope |r|              */
    double weight_gate;            /* 0.1   icp_test_runner.cpp:1785: slot kept when s > weight_gate         */
    double min_normal_norm;        /* 1e-6  icp_test_runner.cpp:1750 */
    int32_t min_effective_points;  /* 10    icp_test_runner.cpp:1847 */
    int32_t fixed_iterations;      /* 1: ignore the convergence test and always run max_iterations
                                      (BASELINE config "50 ICP iterations"); default 0 */
} dcreg_icp_params;

/* POD mirror of DegeneracyAnalysisResult (DCReg/include/utils.hpp:427-448). */
typedef struct dcreg_analysis {
    int32_t is_degenerate;
    int32_t degenerate_mask[6];    /* eigen-index order (ascending lambda), NOT physical axes */
    int32_t pcg_iterations;        /* iterations the PCG solve used (0 when the direct solve ran) */
    double cond_schur_rot, cond_schur_trans;
    double cond_diag_rot, cond_diag_trans;
    double cond_full;
    double cond_full_sub_rot, cond_full_sub_trans;
    double eigenvalues_full[6];    /* ascending */
    double singular_values[6];     /* descending */
    double lambda_schur_rot[3], lambda_schur_trans[3];   /* ascending */
    double lambda_sub_rot[3], lambda_sub_trans[3];       /* diagonal blocks, ascending */
    double schur_V_rot[9], schur_V_trans[9];             /* eigenvectors in columns */
    double aligned_V_rot[9], aligned_V_trans[9];         /* paper Alg. 2 (log only) */
    int32_t rot_indices[3], trans_indices[3];
    int32_t schur_singular;        /* 1: H_tt or H_RR not invertible, Schur complements skipped (icp_test_runner.cpp:2464) */
    int32_t reserved1;
    double P_preconditioner[36];   /* paper Eq. 43-46; identity unless SCHUR detection */
    double W_adaptive[36];         /* utils.hpp:446; zero: no released handler writes it (dcreg.hpp:52) */
    double pcg_residual;           /* ||g - H dx||_2 at exit of the PCG solve */
} dcreg_analysis;

/* Per-iteration record: the numeric part of IterationLogData (DCReg/include/utils.hpp:174-249)
 * that pins the path (columns of iteration_details_with_dx.csv, SURVEY.md Appendix B.4). */
typedef struct dcreg_iter_log {
    int32_t iter;
    int32_t status;                /* dcreg_status of this iteration */
    int32_t n_effective;           /* corr_num / effective_points */
    int32_t n_corr_pt;             /* correspondence_pt_count (5th NN within radius) */
    double rmse, fitness, objective;
    double iter_time_ms;           /* IterationLogData::iter_time_ms (utils.hpp:174-249; tic at the top of the iteration,
                                      toc after the update, icp_test_runner.cpp:1695, 1973): device time between the
                                      end of the previous solve step (run start for iteration 0) and the end of this
                                      one, from the GPU's globaltimer */
    double gradient[6];            /* -A^T b */
    double H27[27];                /* 21 upper-tri of A^T A (row-major upper) + 6 rhs A^T b */
    double dx[6];
    double T[16];                  /* pose AFTER the update */
    dcreg_analysis analysis;
} dcreg_iter_log;

typedef struct dcreg_ctx dcreg_ctx;   /* opaque: owns device buffers, stream, (optional) NCCL comm */

/* ---- lifetime ---------------------------------------------------------------------------- */
int dcreg_abi_version(void);
/* Replaces: TestRunner ctor + ICPContext (icp_test_runner.cpp:10-17, utils.hpp:340-425). */
int dcreg_create(int device_id, dcreg_ctx** out);
int dcreg_destroy(dcreg_ctx* ctx);
const char* dcreg_last_error(const dcreg_ctx* ctx);
void dcreg_default_params(dcreg_icp_params* p);
/* cudaStream_t the context launches on (for CUDA-event timing by the caller). */
void* dcreg_stream(dcreg_ctx* ctx);

/* ---- clouds ------------------------------------------------------------------------------ */
/* Source (measure) cloud: n points, `stride` floats between points (3 for xyz, 4 for xyzi).
 * Copied to the device as float4.  Replaces the measure_cloud argument of
 * Point2PlaneICP_SO3_OpenMP (icp_test_runner.h:92-102). */
int dcreg_set_source(dcreg_ctx* ctx, const float* xyz, int64_t n, int stride);
/* Target cloud + its spatial index.  Replaces ICPContext::setTargetCloud's kd-tree build
 * (utils.hpp:393-424): a device hash grid with cell = `cell_size` (pass the search radius;
 * exact 5-NN-within-radius then only needs the 27 surrounding cells). */
int dcreg_set_target(dcreg_ctx* ctx, const float* xyz, int64_t m, int stride, double cell_size);

/* ---- seam 1: correspondence stage (icp_test_runner.cpp:1714-1813) -------------------------
 * For every source slot: q = fl32(R p + t), exact 5-NN in the target, 5th d^2 < radius^2,
 * 5x3 least-squares plane, normalisation, thickness gate.  Writes plane[i] = (nx,ny,nz,d) as
 * doubles (all-zero = no plane) into a device buffer owned by ctx and optionally copies it to
 * `planes_out` (host, 4*n doubles, may be NULL).  n_corr_pt = correspondence_pt_count. */
int dcreg_find_planes(dcreg_ctx* ctx, const double T[16], double search_radius,
                      double* planes_out, int64_t* n_corr_pt);

/* ---- seam 2: fused residual / weight / Jacobian / normal-equation reduction (K1) ----------
 * Replaces icp_test_runner.cpp:1774-1803 + 1863-1919 and the SymmetricHessianComputer functor
 * (hessian_computer.h:62-123): out27 = 21 upper-triangular entries of A^T A in the functor's
 * order followed by the 6 entries of A^T b (= -J^T r); stats = { sum r^2, N_eff, N_slots_with_plane }.
 * d_src / d_plane are DEVICE pointers to n float4 (x,y,z,-) and n float4 (nx,ny,nz,d); a slot
 * with an all-zero normal is skipped.  pose_Rt = R (9, row-major) then t (3). */
int dcreg_reduce_normal_equations(dcreg_ctx* ctx, const void* d_src, const void* d_plane,
                                  int64_t n, const double pose_Rt[12], int use_weight_derivative,
                                  double out27[27], double stats[3]);
/* Same with n double4 planes (48 B/slot): the precision the reference itself uses for the plane. */
int dcreg_reduce_normal_equations_f64plane(dcreg_ctx* ctx, const void* d_src, const void* d_plane,
                                           int64_t n, const double pose_Rt[12],
                                           int use_weight_derivative, double out27[27],
                                           double stats[3]);
/* Host-buffer convenience of the above (copies in, reduces, copies out). plane_is_f64: 0/1. */
int dcreg_reduce_normal_equations_host(dcreg_ctx* ctx, const float* src4, const void* plane4,
                                       int plane_is_f64, int64_t n, const double pose_Rt[12],
                                       int use_weight_derivative, double out27[27], double stats[3]);

/* ---- seam 3: degeneracy analysis + solve (K2) ---------------------------------------------
 * Replaces DCReg::analyzeDegeneracy (dcreg.hpp:45-166), DCReg::solveDegenerateSystem
 * (dcreg.hpp:168-264), the released Schur block (icp_test_runner.cpp:2418-2469) and the
 * stubbed alignAndOrthonormalize / solvePCG (dcreg.hpp:267-287; paper Alg. 1-3).
 * Runs on the device (single-warp kernel); H27 and outputs are HOST pointers. */
int dcreg_analyze_and_solve(dcreg_ctx* ctx, const double H27[27], const dcreg_icp_params* params,
                            dcreg_analysis* out, double dx[6]);
/* DCReg::solvePCG (dcreg.hpp:279-283): A (36, row-major), b (6), P (36) -> x (6). */
int dcreg_solve_pcg(dcreg_ctx* ctx, const double A[36], const double b[6], const double P[36],
                    int max_iterations, double tolerance, double x[6], int* iterations);

/* ---- the outer loop ------------------------------------------------------------------------
 * Replaces TestRunner::Point2PlaneICP_SO3_OpenMP (icp_test_runner.h:92-102,
 * icp_test_runner.cpp:1611-2060).  Uses the clouds set on ctx.  All iterations (correspondences,
 * reduction, analysis, solve, pose update, convergence test) run on the device with no host
 * round trip; the host reads the final pose and the per-iteration log afterwards.
 * log may be NULL (log_cap 0).  *converged mirrors the reference's bool return.
 * Returns DCREG_OK also when not converged; DCREG_NOT_ENOUGH_POINTS / DCREG_NONFINITE_UPDATE
 * when the reference would abort (T_out then holds the last pose, as in the reference). */
int dcreg_icp_run(dcreg_ctx* ctx, const dcreg_icp_params* params, const double T_init[16],
                  double T_out[16], dcreg_iter_log* log, int log_cap, int* n_iterations,
                  int* converged);
/* The same run split in two for callers that pipeline scans: dcreg_icp_enqueue puts the whole run (all max_iterations
 * loop bodies; iterations past convergence exit at once on the device) on the context's stream and returns without any
 * host synchronisation; dcreg_icp_fetch waits for the stream and returns the pose / iteration count / flags of the LAST
 * enqueued run with dcreg_icp_run's return value.  No per-iteration log on this path. */
int dcreg_icp_enqueue(dcreg_ctx* ctx, const dcreg_icp_params* params, const double T_init[16]);
int dcreg_icp_fetch(dcreg_ctx* ctx, double T_out[16], int* n_iterations, int* converged);
/* Many registrations of the SAME source against the SAME target from different initial poses, side by side in one
 * sequence of launches (trial = grid y-dimension; each trial owns its loop state, neighbour records and log slice, and
 * stops on its own convergence test).  Replaces the `num_runs` loop of TestRunner::runSingleTest
 * (icp_test_runner.cpp:331-345: `for run in 0..num_runs: runSingleTest`) and is what a perturbation Monte-Carlo
 * (BASELINE.json configs[4]) calls.  T_init / T_out: n_trials row-major 4x4 matrices; n_iterations / converged / status:
 * n_trials ints (status[t] = what dcreg_icp_run would have returned for trial t; any may be NULL except T_init, T_out);
 * log: n_trials x log_cap records (trial-major) or NULL.  Every trial runs the kernels a dcreg_icp_run from the same
 * T_init runs: counts, masks and iteration counts are identical, poses equal up to the order of the FP64 sums (the
 * source is sorted by target cell once, under trial 0's pose, and a single run of a small cloud uses smaller tiles;
 * 1e-8 on the poses in the tests; a batch itself is reproducible bit for bit).  Not
 * available on a sharded context: trials are independent, distribute them over ranks instead.  Needs the dense grid. */
int dcreg_icp_run_batch(dcreg_ctx* ctx, const dcreg_icp_params* params, int n_trials, const double* T_init,
                        double* T_out, int* n_iterations, int* converged, int* status, dcreg_iter_log* log,
                        int log_cap);
/* Many DIFFERENT source scans registered against the context's target (e.g. every frame of a recorded sequence
 * against one prior map, each from its own initial guess), side by side: scan s = points
 * [scan_offsets[s], scan_offsets[s+1]) of xyz (`stride` floats per point), trial = scan.  T_init / T_out /
 * n_iterations / converged / status / log as in dcreg_icp_run_batch (log trial-major, n_scans x log_cap).
 * fitness of scan s is over its own point count.  The context's source (dcreg_set_source) is not replaced.
 * Every scan runs the kernels a dcreg_icp_run of that scan alone from the same T_init runs (the scan is sorted by
 * target cell under its own T_init and uses its own lever arm): counts, masks and iteration counts are identical,
 * poses equal up to the grouping of the FP64 sums (1e-8 in the tests); a one-scan call IS a dcreg_icp_run, bit for bit,
 * and a call is reproducible bit for bit.  n_scans in [1, 65535]; scan_offsets[0] = 0 and strictly increasing (no empty
 * scan); at most 0x1fffffff points in all.  Needs the dense grid; not available on a sharded context (distribute the
 * scans over ranks instead). */
int dcreg_icp_run_scans(dcreg_ctx* ctx, const dcreg_icp_params* params, int n_scans,
                        const float* xyz, int stride, const int64_t* scan_offsets,
                        const double* T_init, double* T_out, int* n_iterations, int* converged, int* status,
                        dcreg_iter_log* log, int log_cap);
/* Same loop, but correspondences are supplied by the caller each iteration through a callback
 * (host kd-tree mode, "PR1"): planes are 4*n doubles (nx,ny,nz,d), all-zero = none. */
typedef int (*dcreg_plane_callback)(void* user, const double T[16], double* planes4,
                                    int64_t* n_corr_pt);
int dcreg_icp_run_host_planes(dcreg_ctx* ctx, const dcreg_icp_params* params,
                              const double T_init[16], dcreg_plane_callback cb, void* user,
                              double T_out[16], dcreg_iter_log* log, int log_cap,
                              int* n_iterations, int* converged);
/* Post-loop covariance (icp_test_runner.cpp:2014-2037): inverse of the last H with the 1e-9
 * eigenvalue floor, or 1e6*I when not converged.  cov: 36 doubles. */
int dcreg_last_covariance(dcreg_ctx* ctx, double cov[36]);
/* The same for each of the first n_trials trials of the last run (dcreg_icp_run: 1; dcreg_icp_run_batch /
 * dcreg_icp_run_scans: their trial count): cov = n_trials x 36 doubles, trial-major.  Trial 0 equals
 * dcreg_last_covariance bit for bit.  n_trials above the last run's trial count is refused. */
int dcreg_last_covariances(dcreg_ctx* ctx, int n_trials, double* cov);

/* Post-run point-to-point metrics on the device.  Replaces calculatePointToPointError
 * (DCReg/include/utils.hpp:538-589; callers icp_test_runner.cpp:506-510 and :1463-1470): aligned = fl32(T * source);
 * out = { P2P RMSE (over all source points, distances below error_threshold), P2P fitness, Chamfer distance,
 * number of source points within the threshold }.  Needs dcreg_set_source + dcreg_set_target. */
int dcreg_point_to_point_metrics(dcreg_ctx* ctx, const double T[16], double error_threshold, double out[4]);

/* dcreg_point_to_point_metrics for n_poses poses at once: T = n_poses row-major 4x4, out = n_poses x 4
 * {rmse, fitness, chamfer, n_valid}, pose-major.  Row i equals dcreg_point_to_point_metrics(ctx, T + 16 i, ...) bit
 * for bit.  Same preconditions (source + target set, dense target grid); n_poses >= 1.  The Chamfer half searches a
 * grid over the source in its own frame (built on first use, cell size of the target grid, kept until the next
 * dcreg_set_source / dcreg_set_target), so the source's bounding box must also fit a dense grid.  One host
 * synchronisation per call. */
int dcreg_point_to_point_metrics_batch(dcreg_ctx* ctx, int n_poses, const double* T, double error_threshold,
                                       double* out);

/* ---- multi-GPU: point-block sharding (SURVEY.md §8e) ---------------------------------------
 * Each rank holds a contiguous block of source slots; the 27+5 accumulators are summed over ranks
 * once per iteration (inside the reducing kernel over peer memory, see dcreg_comm_mode; one
 * ncclAllReduce of 32 doubles on the context's stream as the fallback), then every rank runs K2
 * redundantly on bit-identical sums.  nccl_unique_id is the 128-byte ncclUniqueId created by dcreg_comm_unique_id on
 * rank 0 and distributed by the caller (e.g. torch.distributed broadcast). */
int dcreg_comm_unique_id(dcreg_ctx* ctx, uint8_t id_out[128]);
int dcreg_comm_init(dcreg_ctx* ctx, const uint8_t nccl_unique_id[128], int rank, int nranks);
int dcreg_comm_destroy(dcreg_ctx* ctx);
/* How the per-iteration sum over ranks is carried: 0 = no communicator, 1 = ncclAllReduce behind the reducing kernel
 * (fallback), 2 = peer-memory mailboxes over NVLink inside the reducing kernel's last block (one kernel per iteration,
 * bit-identical sums on every rank).  dcreg_comm_init picks 2 when every rank could map every peer (cudaIpc). */
int dcreg_comm_mode(const dcreg_ctx* ctx);
/* Total number of source points over all ranks (denominator of `fitness`); defaults to local n. */
int dcreg_set_global_source_count(dcreg_ctx* ctx, int64_t n_total);

/* ---- instrumentation ----------------------------------------------------------------------- */
/* Number of kernels this context has launched since creation (bench.py's gpu_launches). */
int64_t dcreg_launch_count(const dcreg_ctx* ctx);
/* Device pointers of the ctx-owned source float4 array and plane arrays (for the K1 seam). */
void* dcreg_device_source(dcreg_ctx* ctx);
void* dcreg_device_planes_f64(dcreg_ctx* ctx);
void* dcreg_device_planes_f32(dcreg_ctx* ctx);   /* filled by dcreg_freeze_planes_f32 */
/* Round the ctx's double planes to float4 on the device (the 32 B/slot K1 layout). */
int dcreg_freeze_planes_f32(dcreg_ctx* ctx);
/* Enqueue `reps` K1 launches over the ctx-owned source + planes (plane_is_f64 0/1) and return
 * the average device time per launch in milliseconds, measured with CUDA events on ctx's stream.
 * If flush_l2 != 0 a >L2-sized buffer is rewritten before every launch (outside the events). */
int dcreg_time_reduce(dcreg_ctx* ctx, int plane_is_f64, const double pose_Rt[12],
                      int use_weight_derivative, int reps, int flush_l2, float* ms_per_launch);
/* Profiling aid for the fused loop: enqueue `reps` loop bodies from pose T (source sorted as dcreg_icp_run does) and
 * return the average device time per body in milliseconds.  what = 0: the iteration kernel alone at the fixed
 * pose T; what = 1: iteration kernel + solve/update kernel, i.e. `reps` real iterations (no convergence stop). */
int dcreg_time_iteration(dcreg_ctx* ctx, const dcreg_icp_params* params, const double T[16], int what,
                         int reps, float* ms_per_body);
/* Profiling aid: run `iters` real loop iterations from pose T and record the phase time stamps (GPU globaltimer, ns) of
 * the LAST one.  out: (n_blocks + 1) x 16 values; row b < n_blocks, thread 0 of block b: [0] start (pose loaded),
 * [1] certificates done, [2] searches done, [3] fit list built, [4] fits done, [5] rows / Gram done, and for the block
 * that finished the reduction [6] partials summed, [7] sums ready, [8] solve step done; row n_blocks: the solve step's
 * own stamps [0] entry, [1] block inverses, [2] Schur eigen-decompositions, [3] preconditioner, [4] solve, [5] pose
 * update, and [15] = index of the block that ran it. */
int dcreg_iteration_timeline(dcreg_ctx* ctx, const dcreg_icp_params* params, const double T[16], int iters,
                             uint64_t* out, int out_cap_blocks, int* n_blocks);
/* Profiling counters of the loop's iteration kernel since the last call: out = { source slots that ran a neighbour
 * search, source slots that ran a plane fit } (the others reused the previous iteration's result, see DESIGN.md).
 * enable != 0 switches the counting on (off by default), 0 switches it off. */
int dcreg_iteration_counters(dcreg_ctx* ctx, int enable, uint64_t out[2]);

#ifdef __cplusplus
}
#endif
#endif /* DCREG_B200_H */
