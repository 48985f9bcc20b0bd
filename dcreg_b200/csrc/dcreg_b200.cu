// dcreg_b200.cu - kernels + C ABI of the B200-native ICP / degeneracy engine (see include/dcreg_b200.h).
//
// Data layout in HBM (per context):
//   src      float4[N]   body-frame source points (x,y,z,-), uploaded once per scan
//   tgt grid float4[M]   target points grouped by hash-grid cell + keys/start/count tables
//   planes64 double4[N]  (nx,ny,nz,d) per source slot, only materialised for the seams / host-plane mode
//   planes32 float4[N]   the 32 B/slot frozen-plane layout of the K1 benchmark
//   scans    float4[sum n_s]  dcreg_icp_run_scans: many source scans back to back (own buffers, sorted per scan)
//   per trial (dcreg_icp_run: one, dcreg_icp_run_batch: many, dcreg_icp_run_scans: one per scan): neighbour records /
//   plane cache (100 B per slot; scans: one per slot of the scan set),
//   partials double[grid.x][32], acc double[32], ticket, state (pose, flags, warm-start bases), log records
// One ICP iteration = ONE kernel (icp_iter2_kernel): correspondences + residual + Jacobian + 27-sum reduction; the block
// that finishes a trial's reduction sums the block partials, [adds the other ranks' sums through peer-memory mailboxes,
// peer_reduce.cuh,] and its first warp runs the K2 step (analysis, solve, pose update, convergence flag), so nothing
// returns to the host inside the loop and the loop bodies of a run are replayed as one CUDA graph.  Baseline methods,
// hash grids and the NCCL fallback of a sharded run keep K2 as a second kernel (k2_step_kernel).
#include <cub/device/device_radix_sort.cuh>
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/dcreg_b200.h"
#include "corr.cuh"
#include "k1_reduce.cuh"
#include "k1_stream.cuh"
#include "k2_solve.cuh"
#include "loop_plan.hpp"
#include "p2p_bound.hpp"
#include "peer_reduce.cuh"

using k2::IcpState;
using k2::kAcc;

// ------------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------------
namespace {

constexpr int kBlock = 256;

// Programmatic dependent launch (sm_90+): the loop's two kernels are launched with the programmatic-stream-
// serialization attribute, so kernel k+1 is scheduled while kernel k still runs; pdl_wait() blocks until kernel k
// has completed and its writes are visible, pdl_release() lets kernel k+2 be scheduled.  Hides ~2 us of launch
// latency per kernel on the loop's critical path.  Without the attribute both are no-ops.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_release() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

__device__ __forceinline__ k1::Pose load_pose(const IcpState* st) {
    k1::Pose P;
#pragma unroll
    for (int i = 0; i < 9; ++i) P.R[i] = st->R[i];
#pragma unroll
    for (int i = 0; i < 3; ++i) P.t[i] = st->t[i];
    return P;
}

// Ticket: returns true in every thread of the last block to arrive.
__device__ __forceinline__ bool last_block_ticket(unsigned int* counter) {
    __shared__ bool is_last;
    __threadfence();
    if (threadIdx.x == 0) {
        const unsigned int t = atomicAdd(counter, 1u);
        is_last = (t == gridDim.x - 1);
    }
    __syncthreads();
    if (is_last) __threadfence();
    return is_last;
}

// K2 executed by warp 0 of the block that finished a trial's reduction (k2_solve.cuh).  A separate function with its
// own register allocation and stack frame: the iteration kernels are capped at 85 registers for 3 blocks per SM and
// must not pay for the solve's live state.  acc: the body-frame sums in shared memory.
static_assert(sizeof(k2::WarpSmem) <= 8 * k1::kTRow * sizeof(double), "k2::WarpSmem must fit one warp's transpose buffer");
static_assert(sizeof(corr::WarpKnnSmem) <= 8 * k1::kTRow * sizeof(double), "corr::WarpKnnSmem must fit one warp's transpose buffer");
__device__ __noinline__ void solve_step_in_kernel(const double* acc, IcpState* st, const dcreg_icp_params* prm,
                                                  dcreg_iter_log* log, int log_cap, k2::WarpSmem* sm, const float* src_radius,
                                                  double coherent_step, unsigned int* n_active, unsigned long long* dbg) {
    // only the "Ours" method (Schur detection + PCG, the warp-cooperative step) is folded; the baseline methods' generic
    // single-thread step needs a 3.7 KB stack frame, which every thread of the iteration kernel would have to reserve:
    // they keep the separate solve kernel (k2_step_kernel)
    const int lane = threadIdx.x & 31;
    const double lever = src_radius ? (double)*src_radius : 1.0e30;
    const double max_step = coherent_step * prm->search_radius;
    k2::icp_step_warp_ours(acc, st, *prm, log, log_cap, *sm, lever, max_step, dbg);    // all 32 lanes cooperate
    __syncwarp();
    if (lane == 0 && n_active && st->done) atomicSub(n_active, 1u);
}

struct IterArgs {
    const float4* src;        // source points, w = bit-cast original index (spatially sorted copy or the original)
    long long n;
    corr::Grid grid;
    IcpState* state;
    double* partials;
    unsigned int* counter;
    double* acc;
    double4* planes_out;      // optional: materialise the planes at the ORIGINAL slot index (seam 1)
    dcreg_icp_params prm;
};

struct IterSmem {
    double tbuf[kBlock / 32][8 * k1::kTRow];   // per-warp DMMA transpose buffers
    k1::GramSmem gram;
};

// One ICP iteration on the device: stage S1 (correspondences: exact 5-NN in the grid, plane fit, gates) fused with
// the residual / weight / Jacobian row and the Gram accumulation (S4-S5).  One source point per thread per trip;
// no per-thread accumulator block: the 8x8 Gram is accumulated with DMMA (two registers per lane).
template <bool kUseWd>
__global__ void __launch_bounds__(kBlock, 3) icp_iteration_kernel(const __grid_constant__ IterArgs a) {
    __shared__ IterSmem sm;
    if (a.state->done) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const k1::Pose P = load_pose(a.state);
    double c0 = 0.0, c1 = 0.0, e0 = 0.0, e1 = 0.0;
    int neff = 0, npt = 0;
    const double r2max = a.prm.search_radius * a.prm.search_radius;
    const long long n32 = (a.n + 31) & ~31ll;                 // whole warps enter the DMMA section together
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n32;
         i += (long long)gridDim.x * blockDim.x) {
        double px = 0.0, py = 0.0, pz = 0.0, nx = 0.0, ny = 0.0, nz = 0.0, d = 0.0;
        bool ok = false;
        if (i < a.n) {
            const float4 p4 = __ldg(&a.src[i]);
            px = (double)p4.x; py = (double)p4.y; pz = (double)p4.z;
            // q = fl32(R p + t)  (utils.hpp:630-636)
            const float qx = (float)(P.R[0] * px + P.R[1] * py + P.R[2] * pz + P.t[0]);
            const float qy = (float)(P.R[3] * px + P.R[4] * py + P.R[5] * pz + P.t[1]);
            const float qz = (float)(P.R[6] * px + P.R[7] * py + P.R[8] * pz + P.t[2]);
            corr::Knn5 nn;
            corr::knn_init(nn);
            corr::knn_search(a.grid, qx, qy, qz, nn);
            int npos[5];
            corr::knn_positions(a.grid, nn, npos);
            if (npos[4] >= 0 && (double)corr::knn_d2(nn, 4) < r2max) {       // icp_test_runner.cpp:1726
                npt += 1;                                                     // :1731
                ok = corr::fit_plane(a.grid, npos, a.prm.min_normal_norm, a.prm.plane_thickness, nx, ny, nz, d);
            }
            if (a.planes_out)
                a.planes_out[__float_as_int(p4.w)] = ok ? make_double4(nx, ny, nz, d) : make_double4(0.0, 0.0, 0.0, 0.0);
        }
        double c[8];
        k1::slot_front<kUseWd>(P, px, py, pz, nx, ny, nz, d, ok, c, neff, a.prm.weight_slope, a.prm.weight_gate);
        __syncwarp();
        k1::gram_accumulate_dmma(sm.tbuf[warp], lane, c, c0, c1, e0, e1);
    }
    k1::finish_block(c0 + e0, c1 + e1, neff, npt, sm.gram, a.partials, a.counter, a.state->R, a.acc);
}

// ---- the loop's iteration kernel (dense target grid) -------------------------------------------------------------
// One thread per source slot (the source is sorted by target cell once per run):
//   1. q = fl32(R p + t); squared distances from q to the slot's SEVEN nearest target points of its last search.
//   2. skip test.  That search also left lb8, a lower bound on the squared distance from q_scan (where the query then
//      was) to every target point outside the seven.  The query has moved by delta = |q - q_scan|; while
//          (5th smallest of the seven new distances) + delta < sqrt(lb8)
//      (with margins that dwarf the float32 evaluation error of a squared distance) no outside point can be among
//      the five nearest, so the seven are only re-ranked by their new distances (index rule on ties) and no cell is
//      touched.  On a uniform surface the 8th neighbour is ~26 % farther than the 5th, so once the pose moves by
//      less than a few centimetres per iteration almost every slot takes this path.
//   3. otherwise an exact bounded 7-NN search (corr::knn_search_lb): bound = 1.21 x the largest of the seven new
//      distances (seven distinct real points bound the 7th distance; the look-ahead is what finds a gap even when
//      the 8th candidate is far), or the search radius on the first iteration.
//   4. neighbour record to HBM (next iteration's seeds); plane fit to the first five, reused while the ordered
//      list of five stays the same (same five rows in the same order give the same QR bit for bit); residual /
//      weight / Jacobian row; DMMA Gram accumulation.  Searches and fits of a tile (<= 256 slots, Iter2Args::tile) go through work lists.
// Tail: packed per-block partial, atomic ticket, last block reduces (k1s::finish_packed).
// Record per slot (3 int4): {pos0..pos3}, {pos4..pos6, bits(lb8)}, {bits(q_scan.xyz), flags};
// pos = position in the grid's point array (ascending (d2, index) at the time of writing), -1 = none.
constexpr int kNnRec = 3;
constexpr float kNnLook = 1.21f;              // squared-distance look-ahead beyond the seed bound (any value >= 1 is exact)
constexpr double kCoherentStep = 0.05;        // records are used once no source point moves more than this x search radius per iteration

constexpr int kStampSlots = 16;                // per-block phase time stamps of the loop kernel (profiling only)
#define DCREG_STAMP(k) do { if (a.stamps && tid == 0) a.stamps[(size_t)blockIdx.x * kStampSlots + (k)] = k2::globaltimer_ns(); } while (0)

constexpr int kSearchListMax = 96;            // more searching slots than this in a tile: every thread searches for itself

struct Iter2Smem {
    double tbuf[kBlock / 32][8 * k1::kTRow];    // per-warp DMMA transpose buffers (also: corr::WarpKnnSmem, the warp's Gram,
                                                // and - in the last block, after the reduction - k2::WarpSmem)
    k1s::TailSmem tail;
    // coherent mode, per tile (<= kBlock slots)
    float4 q[kBlock];                           // query (x, y, z), w = search bound B
    int res[kBlock][10];                        // pos0..pos6, bits(lb), bits(d2 of the 5th), 1 = no search / 0 = searched / 2 = search pending
    int key[kBlock][5];                         // the five positions in distance order (slots that need a fit)
    double4 plane[kBlock];
    signed char fitres[kBlock];
    int listS[kBlock], listF[kBlock];
    corr::RowRange rowtab[kSearchListMax][9];   // cell rows of the tile's listed searches (cell = radius)
    int nS, nF;
};

// Grid = (blocks per trial, trials).  A trial is one registration (one initial pose) of the context's source against
// its target (icp_test_runner.cpp:331-345 runs `num_runs` of them back to back; dcreg_icp_run_batch runs them side by
// side).  Everything a trial owns is an array indexed by blockIdx.y: loop state, ticket, partials, sums, neighbour
// records, plane cache, log.  dcreg_icp_run is the one-trial case.
struct Iter2Args {
    IterArgs it;              // it.state / it.partials / it.counter / it.acc: per-trial arrays ([B], [B][grid.x][32], [B], [B][32])
    int4* nn;                 // [B][kNnRec n] neighbour records
    double4* plane_cache;     // [B][n] plane fitted to the slot's current five neighbours (reused while the set stays)
    signed char* fit_state;   // [B][n] 0 = nothing cached, 1 = cached fit failed its gates, 2 = cached plane valid
    int* plane_key;           // [B][5 n] the five positions (in distance order) the cached plane was fitted to
    // the solve / update step (K2) runs in the last block of every trial: no second launch, no host, no acc round trip
    int fold_k2;              // 0: stop after writing the sums (sharded run over NCCL: all-reduce + k2_step_kernel follow)
    dcreg_iter_log* log;      // [B][log_cap] or null
    int log_cap;
    const float* src_radius;  // max |p| over the source (lever arm of a rotation step); [B] when scan_off is set
    double coherent_step;
    unsigned int* n_active;   // trials still running (decremented by the step that finishes one); host polls it
    peer::View peer;          // multi-GPU: the sum over ranks, inside the last block (peer_reduce.cuh)
    unsigned long long* stamps;   // profiling only (dcreg_iteration_timeline): [grid.x][kStampSlots] globaltimer values, or null
    int coop_max;             // more searching slots than this in a tile: every thread searches for itself (kSearchListMax)
    int force;                // 0: mode and seeds from the loop state (written by K2); 1: coherent mode, seeds = use_seeds
    int use_seeds;            // (force) records of the previous launch are valid
    float r2_up;              // search radius^2 rounded up to float
    float look;               // squared-distance look-ahead beyond the seed bound (kNnLook)
    unsigned int* stats;      // optional [2]: slots that searched, slots that refitted (profiling)
    int tile;                 // source slots per block and pass (<= kBlock; plan_iteration: chosen so the blocks fill whole SM rounds)
    // many scans (dcreg_icp_run_scans, icp_iter2_kernel<., true>): [B + 1], trial t reads slots [scan_off[t], scan_off[t+1])
    // of it.src and its records sit at scan_off[t].  Otherwise null: every trial reads the same it.n slots, records at trial * it.n
    const long long* scan_off;
};

__device__ __forceinline__ void cswap5(unsigned long long& ka, int& pa, unsigned long long& kb, int& pb) {
    if (kb < ka) {                                    // one 64-bit compare = (distance, then index) order (corr::knn_key)
        const unsigned long long tk = ka; ka = kb; kb = tk;
        const int tp = pa; pa = pb; pb = tp;
    }
}

// kScans: trial t registers scan t of a scan set (Iter2Args::scan_off); a separate instance, so that the loop of
// dcreg_icp_run / dcreg_icp_run_batch keeps its code
template <bool kUseWd, bool kScans>
__global__ void __launch_bounds__(kBlock, 3) icp_iter2_kernel(const __grid_constant__ Iter2Args a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Iter2Smem& sm = *reinterpret_cast<Iter2Smem*>(smem_raw);
    const IterArgs& A = a.it;
    pdl_wait();                                   // the pose / mode flags come from the previous iteration's solve step
    pdl_release();
    const int trial = (int)blockIdx.y;
    IcpState* const st = A.state + trial;
    if (st->done) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const k1::Pose P = load_pose(st);
    const corr::Grid& g = A.grid;
    const unsigned int epoch0 = peer::load_epoch(a.peer);     // (after pdl_wait: the previous launch has advanced it)
    DCREG_STAMP(0);
    // this trial's source slots and its slices of the per-slot records
    const float4* src = A.src;
    long long n = A.n;
    int4* rec_nn = a.nn + (size_t)trial * kNnRec * A.n;
    double4* rec_plane = a.plane_cache + (size_t)trial * A.n;
    signed char* rec_fit = a.fit_state + (size_t)trial * A.n;
    int* rec_key = a.plane_key + (size_t)trial * 5 * A.n;
    if constexpr (kScans) {                       // scan `trial`: its own slots; its records start at its first slot
        const long long s0 = a.scan_off[trial];
        n = a.scan_off[trial + 1] - s0;
        src += s0;
        rec_nn = a.nn + (size_t)kNnRec * s0; rec_plane = a.plane_cache + s0; rec_fit = a.fit_state + s0; rec_key = a.plane_key + (size_t)5 * s0;
    }
    // mode (uniform over the grid): while the pose still moves by more than ~5 % of the search radius per iteration
    // nothing can be reused; the lean path (plain 5-NN search, no records) is ~25 % cheaper than searching with a
    // certificate.  K2 flips `coherent` from the size of its update.
    const bool coherent = a.force ? true : (st->coherent != 0);
    const bool use_seeds = a.force ? (a.use_seeds != 0) : (coherent && st->seeds != 0);
    double c0 = 0.0, c1 = 0.0, e0 = 0.0, e1 = 0.0;
    int neff = 0, npt = 0;
    unsigned n_search = 0, n_fit = 0;
    const double r2max = A.prm.search_radius * A.prm.search_radius;
    {
        // ---- tiles of a.tile (<= 256) slots with per-tile work lists, so that searches and fits run densely packed.  Lean mode (the
        // pose still moves a lot) uses the same phases: every slot searches (plain 5-NN), every accepted slot fits.
        for (long long base = (long long)blockIdx.x * a.tile; base < n; base += (long long)gridDim.x * a.tile) {
            const long long i = base + tid;
            const bool valid = tid < a.tile && i < n;
            if (tid == 0) { sm.nS = 0; sm.nF = 0; }
            __syncthreads();
            // -- 1. query, previous seven, certificate
            double px = 0.0, py = 0.0, pz = 0.0;
            bool need = false;
            if (valid) {
                const float4 p4 = __ldg(&src[i]);
                px = (double)p4.x; py = (double)p4.y; pz = (double)p4.z;
                // q = fl32(R p + t)  (utils.hpp:630-636)
                const float qx = (float)(P.R[0] * px + P.R[1] * py + P.R[2] * pz + P.t[0]);
                const float qy = (float)(P.R[3] * px + P.R[4] * py + P.R[5] * pz + P.t[1]);
                const float qz = (float)(P.R[6] * px + P.R[7] * py + P.R[8] * pz + P.t[2]);
                float B = a.r2_up;
                need = true;
                if (use_seeds) {
                    const int4 s0 = rec_nn[kNnRec * i], s1 = rec_nn[kNnRec * i + 1], s2 = rec_nn[kNnRec * i + 2];   // one round trip
                    if (s1.z >= 0) {                                          // all seven seeds exist
                        corr::KnnM nn;
                        nn.pos[0] = s0.x; nn.pos[1] = s0.y; nn.pos[2] = s0.z; nn.pos[3] = s0.w;
                        nn.pos[4] = s1.x; nn.pos[5] = s1.y; nn.pos[6] = s1.z;
#pragma unroll
                        for (int k = 0; k < corr::kSeeds; ++k) {
                            const float4 t = __ldg(&g.pts[nn.pos[k]]);
                            nn.key[k] = corr::knn_key(corr::dist2(qx, qy, qz, t), __float_as_int(t.w));
                        }
                        // 16-exchange sorting network on (d2, index)
#define DCREG_CS(x, y) cswap5(nn.key[x], nn.pos[x], nn.key[y], nn.pos[y])
                        DCREG_CS(0, 6); DCREG_CS(2, 3); DCREG_CS(4, 5); DCREG_CS(0, 2); DCREG_CS(1, 4); DCREG_CS(3, 6);
                        DCREG_CS(0, 1); DCREG_CS(2, 5); DCREG_CS(3, 4); DCREG_CS(1, 2); DCREG_CS(4, 6); DCREG_CS(2, 3);
                        DCREG_CS(4, 5); DCREG_CS(1, 2); DCREG_CS(3, 4); DCREG_CS(5, 6);
#undef DCREG_CS
                        B = fminf(B, corr::knn_d2(nn, 6) * a.look);
                        const float ex = qx - __int_as_float(s2.x), ey = qy - __int_as_float(s2.y), ez = qz - __int_as_float(s2.z);
                        const float delta = sqrtf(ex * ex + ey * ey + ez * ez);
                        const float lb = __int_as_float(s1.w);
                        // nothing outside the seven was closer than sqrt(lb) to q_scan; it is now at least sqrt(lb) - delta away
                        need = !((sqrtf(corr::knn_d2(nn, 4)) + delta) * 1.00002f + 1e-7f < sqrtf(lb) * 0.99998f);
                        if (!need) {
#pragma unroll
                            for (int k = 0; k < corr::kSeeds; ++k) sm.res[tid][k] = nn.pos[k];
                            sm.res[tid][7] = s1.w; sm.res[tid][8] = __float_as_int(corr::knn_d2(nn, 4)); sm.res[tid][9] = 1;
                        }
                    }
                }
                sm.q[tid] = make_float4(qx, qy, qz, B);
                if (need) { sm.res[tid][9] = 2; ++n_search; }
            }
            {   // search list of the tile (slot order)
                const unsigned bits = __ballot_sync(0xffffffffu, need);
                int wbase = 0;
                if (lane == 0 && bits) wbase = atomicAdd(&sm.nS, __popc(bits));
                wbase = __shfl_sync(0xffffffffu, wbase, 0);
                if (need) sm.listS[wbase + __popc(bits & ((1u << lane) - 1u))] = tid;
            }
            DCREG_STAMP(1);
            __syncthreads();
            // -- 2. searches: few -> one warp per listed slot (the other slots' threads are not held up by a
            //       15 us sequential search); many -> every thread searches for its own slot
            const int nS = sm.nS;
            if (coherent && nS <= a.coop_max) {
                corr::WarpKnnSmem& W = *reinterpret_cast<corr::WarpKnnSmem*>(sm.tbuf[warp]);
                // cell = radius: the 9 cell rows of EVERY listed search are set up by all threads first (one memory round
                // trip for the tile instead of one at the head of each of a warp's searches)
                const bool pre_rows = g.rings == 1 && nS <= kSearchListMax;
                if (pre_rows) {
                    for (int e = tid; e < nS * 9; e += kBlock) {
                        const int sidx = e / 9, r = e - sidx * 9;
                        const float4 q = sm.q[sm.listS[sidx]];
                        sm.rowtab[sidx][r] = corr::knn_row_range(g, q.x, q.y, q.z, q.w, r);
                    }
                    __syncthreads();
                }
                for (int w = warp; w < nS; w += kBlock / 32) {
                    const int t = sm.listS[w];
                    const float4 q = sm.q[t];
                    corr::KnnM r;
                    float lbq = a.r2_up * 0.9999f;    // nothing beyond the rings of cells is closer than the radius
                    const bool got = corr::knn_warp_search(g, q.x, q.y, q.z, q.w, W, r, lbq,
                                                           (a.stamps && warp == 0) ? reinterpret_cast<long long*>(a.stamps + (size_t)blockIdx.x * kStampSlots + 9) : nullptr,
                                                           pre_rows ? sm.rowtab[w] : nullptr);
                    if (got) {
                        if (lane < corr::kSeeds) sm.res[t][lane] = W.opos[lane];
                        if (lane == 7) sm.res[t][7] = __float_as_int(lbq);
                        if (lane == 8) sm.res[t][8] = __float_as_int(corr::knn_d2(r, 4));
                        if (lane == 9) sm.res[t][9] = 0;
                    }
                    __syncwarp();
                }
                __syncthreads();
            }
            DCREG_STAMP(2);
            if (valid && sm.res[tid][9] == 2) {       // too many for the list, or more than 64 candidates inside the bound
                const float4 q = sm.q[tid];
                if (coherent) {
                    corr::KnnM r;
                    float lbq = a.r2_up * 0.9999f;
                    corr::knn_search_lb(g, q.x, q.y, q.z, q.w, r, lbq);
#pragma unroll
                    for (int k = 0; k < corr::kSeeds; ++k) sm.res[tid][k] = r.pos[k];
                    sm.res[tid][7] = __float_as_int(lbq); sm.res[tid][8] = __float_as_int(corr::knn_d2(r, 4));
                } else {                              // lean: plain exact 5-NN, nothing kept for the next iteration
                    corr::Knn5 r;
                    corr::knn_init(r);
                    corr::knn_search(g, q.x, q.y, q.z, r);
                    int rpos[5];
                    corr::knn_positions(g, r, rpos);
#pragma unroll
                    for (int k = 0; k < 5; ++k) sm.res[tid][k] = rpos[k];
                    sm.res[tid][5] = -1; sm.res[tid][6] = -1; sm.res[tid][7] = 0; sm.res[tid][8] = __float_as_int(corr::knn_d2(r, 4));
                }
                sm.res[tid][9] = 0;
            }
            // -- 3a. record; which five; cached plane?
            double nx = 0.0, ny = 0.0, nz = 0.0, d = 0.0;
            bool ok = false, want_fit = false, have5 = false;
            float d5 = 0.0f;
            if (valid) {
                int pos[corr::kSeeds];
#pragma unroll
                for (int k = 0; k < corr::kSeeds; ++k) pos[k] = sm.res[tid][k];
                d5 = __int_as_float(sm.res[tid][8]);
                if (coherent) {
                    rec_nn[kNnRec * i] = make_int4(pos[0], pos[1], pos[2], pos[3]);
                    rec_nn[kNnRec * i + 1] = make_int4(pos[4], pos[5], pos[6], sm.res[tid][7]);
                    if (sm.res[tid][9] == 0) {                                // searched: remember where
                        const float4 q = sm.q[tid];
                        rec_nn[kNnRec * i + 2] = make_int4(__float_as_int(q.x), __float_as_int(q.y), __float_as_int(q.z), 0);
                    }
                }
                // (a lean search is not bounded by the radius: its five may lie outside and then need no plane)
                have5 = pos[4] >= 0 && (coherent || (double)d5 < r2max);
                // The plane is a function of the five target points IN THEIR ORDER (the rows of the 5x3 system keep the
                // reference's distance order, so the QR rounds exactly as a fresh fit would): the cache key is the
                // ordered list.  A pure re-ranking therefore refits; the fit list keeps that cheap.
                const int key[5] = {pos[0], pos[1], pos[2], pos[3], pos[4]};
                int fit = 0;                                                  // 1 = gates failed, 2 = plane valid
                if (have5) {
                    int cached = 0;
                    if (use_seeds) {
                        const int* kp = rec_key + 5 * i;
                        if (kp[0] == key[0] && kp[1] == key[1] && kp[2] == key[2] && kp[3] == key[3] && kp[4] == key[4])
                            cached = (int)rec_fit[i];
                    }
                    if (cached == 2) {
                        const double4 c = rec_plane[i];
                        nx = c.x; ny = c.y; nz = c.z; d = c.w;
                        fit = 2;
                    } else if (cached == 1) {
                        fit = 1;
                    } else {
                        want_fit = true;
#pragma unroll
                        for (int k = 0; k < 5; ++k) sm.key[tid][k] = key[k];
                    }
                }
                if (!want_fit) { if (coherent) rec_fit[i] = (signed char)fit; ok = fit == 2; }
            }
            {   // fit list of the tile
                const unsigned bits = __ballot_sync(0xffffffffu, want_fit);
                int wbase = 0;
                if (lane == 0 && bits) wbase = atomicAdd(&sm.nF, __popc(bits));
                wbase = __shfl_sync(0xffffffffu, wbase, 0);
                if (want_fit) sm.listF[wbase + __popc(bits & ((1u << lane) - 1u))] = tid;
            }
            DCREG_STAMP(3);
            __syncthreads();
            // -- 3b. fits, densely packed into the first warps
            const int nF = sm.nF;
            for (int f = tid; f < nF; f += kBlock) {
                const int t = sm.listF[f];
                int key[5];
#pragma unroll
                for (int k = 0; k < 5; ++k) key[k] = sm.key[t][k];
                double fx = 0.0, fy = 0.0, fz = 0.0, fd = 0.0;
                const int fit = corr::fit_plane_reg(g, key, A.prm.min_normal_norm, A.prm.plane_thickness, fx, fy, fz, fd) ? 2 : 1;
                sm.plane[t] = make_double4(fx, fy, fz, fd);
                sm.fitres[t] = (signed char)fit;
                if (coherent) {
                    const long long it = base + t;
                    if (fit == 2) rec_plane[it] = make_double4(fx, fy, fz, fd);
                    int* kp = rec_key + 5 * it;
#pragma unroll
                    for (int k = 0; k < 5; ++k) kp[k] = key[k];
                    rec_fit[it] = (signed char)fit;
                }
                ++n_fit;
            }
            __syncthreads();
            DCREG_STAMP(4);
            // -- 3c. gate, row, Gram
            if (valid) {
                if (want_fit) {
                    const double4 c = sm.plane[tid];
                    nx = c.x; ny = c.y; nz = c.z; d = c.w;
                    ok = sm.fitres[tid] == 2;
                }
                if (have5 && (double)d5 < r2max) npt += 1;                    // icp_test_runner.cpp:1726, 1731
                else ok = false;
                if (!ok) { nx = 0.0; ny = 0.0; nz = 0.0; d = 0.0; }
            }
            double c[8];
            k1::slot_front<kUseWd>(P, px, py, pz, nx, ny, nz, d, ok, c, neff, A.prm.weight_slope, A.prm.weight_gate);
            __syncwarp();
            k1::gram_accumulate_dmma(sm.tbuf[warp], lane, c, c0, c1, e0, e1);
            __syncthreads();
        }
    }
    DCREG_STAMP(5);
    if (a.stats) {
        n_search = __reduce_add_sync(0xffffffffu, n_search);
        n_fit = __reduce_add_sync(0xffffffffu, n_fit);
        if (lane == 0 && (n_search | n_fit)) { atomicAdd(&a.stats[0], n_search); atomicAdd(&a.stats[1], n_fit); }
    }
    // ---- tail: the warp's 8x8 Gram -> packed totals (k1s::kPk layout), then the grid reduction
    c0 += e0; c1 += e1;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        neff += __shfl_xor_sync(0xffffffffu, neff, off);
        npt += __shfl_xor_sync(0xffffffffu, npt, off);
    }
    double* G = sm.tbuf[warp];
    G[2 * lane] = c0; G[2 * lane + 1] = c1;
    __syncwarp();
    double mine = 0.0;
    if (lane < 21) {
        int i = 0, rem = lane;
        while (rem >= 6 - i) { rem -= 6 - i; ++i; }
        const int j = i + rem;
        mine = 0.5 * (G[i * 8 + j] + G[j * 8 + i]);
    } else if (lane < 27) {
        const int i = lane - 21;
        mine = 0.5 * (G[i * 8 + 6] + G[6 * 8 + i]);
    } else if (lane == k1s::kPkR2) mine = G[7 * 8 + 7];
    else if (lane == k1s::kPkB2) mine = G[6 * 8 + 6];
    else if (lane == k1s::kPkNeff) mine = (double)neff;
    else if (lane == k1s::kPkNpt) mine = (double)npt;
    // ---- grid reduction of this trial, [sum over ranks], congruence, solve + pose update: all in the last block
    if (!k1s::reduce_to_fin(mine, sm.tail, A.partials + (size_t)trial * gridDim.x * k1s::kPk, A.counter + trial,
                            (int)blockIdx.x, (int)gridDim.x)) return;
    DCREG_STAMP(6);
    peer::all_reduce32(a.peer, sm.tail.fin, sm.tail.red, epoch0);
    k1s::congruence(sm.tail.fin, st->R, sm.tail.acc);
    __syncthreads();
    DCREG_STAMP(7);
    if (tid < kAcc) A.acc[(size_t)trial * kAcc + tid] = sm.tail.acc[tid];
    if (a.fold_k2 && warp == 0) {
        solve_step_in_kernel(sm.tail.acc, st, &A.prm, a.log ? a.log + (size_t)trial * a.log_cap : nullptr, a.log_cap,
                             reinterpret_cast<k2::WarpSmem*>(sm.tbuf[0]),
                             kScans ? a.src_radius + trial : a.src_radius, a.coherent_step, a.n_active,
                             a.stamps ? a.stamps + (size_t)gridDim.x * kStampSlots : nullptr);
        DCREG_STAMP(8);
        if (a.stamps && tid == 0) a.stamps[(size_t)gridDim.x * kStampSlots + 15] = blockIdx.x;      // which block was last
    }
}

// K2 as its own kernel: baseline methods (their generic single-thread step), hash-grid runs, the host-plane loop and the
// NCCL fallback of a sharded run.  One warp per trial (blockIdx.x).
// K2 executes a few thousand warp instructions exactly once per launch (round 1 ncu: top stall no_instruction, 14 cycles
// per instruction).  Thanks to the programmatic dependent launch it starts while the
// iteration kernel is still running, so it first executes the SAME code on a scratch copy of the state with the
// previous iteration's sums (same branches, harmless stores), which pulls the instructions into the SM's caches;
// only then does it wait for the iteration kernel and do the real step.
static_assert(kAcc == 32, "k2_step_kernel copies acc with one element per lane");
struct K2Scratch {
    double acc_prev[kAcc];
    IcpState state;
};

// One warp per trial (blockIdx.x): acc_all [B][kAcc], st_all [B], log_all [B][log_cap].  scratch (rehearsal) only for B = 1.
// src_radius: one lever arm for every trial, or [B] (radius_per_trial: one per scan of dcreg_icp_run_scans).
__global__ void __launch_bounds__(32) k2_step_kernel(const double* acc_all, IcpState* st_all, dcreg_icp_params prm,
                                                     dcreg_iter_log* log_all, int log_cap, const float* src_radius,
                                                     int radius_per_trial, double coherent_step, K2Scratch* scratch,
                                                     unsigned int* n_active) {
    __shared__ k2::WarpSmem sm;
    pdl_release();
    const int lane = threadIdx.x;
    const double* acc = acc_all + (size_t)blockIdx.x * kAcc;
    IcpState* st = st_all + blockIdx.x;
    dcreg_iter_log* log = log_all ? log_all + (size_t)blockIdx.x * log_cap : nullptr;
    const double max_step = coherent_step * prm.search_radius;
    if (src_radius && radius_per_trial) src_radius += blockIdx.x;
    const bool warp_path = prm.detection == DCREG_DET_SCHUR_CONDITION_NUMBER && prm.handling == DCREG_HAND_PRECONDITIONED_CG;
#pragma unroll 1
    for (int pass = scratch ? 0 : 1; pass < 2; ++pass) {
        const double* acc_use = acc;
        IcpState* st_use = st;
        dcreg_iter_log* log_use = log;
        if (pass == 0) {                                  // rehearsal: nothing the previous kernels still write is read
            for (int e = lane; e < (int)(sizeof(IcpState) / sizeof(int)); e += 32)
                reinterpret_cast<int*>(&scratch->state)[e] = reinterpret_cast<const int*>(st)[e];
            __syncwarp();
            acc_use = scratch->acc_prev; st_use = &scratch->state; log_use = nullptr;
        } else {
            pdl_wait();                                   // acc comes from the iteration kernel (or the all-reduce) before
            if (st->done) return;
        }
        // mode of the next iteration kernel: records pay off once no source point moves more than ~5 % of the search radius
        const double lever = src_radius ? (double)*src_radius : 1.0e30;
        if (warp_path) {
            k2::icp_step_warp_ours(acc_use, st_use, prm, log_use, log_cap, sm, lever, max_step);   // all 32 lanes cooperate
        } else if (lane == 0) {
            k2::icp_step(acc_use, st_use, prm, log_use, log_cap, lever, max_step);    // baseline methods: generic single-thread path
        }
        __syncwarp();
        if (pass == 1 && scratch) scratch->acc_prev[lane] = acc[lane];              // kAcc == 32: next launch's rehearsal input
        if (pass == 1 && lane == 0 && n_active && st->done) atomicSub(n_active, 1u);
    }
}

__global__ void k2_analyze_kernel(const double* v27, dcreg_icp_params prm, dcreg_analysis* out, double* dx) {
    if (threadIdx.x != 0) return;
    k2::analyze_and_solve<true>(v27, prm, out, dx);
}

// Post-run log fill: one thread per iteration record recomputes the FULL analysis from the record's H27
// (same code, same inputs => identical mask / P / PCG counts as the in-loop critical path wrote) and thereby adds the
// log-only quantities without putting them on the loop's critical path.
__global__ void log_fill_kernel(dcreg_iter_log* logs, int log_cap, const IcpState* states, dcreg_icp_params prm) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const IcpState* st = states + blockIdx.y;
    dcreg_iter_log* log = logs + (size_t)blockIdx.y * log_cap;
    const int n = st->iter < log_cap ? st->iter : log_cap;
    if (i >= n) return;
    if (log[i].status != DCREG_OK) return;
    double dx[6];
    k2::analyze_and_solve<true>(log[i].H27, prm, &log[i].analysis, dx);
}

__global__ void pcg_kernel(const double* A, const double* b, const double* P, int max_it, double tol, double* x,
                           int* iters) {
    if (threadIdx.x != 0) return;
    double res;
    *iters = k2::pcg6(A, b, P, max_it, tol, x, &res);
}

// icp_test_runner.cpp:2014-2037.  One block per trial: st [B], cov [B][36].
__global__ void covariance_kernel(const IcpState* st, double* cov) {
    if (threadIdx.x != 0) return;
    st += blockIdx.x;
    cov += (size_t)blockIdx.x * 36;
    bool ok = false;
    if (st->converged) {
        double A[36], Inv[36];
        for (int i = 0; i < 36; ++i) A[i] = st->H_last[i];
        if (dla::fullpiv_inverse<6>(A, Inv)) {
            ok = true;
            double W[36], lam[6], V[36];
            for (int i = 0; i < 6; ++i)
                for (int j = 0; j < 6; ++j) W[i * 6 + j] = 0.5 * (Inv[i * 6 + j] + Inv[j * 6 + i]);
            dla::jacobi_eigh<6>(W, lam, V);
            if (lam[0] <= 1e-12) {
                for (int i = 0; i < 6; ++i) lam[i] = fmax(lam[i], 1e-9);
                for (int i = 0; i < 6; ++i)
                    for (int j = 0; j < 6; ++j) {
                        double s = 0.0;
                        for (int k = 0; k < 6; ++k) s += V[i * 6 + k] * lam[k] * V[j * 6 + k];
                        cov[i * 6 + j] = s;
                    }
            } else {
                for (int i = 0; i < 36; ++i) cov[i] = Inv[i];
            }
        }
    }
    if (!ok)
        for (int i = 0; i < 36; ++i) cov[i] = (i % 7 == 0) ? 1e6 : 0.0;
}

// scan_off (optional, [n_scans + 1]): the points form scans and radius[s] gets the max over scan s alone
__global__ void pack_source_kernel(const float* __restrict__ in, long long n, int stride, float4* __restrict__ out,
                                   float* __restrict__ radius, const long long* __restrict__ scan_off = nullptr,
                                   int n_scans = 0) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    float r = 0.0f;
    if (i < n) {
        const float x = in[i * stride], y = in[i * stride + 1], z = in[i * stride + 2];
        out[i] = make_float4(x, y, z, __int_as_float((int)i));   // w = slot index
        r = sqrtf(x * x + y * y + z * z);
        if (!(r < 3.0e38f)) r = 0.0f;                            // NaN / Inf points do not define a lever arm
    }
    if (radius && scan_off) {
        const int s = i < n ? corr::scan_of(scan_off, n_scans, i) : -1;
        const int s0 = __shfl_sync(0xffffffffu, s, 0);
        if (__all_sync(0xffffffffu, s == s0)) {                 // the whole warp in one scan: one atomic
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) r = fmaxf(r, __shfl_xor_sync(0xffffffffu, r, off));
            if ((threadIdx.x & 31) == 0 && r > 0.0f) atomicMax(reinterpret_cast<int*>(radius + s0), __float_as_int(r));
        } else if (s >= 0 && r > 0.0f) {
            atomicMax(reinterpret_cast<int*>(radius + s), __float_as_int(r));
        }
    } else if (radius) {                                        // max |p|: lever arm that turns a rotation step into metres
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) r = fmaxf(r, __shfl_xor_sync(0xffffffffu, r, off));
        if ((threadIdx.x & 31) == 0 && r > 0.0f) atomicMax(reinterpret_cast<int*>(radius), __float_as_int(r));
    }
}

__global__ void planes_to_f32_kernel(const double4* __restrict__ in, long long n, float4* __restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double4 v = in[i];
    out[i] = make_float4((float)v.x, (float)v.y, (float)v.z, (float)v.w);
}

__global__ void flush_l2_kernel(float4* buf, long long n, float v) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        buf[i] = make_float4(v, v, v, v);
}

// one thread per trial: T = [n_trials][16] row-major 4x4 initial poses.  scan_off (optional, [n_trials + 1]): trial t
// registers scan t, whose own point count is the denominator of its fitness (instead of n_total)
__global__ void init_state_kernel(IcpState* states, const double* T, long long n_total, unsigned int* counters, int n_trials,
                                  unsigned int* n_active, const long long* scan_off = nullptr) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b == 0 && n_active) *n_active = (unsigned)n_trials;
    if (b >= n_trials) return;
    IcpState* st = states + b;
    const double* Tb = T + (size_t)b * 16;
    for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 3; ++c) st->R[r * 3 + c] = Tb[r * 4 + c];
        st->t[r] = Tb[r * 4 + 3];
    }
    st->iter = 0; st->done = 0; st->converged = 0; st->status = DCREG_OK;
    for (int i = 0; i < 36; ++i) st->H_last[i] = (i % 7 == 0) ? 1.0 : 0.0;
    st->n_source_total = scan_off ? scan_off[b + 1] - scan_off[b] : n_total;
    st->step_rot = 1.0e30; st->step_trans = 1.0e30; st->seeds = 0; st->coherent_used = 0; st->coherent = 0; st->warm = 0;
    st->t_last = k2::globaltimer_ns();                      // tic of iteration 0 (icp_test_runner.cpp:1695)
    counters[b] = 0u;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// NCCL through dlopen (so the library loads without it; torch's bundled copy is reused when present)
// ------------------------------------------------------------------------------------------------
namespace {
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(ncclUniqueId*) = nullptr;
    int (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    int (*CommDestroy)(ncclComm_t) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    bool load(std::string& err) {
        if (lib) return true;
        const char* names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char* nm : names) {
            lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
            if (lib) break;
        }
        if (!lib) { err = std::string("dlopen libnccl failed: ") + dlerror(); return false; }
        GetUniqueId = (int (*)(ncclUniqueId*))dlsym(lib, "ncclGetUniqueId");
        CommInitRank = (int (*)(ncclComm_t*, int, ncclUniqueId, int))dlsym(lib, "ncclCommInitRank");
        CommDestroy = (int (*)(ncclComm_t))dlsym(lib, "ncclCommDestroy");
        AllReduce = (int (*)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t))dlsym(lib, "ncclAllReduce");
        AllGather = (int (*)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t))dlsym(lib, "ncclAllGather");
        GetErrorString = (const char* (*)(int))dlsym(lib, "ncclGetErrorString");
        if (!GetUniqueId || !CommInitRank || !CommDestroy || !AllReduce) { err = "libnccl: missing symbols"; return false; }
        return true;
    }
};
NcclApi g_nccl;
constexpr int kNcclFloat64 = 8;   // ncclDouble
constexpr int kNcclInt8 = 0;      // ncclInt8 / ncclChar
constexpr int kNcclSum = 0;
}  // namespace

// ------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------
struct dcreg_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    std::string err;
    long long launches = 0;

    float4* d_src = nullptr; long long n_src = 0; long long n_src_cap = 0; long long n_src_total = 0;
    float* d_stage = nullptr; size_t stage_bytes = 0;

    float4* d_tgt = nullptr; long long n_tgt = 0;
    corr::Grid grid{}; long long grid_cells = 0; bool has_grid = false;
    double4* d_plane_cache = nullptr; signed char* d_fit_state = nullptr;   // plane of the slot's current five neighbours
    int* d_plane_key = nullptr;                                             // ... and which five (ascending positions)
    bool force_coherent = false;                                           // profiling (dcreg_time_iteration what = 0)
    float* d_src_radius = nullptr;                                         // max |p| over the source cloud (device)
    unsigned int* d_iter_stats = nullptr;                                  // optional profiling counters of the iteration kernel
    int4* d_nn = nullptr; long long nn_cap = 0; bool nn_valid = false;   // neighbours of the sorted source (seeds of the next iteration)
    float4* d_src_sorted = nullptr; long long src_sorted_cap = 0;     // source in target-cell order (w = original index)
    float4* d_sort_tmp = nullptr;                                     // ... before the in-cell ranking
    int* d_cell_tmp = nullptr; long long cell_tmp_cap = 0;            // counts / fill cursors for the source sort
    int* d_pt_cell = nullptr; long long pt_cell_cap = 0;
    int* d_tile_sums = nullptr; long long tile_sums_cap = 0;
    double cell_size = 0.0;
    // dcreg_point_to_point_metrics_batch: grid over the source in its own frame (cell_size), dropped by set_source /
    // set_target; pose records + partial sums + results of one chunk of poses
    corr::Grid src_grid{}; bool has_src_grid = false;
    double* d_p2p = nullptr; long long p2p_cap = 0;

    double4* d_planes64 = nullptr; float4* d_planes32 = nullptr; long long planes_cap = 0;

    // per-trial arrays (dcreg_icp_run = 1 trial, dcreg_icp_run_batch = many): [trials_cap] each
    int trials_cap = 0;
    double* d_partials = nullptr; int partials_blocks = 0;
    unsigned int* d_counter = nullptr;
    double* d_acc = nullptr;
    IcpState* d_state = nullptr;
    unsigned int* d_n_active = nullptr;   // trials still running
    double* d_T_init = nullptr; int T_init_cap = 0;
    int nn_trials = 0;                    // trials the per-slot record arrays (d_nn, d_plane_cache, ...) are sized for
    dcreg_iter_log* d_log = nullptr; long long log_cap = 0;   // records, [trials][log_cap of the run]
    int last_trials = 0;                  // trials of the last run (their states are what dcreg_last_covariances reads)
    double* d_cov = nullptr; int cov_cap = 0;                 // [cov_cap][36] covariances of dcreg_last_covariances
    // the scans of dcreg_icp_run_scans, in buffers of their own (the source of dcreg_set_source stays in place)
    float4* d_scan = nullptr; long long scan_cap = 0;                 // as uploaded
    float4* d_scan_sorted = nullptr; long long scan_sorted_cap = 0;   // each scan in target-cell order
    unsigned long long* d_scan_keys = nullptr; long long scan_keys_cap = 0;   // radix sort keys, in | out
    int* d_scan_slots = nullptr; long long scan_slots_cap = 0;                // radix sort values, in | out
    void* d_scan_sort_tmp = nullptr; size_t scan_sort_tmp_bytes = 0;
    long long* d_scan_off = nullptr; long long scan_off_cap = 0;      // [n_scans + 1]
    float* d_scan_radius = nullptr; long long scan_radius_cap = 0;    // [n_scans] lever arms
    bool loop_attr_done = false, k1_attr_done[8] = {false, false, false, false, false, false, false, false};
    // CUDA graphs of one chunk of loop iterations, keyed on the kernel arguments (a few shapes alternate in practice:
    // with / without a log, one trial / a batch); most recently used first
    struct LoopGraph { std::vector<unsigned char> key; cudaGraphExec_t exec; };
    std::vector<LoopGraph> graphs; bool graph_off = false;
    long long graph_launches = 0;
    void drop_graphs() { for (auto& g : graphs) if (g.exec) cudaGraphExecDestroy(g.exec); graphs.clear(); }
    double* d_small = nullptr;       // scratch for the seams (>= 512 doubles)
    K2Scratch* d_k2_scratch = nullptr;   // K2's rehearsal state (see k2_step_kernel)
    dcreg_analysis* d_analysis = nullptr;
    float4* d_flush = nullptr; long long flush_n = 0;

    void* h_pinned = nullptr; size_t pinned_bytes = 0;

    ncclComm_t comm = nullptr; int rank = 0, nranks = 1;
    // peer mailboxes for the in-kernel sum over ranks (peer_reduce.cuh); NCCL all-reduce is the fallback
    peer::Mailbox* d_mailbox = nullptr; void* peer_ptr[peer::kMaxRanks] = {nullptr}; bool peer_ok = false;
    peer::View peer_view{};
};

namespace {

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_);                         \
            return DCREG_CUDA_ERROR;                                                               \
        }                                                                                          \
    } while (0)

int ensure_pinned(dcreg_ctx* ctx, size_t bytes) {
    if (ctx->pinned_bytes >= bytes) return DCREG_OK;
    if (ctx->h_pinned) cudaFreeHost(ctx->h_pinned);
    ctx->h_pinned = nullptr; ctx->pinned_bytes = 0;
    CK(cudaMallocHost(&ctx->h_pinned, bytes));
    ctx->pinned_bytes = bytes;
    return DCREG_OK;
}

int ensure_partials(dcreg_ctx* ctx, int blocks) {
    if (ctx->partials_blocks >= blocks) return DCREG_OK;
    if (ctx->d_partials) cudaFree(ctx->d_partials);
    ctx->d_partials = nullptr;
    CK(cudaMalloc(&ctx->d_partials, (size_t)blocks * 72 * sizeof(double)));   // >= k1s::kPart and kAcc
    ctx->partials_blocks = blocks;
    return DCREG_OK;
}

int ensure_planes(dcreg_ctx* ctx, long long n) {
    if (ctx->planes_cap >= n) return DCREG_OK;
    if (ctx->d_planes64) cudaFree(ctx->d_planes64);
    if (ctx->d_planes32) cudaFree(ctx->d_planes32);
    ctx->d_planes64 = nullptr; ctx->d_planes32 = nullptr; ctx->planes_cap = 0;
    CK(cudaMalloc(&ctx->d_planes64, (size_t)n * sizeof(double4)));
    CK(cudaMalloc(&ctx->d_planes32, (size_t)n * sizeof(float4)));
    ctx->planes_cap = n;
    return DCREG_OK;
}

int ensure_log(dcreg_ctx* ctx, long long records) {
    if (ctx->log_cap >= records) return DCREG_OK;
    if (ctx->d_log) cudaFree(ctx->d_log);
    ctx->d_log = nullptr; ctx->log_cap = 0;
    CK(cudaMalloc(&ctx->d_log, (size_t)records * sizeof(dcreg_iter_log)));
    ctx->log_cap = records;
    return DCREG_OK;
}

// grow a device buffer to `n` elements (contents not kept)
template <typename T>
int ensure_buffer(dcreg_ctx* ctx, T** p, long long* cap, long long n) {
    if (*cap >= n) return DCREG_OK;
    if (*p) cudaFree(*p);
    *p = nullptr; *cap = 0;
    CK(cudaMalloc(p, (size_t)n * sizeof(T)));
    *cap = n;
    return DCREG_OK;
}

// per-trial loop state: IcpState, ticket, sums, initial poses
int ensure_trials(dcreg_ctx* ctx, int trials) {
    if (ctx->trials_cap >= trials) return DCREG_OK;
    void* old[] = {ctx->d_counter, ctx->d_acc, ctx->d_state, ctx->d_T_init};
    for (void* p : old)
        if (p) cudaFree(p);
    ctx->d_counter = nullptr; ctx->d_acc = nullptr; ctx->d_state = nullptr; ctx->d_T_init = nullptr; ctx->trials_cap = 0;
    CK(cudaMalloc(&ctx->d_counter, (size_t)trials * sizeof(unsigned int)));
    CK(cudaMemsetAsync(ctx->d_counter, 0, (size_t)trials * sizeof(unsigned int), ctx->stream));
    CK(cudaMalloc(&ctx->d_acc, (size_t)trials * kAcc * sizeof(double)));
    CK(cudaMalloc(&ctx->d_state, (size_t)trials * sizeof(IcpState)));
    CK(cudaMemsetAsync(ctx->d_state, 0, (size_t)trials * sizeof(IcpState), ctx->stream));
    CK(cudaMalloc(&ctx->d_T_init, (size_t)trials * 16 * sizeof(double)));
    ctx->trials_cap = trials;
    ctx->drop_graphs();
    return DCREG_OK;
}

// launch with the programmatic-stream-serialization attribute (see pdl_wait)
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args... args) {
    static int use = -1;
    if (use < 0) use = getenv("DCREG_NO_PDL") ? 0 : 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = use ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

// grid size for streaming kernels: a multiple of the SM count
int stream_grid(const dcreg_ctx* ctx, long long n, int per_sm) {
    long long need = (n + kBlock - 1) / kBlock;
    long long cap = (long long)ctx->sm_count * per_sm;
    if (need < 1) need = 1;
    return (int)(need < cap ? need : cap);
}

// d_radius: max |p| (one float), or with scan_off ([n_scans + 1], device) one per scan
int upload_points(dcreg_ctx* ctx, const float* xyz, long long n, int stride, float4* d_out, float* d_radius,
                  const long long* scan_off = nullptr, int n_scans = 0) {
    const size_t bytes = (size_t)n * stride * sizeof(float);
    if (ctx->stage_bytes < bytes) {
        if (ctx->d_stage) cudaFree(ctx->d_stage);
        ctx->d_stage = nullptr; ctx->stage_bytes = 0;
        CK(cudaMalloc(&ctx->d_stage, bytes));
        ctx->stage_bytes = bytes;
    }
    CK(cudaMemcpyAsync(ctx->d_stage, xyz, bytes, cudaMemcpyHostToDevice, ctx->stream));
    if (d_radius) CK(cudaMemsetAsync(d_radius, 0, (scan_off ? n_scans : 1) * sizeof(float), ctx->stream));
    pack_source_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(ctx->d_stage, n, stride, d_out, d_radius,
                                                                              scan_off, n_scans);
    ctx->launches++;
    CK(cudaGetLastError());
    return DCREG_OK;
}

template <typename PlaneT, bool kUseWd, int kTeamCtas>
int launch_reduce_k(dcreg_ctx* ctx, k1s::Args& a, int g) {
    auto kern = k1s::reduce_stream_kernel<PlaneT, kUseWd, kTeamCtas>;
    const size_t smem = sizeof(k1s::Smem<PlaneT>);
    // function attributes are per device: one flag per context (= per device) and kernel variant, not per process
    bool& configured = ctx->k1_attr_done[(sizeof(PlaneT) == 32 ? 2 : 0) + (kUseWd ? 1 : 0)];
    if (!configured) {
        CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CK(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        configured = true;
    }
    kern<<<g, k1s::kThreads, smem, ctx->stream>>>(a);
    ctx->launches++;
    CK(cudaGetLastError());
    return DCREG_OK;
}

template <typename PlaneT, bool kUseWd>
int launch_reduce_t(dcreg_ctx* ctx, k1s::Args& a) {
    // persistent grid: every SM holds 2 CTAs (launch bounds; 2 x (32 KB / 48 KB ring) fits the 227 KB carveout)
    const long long nchunks = (a.n + 31) / 32;
    long long g = (long long)ctx->sm_count * 2;
    const long long need = (nchunks + k1s::kWarpsPerBlock - 1) / k1s::kWarpsPerBlock;
    if (g > need) g = need;
    if (g < 1) g = 1;
    int rc = ensure_partials(ctx, (int)g);
    if (rc) return rc;
    a.partials = ctx->d_partials;
    // team size (k1_stream.cuh): 1, 2, 4, 37 and 296 CTAs per contiguous range all measured 70-71 us on 10 M slots
    return launch_reduce_k<PlaneT, kUseWd, 1>(ctx, a, (int)g);
}

// slope / gate: dcreg_icp_params::weight_slope / weight_gate (0.9 / 0.1 in the reference, icp_test_runner.cpp:1776, 1785)
int launch_reduce(dcreg_ctx* ctx, const float4* d_src, const void* d_plane, bool f64, long long n,
                  const k1::Pose* pose, int use_wd, double slope = 0.9, double gate = 0.1, double npt_override = -1.0) {
    k1s::Args a{};
    a.src = d_src; a.plane = d_plane; a.n = n;
    if (pose) a.pose = *pose;
    for (int i = 0; i < 9; ++i) a.Rs[i] = ldexp(a.pose.R[i], 896);      // exact: see k1s::f32_raw
    a.slope = slope; a.gate = gate;
    a.npt_override = npt_override;
    if (ctx->peer_ok) a.peer = ctx->peer_view;                          // the sum over ranks happens inside the kernel
    { static int dbg = -1; if (dbg < 0) { const char* e = getenv("DCREG_K1_DEBUG"); dbg = e ? atoi(e) : 0; } a.debug = dbg; }
    a.counter = ctx->d_counter; a.acc = ctx->d_acc;
    if (use_wd) return f64 ? launch_reduce_t<double4, true>(ctx, a) : launch_reduce_t<float4, true>(ctx, a);
    return f64 ? launch_reduce_t<double4, false>(ctx, a) : launch_reduce_t<float4, false>(ctx, a);
}

// Fallback exchange (no peer mapping): one ncclAllReduce of the 32 sums behind the reducing kernel.
int nccl_allreduce_acc(dcreg_ctx* ctx) {
    if (!ctx->comm || ctx->peer_ok) return DCREG_OK;
    int r = g_nccl.AllReduce(ctx->d_acc, ctx->d_acc, kAcc, kNcclFloat64, kNcclSum, ctx->comm, ctx->stream);
    if (r != 0) {
        ctx->err = std::string("ncclAllReduce: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "error");
        return DCREG_NCCL_ERROR;
    }
    return DCREG_OK;
}

// Results of `trials` registrations: final poses, iteration counts, flags, and up to log_cap records per trial.
// status_out[t] = dcreg_status of trial t.
int read_results(dcreg_ctx* ctx, int trials, double* T_out, dcreg_iter_log* log, int log_cap, int* n_iterations,
                 int* converged, int* status_out) {
    int rc = ensure_pinned(ctx, (size_t)trials * sizeof(IcpState));
    if (rc) return rc;
    IcpState* hs = (IcpState*)ctx->h_pinned;
    CK(cudaMemcpyAsync(hs, ctx->d_state, (size_t)trials * sizeof(IcpState), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (int t = 0; t < trials; ++t) {
        if (T_out) {
            double* To = T_out + (size_t)t * 16;
            for (int r = 0; r < 3; ++r) {
                for (int c = 0; c < 3; ++c) To[r * 4 + c] = hs[t].R[r * 3 + c];
                To[r * 4 + 3] = hs[t].t[r];
            }
            To[12] = To[13] = To[14] = 0.0; To[15] = 1.0;
        }
        if (n_iterations) n_iterations[t] = hs[t].iter;
        if (converged) converged[t] = hs[t].converged;
        if (status_out) status_out[t] = hs[t].status;
    }
    if (log && log_cap > 0) {
        if (trials == 1) {
            const int iters = hs[0].iter;
            int nrec = iters < log_cap ? iters : log_cap;
            // a NOT_ENOUGH_POINTS abort still wrote a record at index iters-1; a NONFINITE abort at index iters
            if (hs[0].status == DCREG_NONFINITE_UPDATE && iters < log_cap) nrec = iters + 1;
            if (nrec > 0)
                CK(cudaMemcpyAsync(log, ctx->d_log, (size_t)nrec * sizeof(dcreg_iter_log), cudaMemcpyDeviceToHost, ctx->stream));
        } else {
            CK(cudaMemcpyAsync(log, ctx->d_log, (size_t)trials * log_cap * sizeof(dcreg_iter_log), cudaMemcpyDeviceToHost,
                               ctx->stream));
        }
        CK(cudaStreamSynchronize(ctx->stream));
    }
    if (ctx->peer_ok) {                                 // a peer that never posted (timeout in peer::all_reduce32)
        unsigned int perr = 0;
        CK(cudaMemcpyAsync(&perr, &ctx->d_mailbox->error, sizeof(perr), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        if (perr) { ctx->err = "peer all-reduce timed out waiting for rank " + std::to_string((int)perr - 1); return DCREG_NCCL_ERROR; }
    }
    return DCREG_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
extern "C" {

int dcreg_abi_version(void) { return DCREG_ABI_VERSION; }

void dcreg_default_params(dcreg_icp_params* p) {
    if (!p) return;
    memset(p, 0, sizeof(*p));
    p->search_radius = 1.0; p->max_iterations = 30;
    p->detection = DCREG_DET_SCHUR_CONDITION_NUMBER; p->handling = DCREG_HAND_PRECONDITIONED_CG;
    p->use_weight_derivative = 0;
    p->conv_thresh_rot = 1e-5; p->conv_thresh_trans = 1e-3;
    p->cond_thresh = 10.0; p->eig_thresh = 120.0; p->kappa_target = 1.0;
    p->pcg_tol = 1e-6; p->pcg_max_iter = 10; p->std_reg_gamma = 0.01;
    p->plane_thickness = 0.2; p->weight_slope = 0.9; p->weight_gate = 0.1; p->min_normal_norm = 1e-6;
    p->min_effective_points = 10; p->fixed_iterations = 0;
}

int dcreg_create(int device_id, dcreg_ctx** out) {
    if (!out) return DCREG_BAD_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) return DCREG_NO_DEVICE;   // no CPU fallback
    if (device_id < 0 || device_id >= ndev) return DCREG_BAD_ARG;
    dcreg_ctx* ctx = new dcreg_ctx();
    ctx->device = device_id;
    *out = ctx;   // returned even on failure so the caller can read dcreg_last_error
    CK(cudaSetDevice(device_id));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device_id));
    ctx->sm_count = prop.multiProcessorCount;
    CK(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    {
        const int rc = ensure_trials(ctx, 1);
        if (rc) return rc;
    }
    CK(cudaMalloc(&ctx->d_n_active, sizeof(unsigned int)));
    CK(cudaMemsetAsync(ctx->d_n_active, 0, sizeof(unsigned int), ctx->stream));
    CK(cudaMalloc(&ctx->d_small, 1024 * sizeof(double)));
    if (!getenv("DCREG_NO_K2_REHEARSAL")) {
        CK(cudaMalloc(&ctx->d_k2_scratch, sizeof(K2Scratch)));
        CK(cudaMemsetAsync(ctx->d_k2_scratch, 0, sizeof(K2Scratch), ctx->stream));
    }
    CK(cudaMalloc(&ctx->d_analysis, sizeof(dcreg_analysis)));
    CK(cudaStreamSynchronize(ctx->stream));
    return DCREG_OK;
}

int dcreg_destroy(dcreg_ctx* ctx) {
    if (!ctx) return DCREG_BAD_ARG;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    dcreg_comm_destroy(ctx);
    ctx->drop_graphs();
    void* ptrs[] = {ctx->d_n_active, ctx->d_T_init, ctx->d_sort_tmp, ctx->d_src, ctx->d_stage, ctx->d_tgt, ctx->grid.keys, ctx->grid.cell_start, ctx->grid.hstart,
                    ctx->grid.hcount, ctx->d_src_sorted, ctx->d_cell_tmp, ctx->d_pt_cell, ctx->d_tile_sums,
                    ctx->grid.pts, ctx->grid.pos_of, ctx->d_planes64, ctx->d_planes32, ctx->d_partials, ctx->d_counter, ctx->d_acc,
                    ctx->d_state, ctx->d_log, ctx->d_small, ctx->d_analysis, ctx->d_flush, ctx->d_nn, ctx->d_plane_cache, ctx->d_fit_state, ctx->d_iter_stats, ctx->d_src_radius, ctx->d_plane_key, ctx->d_k2_scratch,
                    ctx->d_cov, ctx->d_scan, ctx->d_scan_sorted, ctx->d_scan_keys, ctx->d_scan_slots, ctx->d_scan_sort_tmp, ctx->d_scan_off, ctx->d_scan_radius,
                    ctx->src_grid.keys, ctx->src_grid.cell_start, ctx->src_grid.hstart, ctx->src_grid.hcount, ctx->src_grid.pts, ctx->src_grid.pos_of, ctx->d_p2p};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    if (ctx->h_pinned) cudaFreeHost(ctx->h_pinned);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return DCREG_OK;
}

const char* dcreg_last_error(const dcreg_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }
void* dcreg_stream(dcreg_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
int64_t dcreg_launch_count(const dcreg_ctx* ctx) { return ctx ? ctx->launches : 0; }
void* dcreg_device_source(dcreg_ctx* ctx) { return ctx ? ctx->d_src : nullptr; }
void* dcreg_device_planes_f64(dcreg_ctx* ctx) { return ctx ? ctx->d_planes64 : nullptr; }
void* dcreg_device_planes_f32(dcreg_ctx* ctx) { return ctx ? ctx->d_planes32 : nullptr; }

static void free_grid(corr::Grid* g);

int dcreg_set_source(dcreg_ctx* ctx, const float* xyz, int64_t n, int stride) {
    if (!ctx) return DCREG_BAD_ARG;
    if (!xyz || n <= 0 || stride < 3) { ctx->err = "dcreg_set_source: empty cloud or stride < 3"; return DCREG_BAD_ARG; }
    CK(cudaSetDevice(ctx->device));
    free_grid(&ctx->src_grid);
    ctx->has_src_grid = false;
    if (ctx->n_src_cap < n) {
        if (ctx->d_src) cudaFree(ctx->d_src);
        ctx->d_src = nullptr; ctx->n_src_cap = 0;
        CK(cudaMalloc(&ctx->d_src, (size_t)n * sizeof(float4)));
        ctx->n_src_cap = n;
    }
    ctx->n_src = n;
    if (ctx->nranks == 1) ctx->n_src_total = n;
    if (!ctx->d_src_radius) CK(cudaMalloc(&ctx->d_src_radius, sizeof(float)));
    return upload_points(ctx, xyz, n, stride, ctx->d_src, ctx->d_src_radius);
}

int dcreg_set_global_source_count(dcreg_ctx* ctx, int64_t n_total) {
    if (!ctx || n_total <= 0) return DCREG_BAD_ARG;
    ctx->n_src_total = n_total;
    return DCREG_OK;
}

// exclusive scan of `n` ints (in -> out) on ctx's stream; tile_sums is ctx-owned scratch
static int device_exclusive_scan(dcreg_ctx* ctx, const int* in, long long n, int* out) {
    const int ntiles = (int)((n + corr::kScanTile - 1) / corr::kScanTile);
    if (ctx->tile_sums_cap < ntiles) {
        if (ctx->d_tile_sums) cudaFree(ctx->d_tile_sums);
        ctx->d_tile_sums = nullptr; ctx->tile_sums_cap = 0;
        CK(cudaMalloc(&ctx->d_tile_sums, (size_t)ntiles * sizeof(int)));
        ctx->tile_sums_cap = ntiles;
    }
    corr::scan_tile_sums_kernel<<<ntiles, 256, 0, ctx->stream>>>(in, (int)n, ctx->d_tile_sums);
    corr::scan_tile_offsets_kernel<<<1, 1024, 0, ctx->stream>>>(ctx->d_tile_sums, ntiles);
    corr::scan_tile_apply_kernel<<<ntiles, 256, 0, ctx->stream>>>(in, (int)n, ctx->d_tile_sums, out);
    ctx->launches += 3;
    CK(cudaGetLastError());
    return DCREG_OK;
}

static void free_grid(corr::Grid* g) {
    void* ptrs[] = {g->keys, g->cell_start, g->hstart, g->hcount, g->pts, g->pos_of};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    *g = corr::Grid{};
}

// Group `m` device points by uniform-grid cell (dense when the bounding box has <= kMaxDenseCells cells, hash table
// otherwise).  Replaces the kd-tree build of ICPContext::setTargetCloud (utils.hpp:393-424).  Synchronises the stream.
static int build_grid(dcreg_ctx* ctx, const float4* d_pts, long long m, double cell_size, corr::Grid* gout,
                      long long* ncells_out) {
    corr::Grid g{};
    g.n = (int)m; g.inv_cell = 1.0 / cell_size; g.rings = 1;
    CK(cudaMalloc(&g.pts, (size_t)m * sizeof(float4)));
    CK(cudaMalloc(&g.pos_of, (size_t)m * sizeof(int)));
    int hb[6] = {1 << 30, 1 << 30, 1 << 30, -(1 << 30), -(1 << 30), -(1 << 30)};
    int* d_bounds = (int*)(ctx->d_small + 512);
    CK(cudaMemcpyAsync(d_bounds, hb, sizeof(hb), cudaMemcpyHostToDevice, ctx->stream));
    corr::grid_bounds_kernel<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(d_pts, (int)m, g.inv_cell, d_bounds);
    ctx->launches++;
    CK(cudaMemcpyAsync(hb, d_bounds, sizeof(hb), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (int k = 0; k < 3; ++k)
        if (hb[k] < -(1 << 19) || hb[3 + k] > (1 << 19)) {
            cudaFree(g.pts); cudaFree(g.pos_of);
            ctx->err = "grid build: coordinates / cell_size exceed the +-2^19 cell range (NaN or huge coordinates?)";
            return DCREG_BAD_ARG;
        }
    const long long nx = (long long)hb[3] - hb[0] + 1, ny = (long long)hb[4] - hb[1] + 1, nz = (long long)hb[5] - hb[2] + 1;
    const long long ncells = nx * ny * nz;
    const unsigned nb = (unsigned)((m + 255) / 256);
    int *pt_cell = nullptr, *fill = nullptr, *counts = nullptr;
    float4* tmp_pts = nullptr;                      // points grouped by cell in arrival order, before the in-cell ranking
    CK(cudaMalloc(&pt_cell, (size_t)m * sizeof(int)));
    cudaError_t e = cudaSuccess;
    int rc = DCREG_OK;
    if (ncells <= corr::kMaxDenseCells) {
        g.dense = 1; g.ox = hb[0]; g.oy = hb[1]; g.oz = hb[2]; g.nx = (int)nx; g.ny = (int)ny; g.nz = (int)nz;
        if (ncells_out) *ncells_out = ncells;
        CK(cudaMalloc(&g.cell_start, (size_t)(ncells + 1) * sizeof(int)));
        CK(cudaMalloc(&counts, (size_t)(ncells + 1) * sizeof(int)));
        CK(cudaMalloc(&fill, (size_t)ncells * sizeof(int)));
        CK(cudaMemsetAsync(counts, 0, (size_t)(ncells + 1) * sizeof(int), ctx->stream));
        CK(cudaMemsetAsync(fill, 0, (size_t)ncells * sizeof(int), ctx->stream));
        corr::grid_count_dense_kernel<<<nb, 256, 0, ctx->stream>>>(d_pts, (int)m, g, pt_cell, counts);
        rc = device_exclusive_scan(ctx, counts, ncells + 1, g.cell_start);
        CK(cudaMalloc(&tmp_pts, (size_t)m * sizeof(float4)));
        corr::grid_scatter_kernel<<<nb, 256, 0, ctx->stream>>>(d_pts, (int)m, pt_cell, g.cell_start, fill, tmp_pts, 0);
        corr::grid_rank_cells_kernel<<<nb, 256, 0, ctx->stream>>>(tmp_pts, (int)m, pt_cell, g.cell_start, nullptr, g.pts, g.pos_of);
        ctx->launches += 3;
        e = cudaStreamSynchronize(ctx->stream);
    } else {
        unsigned int cap = 1024;
        while ((long long)cap < 2 * m) cap <<= 1;
        g.dense = 0; g.mask = cap - 1;
        if (ncells_out) *ncells_out = 0;
        CK(cudaMalloc(&g.keys, (size_t)cap * sizeof(unsigned long long)));
        CK(cudaMalloc(&g.hstart, (size_t)cap * sizeof(int)));
        CK(cudaMalloc(&g.hcount, (size_t)cap * sizeof(int)));
        CK(cudaMalloc(&fill, (size_t)cap * sizeof(int)));
        CK(cudaMemsetAsync(g.keys, 0xff, (size_t)cap * sizeof(unsigned long long), ctx->stream));
        CK(cudaMemsetAsync(g.hcount, 0, (size_t)cap * sizeof(int), ctx->stream));
        CK(cudaMemsetAsync(fill, 0, (size_t)cap * sizeof(int), ctx->stream));
        corr::grid_insert_hash_kernel<<<nb, 256, 0, ctx->stream>>>(d_pts, (int)m, g, pt_cell);
        rc = device_exclusive_scan(ctx, g.hcount, cap, g.hstart);
        CK(cudaMalloc(&tmp_pts, (size_t)m * sizeof(float4)));
        corr::grid_scatter_kernel<<<nb, 256, 0, ctx->stream>>>(d_pts, (int)m, pt_cell, g.hstart, fill, tmp_pts, 0);
        corr::grid_rank_cells_kernel<<<nb, 256, 0, ctx->stream>>>(tmp_pts, (int)m, pt_cell, g.hstart, g.hcount, g.pts, g.pos_of);
        ctx->launches += 3;
        e = cudaStreamSynchronize(ctx->stream);
    }
    cudaFree(pt_cell); cudaFree(fill);
    if (tmp_pts) cudaFree(tmp_pts);
    if (counts) cudaFree(counts);
    if (rc) { free_grid(&g); return rc; }
    if (e != cudaSuccess) { free_grid(&g); ctx->err = std::string("grid build: ") + cudaGetErrorString(e); return DCREG_CUDA_ERROR; }
    CK(cudaGetLastError());
    *gout = g;
    return DCREG_OK;
}

int dcreg_set_target(dcreg_ctx* ctx, const float* xyz, int64_t m, int stride, double cell_size) {
    if (!ctx) return DCREG_BAD_ARG;
    if (!xyz || m <= 0 || stride < 3 || !(cell_size > 0.0) || m > 0x7fffffffLL) {
        ctx->err = "dcreg_set_target: empty cloud, stride < 3, cell_size <= 0 or too many points";
        return DCREG_BAD_ARG;
    }
    CK(cudaSetDevice(ctx->device));
    if (ctx->d_tgt) cudaFree(ctx->d_tgt);
    ctx->d_tgt = nullptr;
    free_grid(&ctx->grid);
    ctx->has_grid = false;
    free_grid(&ctx->src_grid);   // built with the target's cell size
    ctx->has_src_grid = false;
    CK(cudaMalloc(&ctx->d_tgt, (size_t)m * sizeof(float4)));
    ctx->n_tgt = m;
    int rc = upload_points(ctx, xyz, m, stride, ctx->d_tgt, nullptr);
    if (rc) return rc;
    ctx->cell_size = cell_size;
    if ((rc = build_grid(ctx, ctx->d_tgt, m, cell_size, &ctx->grid, &ctx->grid_cells))) return rc;
    ctx->has_grid = true;
    return DCREG_OK;
}

// Post-run point-to-point metrics, replaces calculatePointToPointError (DCReg/include/utils.hpp:538-589; called at
// icp_test_runner.cpp:506-510 and once per CSV row at :1463-1470): forward exact 1-NN aligned source -> target
// (RMSE over ALL source points of the distances below the threshold, fitness, mean distance), backward exact 1-NN
// target -> aligned source, Chamfer = mean of the two mean distances.  out = { rmse, fitness, chamfer, n_valid }.
int dcreg_point_to_point_metrics(dcreg_ctx* ctx, const double T[16], double error_threshold, double out[4]) {
    if (!ctx) return DCREG_BAD_ARG;
    if (!T || !out) { ctx->err = "p2p metrics: null pointer"; return DCREG_BAD_ARG; }
    if (!ctx->d_src || !ctx->has_grid || !ctx->d_tgt) { ctx->err = "p2p metrics: set source and target first"; return DCREG_BAD_ARG; }
    if (!ctx->grid.dense) { ctx->err = "p2p metrics need the dense grid (target bounding box too large for this cell size)"; return DCREG_BAD_ARG; }
    CK(cudaSetDevice(ctx->device));
    const long long n = ctx->n_src, m = ctx->n_tgt;
    double* dT = ctx->d_small + 640;
    CK(cudaMemcpyAsync(dT, T, 12 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    const int gridf = stream_grid(ctx, n, 8), gridb = stream_grid(ctx, m, 8);
    int rc = ensure_partials(ctx, gridf > gridb ? gridf : gridb);
    if (rc) return rc;
    std::vector<double> hp((size_t)3 * (gridf > gridb ? gridf : gridb));
    // forward
    corr::nn1_metrics_kernel<<<gridf, kBlock, 0, ctx->stream>>>(ctx->d_src, n, dT, ctx->grid, error_threshold, ctx->d_partials);
    ctx->launches++;
    CK(cudaMemcpyAsync(hp.data(), ctx->d_partials, (size_t)3 * gridf * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    double sum_fwd = 0, sum_sq = 0, valid = 0;
    for (int b = 0; b < gridf; ++b) { sum_fwd += hp[3 * b]; sum_sq += hp[3 * b + 1]; valid += hp[3 * b + 2]; }
    // backward: grid over the aligned source
    float4* d_aligned = nullptr;
    CK(cudaMalloc(&d_aligned, (size_t)n * sizeof(float4)));
    corr::transform_points_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(ctx->d_src, n, dT, d_aligned);
    ctx->launches++;
    corr::Grid ga{};
    rc = build_grid(ctx, d_aligned, n, ctx->cell_size, &ga, nullptr);
    if (rc == DCREG_OK && !ga.dense) { rc = DCREG_BAD_ARG; ctx->err = "p2p metrics: aligned cloud spans too many cells"; }
    double sum_bwd = 0;
    if (rc == DCREG_OK) {
        corr::nn1_metrics_kernel<<<gridb, kBlock, 0, ctx->stream>>>(ctx->d_tgt, m, nullptr, ga, error_threshold, ctx->d_partials);
        ctx->launches++;
        cudaMemcpyAsync(hp.data(), ctx->d_partials, (size_t)3 * gridb * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
        cudaError_t e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) { rc = DCREG_CUDA_ERROR; ctx->err = cudaGetErrorString(e); }
        for (int b = 0; b < gridb; ++b) sum_bwd += hp[3 * b];
    }
    free_grid(&ga);
    cudaFree(d_aligned);
    if (rc) return rc;
    out[0] = sqrt(sum_sq / (double)n);
    out[1] = valid / (double)n;
    out[2] = 0.5 * (sum_fwd / (double)n + sum_bwd / (double)m);
    out[3] = valid;
    return DCREG_OK;
}

// upper bound of |p| over the points of a dense grid, from its cell box
static double grid_box_radius(const corr::Grid& g) {
    const double cell = 1.0 / g.inv_cell;
    const int lo[3] = {g.ox, g.oy, g.oz}, len[3] = {g.nx, g.ny, g.nz};
    double s = 0.0;
    for (int k = 0; k < 3; ++k) {
        const double a = fmax(fabs((double)lo[k]), fabs((double)lo[k] + len[k])) * cell;
        s += a * a;
    }
    return sqrt(s) * (1.0 + 1e-9);
}

// Partial sums of one chunk of poses stay below this many doubles (32 MB); the chunk size does not change results.
constexpr long long kP2pChunkDoubles = 1LL << 22;

// dcreg_point_to_point_metrics for many poses: the forward pass is nn1_metrics_kernel's decomposition per pose
// (blockIdx.y), the backward pass searches one cached grid over the source in its own frame instead of building a
// grid over every aligned copy (nn1_search_posed, exact by the bound of p2p_bound.hpp), and p2p_finish_kernel forms
// each pose's metrics from its partials in the host's summation order.  No device allocation once the buffers have grown,
// one synchronisation per call.
int dcreg_point_to_point_metrics_batch(dcreg_ctx* ctx, int n_poses, const double* T, double error_threshold, double* out) {
    if (!ctx) return DCREG_BAD_ARG;
    if (n_poses < 1) { ctx->err = "p2p metrics batch: n_poses < 1"; return DCREG_BAD_ARG; }
    if (!T || !out) { ctx->err = "p2p metrics batch: null pointer"; return DCREG_BAD_ARG; }
    if (!ctx->d_src || !ctx->has_grid || !ctx->d_tgt) { ctx->err = "p2p metrics batch: set source and target first"; return DCREG_BAD_ARG; }
    if (!ctx->grid.dense) { ctx->err = "p2p metrics batch needs the dense grid (target bounding box too large for this cell size)"; return DCREG_BAD_ARG; }
    CK(cudaSetDevice(ctx->device));
    const long long n = ctx->n_src, m = ctx->n_tgt;
    if (!ctx->has_src_grid) {
        if (n > 0x7fffffffLL) { ctx->err = "p2p metrics batch: too many source points"; return DCREG_BAD_ARG; }
        corr::Grid g{};
        int rc = build_grid(ctx, ctx->d_src, n, ctx->cell_size, &g, nullptr);
        if (rc) return rc;
        if (!g.dense) {
            free_grid(&g);
            ctx->err = "p2p metrics batch needs a dense grid over the source (source bounding box too large for this cell size)";
            return DCREG_BAD_ARG;
        }
        ctx->src_grid = g; ctx->has_src_grid = true;
    }
    const corr::Grid& gs = ctx->src_grid;
    const int gridf = stream_grid(ctx, n, 8), gridb = stream_grid(ctx, m, 8);
    const long long part = 3LL * gridf + gridb;                  // partial sums per pose
    long long chunk = std::min<long long>({(long long)n_poses, 65535LL, std::max<long long>(1, kP2pChunkDoubles / part)});
    if (const char* s = getenv("DCREG_P2P_CHUNK")) {             // smaller chunks, for tests of the chunking
        const long long c = atoll(s);
        if (c >= 1 && c < chunk) chunk = c;
    }
    // layout of d_p2p: pose records [n_poses][kPoseRec] | results [n_poses][4] | forward partials | backward partials
    int rc = ensure_buffer(ctx, &ctx->d_p2p, &ctx->p2p_cap, (long long)n_poses * (corr::kPoseRec + 4) + chunk * part);
    if (rc) return rc;
    double* d_rec = ctx->d_p2p;
    double* d_out = d_rec + (size_t)n_poses * corr::kPoseRec;
    double* d_pf = d_out + (size_t)n_poses * 4;
    double* d_pb = d_pf + (size_t)chunk * 3 * gridf;
    const double pmax = grid_box_radius(gs), ymax = grid_box_radius(ctx->grid);
    std::vector<double> rec((size_t)n_poses * corr::kPoseRec, 0.0);
    for (int k = 0; k < n_poses; ++k) {
        double* r = &rec[(size_t)k * corr::kPoseRec];
        memcpy(r, T + (size_t)k * 16, 12 * sizeof(double));
        const p2p_bound::Bound b = p2p_bound::backward_bound(T + (size_t)k * 16, pmax, ymax);
        r[12] = b.margin; r[13] = b.shrink;
    }
    CK(cudaMemcpyAsync(d_rec, rec.data(), rec.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    for (long long c0 = 0; c0 < n_poses; c0 += chunk) {
        const int cnt = (int)std::min<long long>(chunk, n_poses - c0);
        const double* r = d_rec + (size_t)c0 * corr::kPoseRec;
        corr::nn1_metrics_poses_kernel<<<dim3(gridf, cnt), kBlock, 0, ctx->stream>>>(ctx->d_src, n, r, ctx->grid, error_threshold, d_pf);
        corr::nn1_chamfer_poses_kernel<<<dim3(gridb, cnt), kBlock, 0, ctx->stream>>>(ctx->d_tgt, m, r, gs, d_pb);
        corr::p2p_finish_kernel<<<(cnt + 127) / 128, 128, 0, ctx->stream>>>(d_pf, gridf, d_pb, gridb, cnt, n, m, d_out + (size_t)c0 * 4);
        ctx->launches += 3;
        CK(cudaGetLastError());
    }
    CK(cudaMemcpyAsync(out, d_out, (size_t)n_poses * 4 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return DCREG_OK;
}

// Spatial sort of the source by the target cell of T*p (dense grids only): consecutive threads of the iteration
// kernel then query neighbouring cells, so their candidate loads hit the same lines and their trip counts agree.
// The sorted copy carries the original index in .w; the pose moves little during ICP, so one sort per run suffices.
static int sort_source_by_cell(dcreg_ctx* ctx, const double T[16], const float4** src_out) {
    *src_out = ctx->d_src;
    if (!ctx->grid.dense || ctx->n_src > 0x7fffffffLL) return DCREG_OK;
    const long long n = ctx->n_src, ncells = ctx->grid_cells;
    if (ctx->src_sorted_cap < n) {
        if (ctx->d_src_sorted) cudaFree(ctx->d_src_sorted);
        if (ctx->d_sort_tmp) cudaFree(ctx->d_sort_tmp);
        if (ctx->d_pt_cell) cudaFree(ctx->d_pt_cell);
        ctx->d_src_sorted = nullptr; ctx->d_sort_tmp = nullptr; ctx->d_pt_cell = nullptr; ctx->src_sorted_cap = 0;
        CK(cudaMalloc(&ctx->d_src_sorted, (size_t)n * sizeof(float4)));
        CK(cudaMalloc(&ctx->d_sort_tmp, (size_t)n * sizeof(float4)));
        CK(cudaMalloc(&ctx->d_pt_cell, (size_t)n * sizeof(int)));
        ctx->src_sorted_cap = n;
    }
    if (ctx->cell_tmp_cap < 3 * (ncells + 1)) {
        if (ctx->d_cell_tmp) cudaFree(ctx->d_cell_tmp);
        ctx->d_cell_tmp = nullptr; ctx->cell_tmp_cap = 0;
        CK(cudaMalloc(&ctx->d_cell_tmp, (size_t)3 * (ncells + 1) * sizeof(int)));
        ctx->cell_tmp_cap = 3 * (ncells + 1);
    }
    int* counts = ctx->d_cell_tmp;
    int* start = counts + (ncells + 1);
    int* fill = start + (ncells + 1);
    CK(cudaMemsetAsync(counts, 0, (size_t)(ncells + 1) * sizeof(int), ctx->stream));
    CK(cudaMemsetAsync(fill, 0, (size_t)ncells * sizeof(int), ctx->stream));
    double* dT = ctx->d_small + 640;
    CK(cudaMemcpyAsync(dT, T, 12 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    const unsigned nb = (unsigned)((n + 255) / 256);
    corr::source_cell_kernel<<<nb, 256, 0, ctx->stream>>>(ctx->d_src, (int)n, ctx->grid, dT, ctx->d_pt_cell, counts);
    int rc = device_exclusive_scan(ctx, counts, ncells + 1, start);
    if (rc) return rc;
    corr::grid_scatter_kernel<<<nb, 256, 0, ctx->stream>>>(ctx->d_src, (int)n, ctx->d_pt_cell, start, fill, ctx->d_sort_tmp, 0);
    corr::grid_rank_cells_kernel<<<nb, 256, 0, ctx->stream>>>(ctx->d_sort_tmp, (int)n, ctx->d_pt_cell, start, nullptr, ctx->d_src_sorted, nullptr);
    ctx->launches += 3;
    CK(cudaGetLastError());
    *src_out = ctx->d_src_sorted;
    return DCREG_OK;
}

// The scans of one dcreg_icp_run_scans call: scan s = slots [off[s], off[s+1]) of src (device arrays).
struct ScanSet {
    const float4* src;        // as uploaded (w = slot)
    const long long* off;     // [n + 1]
    const float* radius;      // [n] max |p| per scan (lever arm of its rotation steps)
    int n;
    long long total, largest;
};

// sort_source_by_cell for every scan at once: scan s by the target cell of T_init[s] * p (ctx->d_T_init, written by
// init_state), scans kept contiguous, input order inside a cell.  A stable radix sort on (scan << 32 | cell) keys.
static int sort_scans_by_cell(dcreg_ctx* ctx, const ScanSet& S, const float4** src_out) {
    const long long n = S.total;
    unsigned long long* keys = ctx->d_scan_keys;
    int* slots = ctx->d_scan_slots;
    int scan_bits = 1;
    while ((1LL << scan_bits) < S.n) ++scan_bits;
    const unsigned nb = (unsigned)((n + 255) / 256);
    corr::scan_cell_keys_kernel<<<nb, 256, 0, ctx->stream>>>(S.src, (int)n, S.off, S.n, ctx->grid, ctx->d_T_init, keys, slots);
    ctx->launches++;
    CK(cudaGetLastError());
    size_t tmp = 0;
    CK(cub::DeviceRadixSort::SortPairs(nullptr, tmp, keys, keys + n, slots, slots + n, (int)n, 0, 32 + scan_bits, ctx->stream));
    if (ctx->scan_sort_tmp_bytes < tmp) {
        if (ctx->d_scan_sort_tmp) cudaFree(ctx->d_scan_sort_tmp);
        ctx->d_scan_sort_tmp = nullptr; ctx->scan_sort_tmp_bytes = 0;
        CK(cudaMalloc(&ctx->d_scan_sort_tmp, tmp));
        ctx->scan_sort_tmp_bytes = tmp;
    }
    CK(cub::DeviceRadixSort::SortPairs(ctx->d_scan_sort_tmp, tmp, keys, keys + n, slots, slots + n, (int)n, 0, 32 + scan_bits,
                                       ctx->stream));
    corr::gather_points_kernel<<<nb, 256, 0, ctx->stream>>>(S.src, (int)n, slots + n, ctx->d_scan_sorted);
    ctx->launches++;                                  // (the radix sort's own launches are not counted)
    CK(cudaGetLastError());
    *src_out = ctx->d_scan_sorted;
    return DCREG_OK;
}

static double coherent_step_setting() {
    static double v = -1.0;
    if (v < 0.0) { const char* e = getenv("DCREG_COHERENT_STEP"); v = e ? atof(e) : kCoherentStep; }
    return v;
}

// What one loop body looks like for this context: which kernel, its grid, and whether the solve step is inside it.
struct LoopPlan {
    bool fused2 = false;      // icp_iter2_kernel (dense grid): records, work lists, in-kernel solve step
    bool fold_k2 = false;     // the solve / update step runs in the iteration kernel's last block
    int grid_x = 1, trials = 1;
    Iter2Args b{};            // arguments of the fused2 kernel
    IterArgs a{};             // arguments of the one-thread-per-slot kernel (hash grids, seam 1)
    bool use_wd = false;
    const float* scan_radius = nullptr;   // dcreg_icp_run_scans: one lever arm per trial (scan) for the solve kernel
};

// scans: trial t registers scan t of the set (src = the set's slots, sorted); null = every trial the context's source
static int plan_iteration(dcreg_ctx* ctx, const dcreg_icp_params* prm, const float4* src, double4* planes_out, int trials,
                          dcreg_iter_log* dlog, int log_cap, bool want_fold, LoopPlan* plan, const ScanSet* scans = nullptr) {
    LoopPlan& L = *plan;
    L.trials = trials; L.use_wd = prm->use_weight_derivative != 0;
    L.scan_radius = scans ? scans->radius : nullptr;
    IterArgs& a = L.a;
    a.src = src; a.n = scans ? scans->total : ctx->n_src; a.grid = ctx->grid; a.state = ctx->d_state;
    a.counter = ctx->d_counter; a.acc = ctx->d_acc;
    a.planes_out = planes_out; a.prm = *prm;
    {   // rings of cells that cover the search radius (exactness of the 5-NN-within-radius rule)
        const int rings = (int)ceil(prm->search_radius / ctx->cell_size - 1e-9);
        if (rings < 1 || rings > 4) {
            ctx->err = "search_radius / target cell_size must be in (0, 4]: rebuild the target index with a larger cell";
            return DCREG_BAD_ARG;
        }
        a.grid.rings = rings;
    }
    L.fused2 = ctx->grid.dense && !planes_out && a.n <= 0x1fffffffLL && !getenv("DCREG_FUSED_SEARCH");
    if (trials > 1 && !L.fused2) {
        ctx->err = "batched trials need the dense target grid (target bounding box / cell size too large for it)";
        return DCREG_BAD_ARG;
    }
    if (L.fused2) {
        // per-slot records: [trials][slots], or one record per slot of the scan set
        const long long slots = a.n;
        const int rec_trials = scans ? 1 : trials;
        if (ctx->nn_cap < slots || ctx->nn_trials < rec_trials) {
            void* old[] = {ctx->d_nn, ctx->d_plane_cache, ctx->d_fit_state, ctx->d_plane_key};
            for (void* p : old)
                if (p) cudaFree(p);
            ctx->d_nn = nullptr; ctx->d_plane_cache = nullptr; ctx->d_fit_state = nullptr; ctx->d_plane_key = nullptr;
            ctx->nn_cap = 0; ctx->nn_trials = 0;
            const size_t tot = (size_t)slots * (size_t)rec_trials;
            CK(cudaMalloc(&ctx->d_nn, tot * kNnRec * sizeof(int4)));
            CK(cudaMalloc(&ctx->d_plane_cache, tot * sizeof(double4)));
            CK(cudaMalloc(&ctx->d_fit_state, tot));
            CK(cudaMalloc(&ctx->d_plane_key, tot * 5 * sizeof(int)));
            ctx->nn_cap = slots; ctx->nn_trials = rec_trials;
            ctx->nn_valid = false;
        }
        // blocks per trial and slots per block: loop_plan.hpp (scans: planned for the largest; blocks past the end of a
        // smaller scan post zero partials)
        const char* tile_env = trials == 1 ? getenv("DCREG_TILE") : nullptr;            // measurement switch
        const loop_plan::Tiles tp = loop_plan::plan_tiles(scans ? scans->largest : slots, trials, ctx->sm_count, kBlock,
                                                          tile_env ? atoi(tile_env) : 0);
        L.grid_x = (int)tp.grid_x;
        L.b.tile = tp.tile;
        int rc = ensure_partials(ctx, L.grid_x * trials);
        if (rc) return rc;
        a.partials = ctx->d_partials;
        Iter2Args& b = L.b;
        b.it = a;
        b.nn = ctx->d_nn; b.plane_cache = ctx->d_plane_cache; b.fit_state = ctx->d_fit_state; b.plane_key = ctx->d_plane_key;
        b.force = ctx->force_coherent ? 1 : 0;
        { static int cm = -1; if (cm < 0) { const char* e = getenv("DCREG_COOP_MAX"); cm = e ? atoi(e) : kSearchListMax; } b.coop_max = cm; }
        b.use_seeds = ctx->nn_valid ? 1 : 0;
        { static float lk = -1.f; if (lk < 0.f) { const char* e = getenv("DCREG_LOOK"); lk = e ? (float)atof(e) : kNnLook; } b.look = lk; }
        b.stats = ctx->d_iter_stats;
        const double r2 = prm->search_radius * prm->search_radius;
        float r2f = (float)r2;
        if ((double)r2f < r2) r2f = nextafterf(r2f, INFINITY);
        b.r2_up = r2f;
        // the solve step inside the kernel unless the sum over ranks has to go through NCCL
        L.fold_k2 = want_fold && !(ctx->comm && !ctx->peer_ok) && !getenv("DCREG_NO_FOLD") &&
                    prm->detection == DCREG_DET_SCHUR_CONDITION_NUMBER && prm->handling == DCREG_HAND_PRECONDITIONED_CG;
        b.fold_k2 = L.fold_k2 ? 1 : 0;
        b.log = dlog; b.log_cap = log_cap;
        b.src_radius = scans ? scans->radius : ctx->d_src_radius; b.coherent_step = coherent_step_setting();
        b.scan_off = scans ? scans->off : nullptr;
        b.n_active = ctx->d_n_active;
        if (ctx->peer_ok) b.peer = ctx->peer_view;
        if (!ctx->loop_attr_done) {          // per device (= per context), not per process
            for (auto kern : {icp_iter2_kernel<true, false>, icp_iter2_kernel<false, false>, icp_iter2_kernel<true, true>,
                              icp_iter2_kernel<false, true>}) {
                CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Iter2Smem)));
                CK(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
            }
            ctx->loop_attr_done = true;
        }
    } else {
        L.grid_x = stream_grid(ctx, a.n, 16);
        int rc = ensure_partials(ctx, L.grid_x);
        if (rc) return rc;
        a.partials = ctx->d_partials;
        L.fold_k2 = false;
    }
    return DCREG_OK;
}

// enqueue the iteration kernel of a plan (inside or outside a stream capture)
static int launch_plan(dcreg_ctx* ctx, LoopPlan& L) {
    if (L.fused2) {
        L.b.use_seeds = ctx->nn_valid ? 1 : 0;
        ctx->nn_valid = true;
        const dim3 grid((unsigned)L.grid_x, (unsigned)L.trials);
        auto kern = L.b.scan_off ? (L.use_wd ? icp_iter2_kernel<true, true> : icp_iter2_kernel<false, true>)
                                 : (L.use_wd ? icp_iter2_kernel<true, false> : icp_iter2_kernel<false, false>);
        CK(launch_pdl(kern, grid, dim3(kBlock), sizeof(Iter2Smem), ctx->stream, L.b));
    } else {
        if (L.use_wd) icp_iteration_kernel<true><<<L.grid_x, kBlock, 0, ctx->stream>>>(L.a);
        else icp_iteration_kernel<false><<<L.grid_x, kBlock, 0, ctx->stream>>>(L.a);
    }
    ctx->launches++;
    CK(cudaGetLastError());
    return DCREG_OK;
}

// the separate solve kernel (one warp per trial): baseline methods, hash-grid / seam paths, NCCL fallback of a sharded run.
// scan_radius: [trials] lever arms of a scan set, or null (the context's source)
static int launch_k2(dcreg_ctx* ctx, const dcreg_icp_params* prm, dcreg_iter_log* dlog, int log_cap, int trials = 1,
                     const float* scan_radius = nullptr) {
    CK(launch_pdl(k2_step_kernel, dim3((unsigned)trials), dim3(32), 0, ctx->stream, (const double*)ctx->d_acc, ctx->d_state, *prm,
                  dlog, log_cap, scan_radius ? scan_radius : (const float*)ctx->d_src_radius, scan_radius ? 1 : 0,
                  coherent_step_setting(),
                  trials == 1 ? ctx->d_k2_scratch : (K2Scratch*)nullptr, ctx->d_n_active));
    ctx->launches++;
    return DCREG_OK;
}

// one loop body: iteration kernel [+ all-reduce + solve kernel when the step is not folded]
static int launch_body(dcreg_ctx* ctx, LoopPlan& L, const dcreg_icp_params* prm, dcreg_iter_log* dlog, int log_cap, bool with_k2) {
    int rc = launch_plan(ctx, L);
    if (rc) return rc;
    if (with_k2 && !L.fold_k2) {
        if ((rc = nccl_allreduce_acc(ctx))) return rc;          // no-op on one GPU / with peer mailboxes
        if ((rc = launch_k2(ctx, prm, dlog, log_cap, L.trials, L.scan_radius))) return rc;
    }
    return DCREG_OK;
}

static int init_state(dcreg_ctx* ctx, const double* T, int trials = 1, const long long* scan_off = nullptr) {
    ctx->nn_valid = false;            // a new run: no neighbours of a previous iteration to seed the search with
    int rc = ensure_trials(ctx, trials);
    if (rc) return rc;
    ctx->last_trials = trials;
    CK(cudaMemcpyAsync(ctx->d_T_init, T, (size_t)trials * 16 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    init_state_kernel<<<(trials + 127) / 128, 128, 0, ctx->stream>>>(ctx->d_state, ctx->d_T_init, ctx->n_src_total, ctx->d_counter,
                                                                   trials, ctx->d_n_active, scan_off);
    ctx->launches++;
    CK(cudaGetLastError());
    return DCREG_OK;
}

int dcreg_find_planes(dcreg_ctx* ctx, const double T[16], double search_radius, double* planes_out,
                      int64_t* n_corr_pt) {
    if (!ctx || !T) return DCREG_BAD_ARG;
    if (!ctx->d_src || !ctx->has_grid) { ctx->err = "dcreg_find_planes: set source and target first"; return DCREG_BAD_ARG; }
    CK(cudaSetDevice(ctx->device));
    int rc = ensure_planes(ctx, ctx->n_src);
    if (rc) return rc;
    dcreg_icp_params prm;
    dcreg_default_params(&prm);
    prm.search_radius = search_radius;
    prm.min_effective_points = 0;
    if ((rc = init_state(ctx, T))) return rc;
    LoopPlan L;
    if ((rc = plan_iteration(ctx, &prm, ctx->d_src, ctx->d_planes64, 1, nullptr, 0, false, &L))) return rc;
    if ((rc = launch_plan(ctx, L))) return rc;
    double acc[kAcc];
    CK(cudaMemcpyAsync(acc, ctx->d_acc, sizeof(acc), cudaMemcpyDeviceToHost, ctx->stream));
    if (planes_out)
        CK(cudaMemcpyAsync(planes_out, ctx->d_planes64, (size_t)ctx->n_src * sizeof(double4), cudaMemcpyDeviceToHost,
                           ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (n_corr_pt) *n_corr_pt = (int64_t)(acc[k2::kAccNpt] + 0.5);
    return DCREG_OK;
}

static int reduce_common(dcreg_ctx* ctx, const void* d_src, const void* d_plane, bool f64, int64_t n,
                         const double pose_Rt[12], int use_wd, double out27[27], double stats[3]) {
    if (!ctx) return DCREG_BAD_ARG;
    if (!d_src || !d_plane || n <= 0 || !pose_Rt || !out27) { ctx->err = "reduce: null pointer or n <= 0"; return DCREG_BAD_ARG; }
    CK(cudaSetDevice(ctx->device));
    k1::Pose P;
    for (int i = 0; i < 9; ++i) P.R[i] = pose_Rt[i];
    for (int i = 0; i < 3; ++i) P.t[i] = pose_Rt[9 + i];
    int rc = launch_reduce(ctx, (const float4*)d_src, d_plane, f64, n, &P, use_wd);
    if (rc) return rc;
    if ((rc = nccl_allreduce_acc(ctx))) return rc;
    double acc[kAcc];
    CK(cudaMemcpyAsync(acc, ctx->d_acc, sizeof(acc), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < 27; ++i) out27[i] = acc[i];
    if (stats) { stats[0] = acc[k2::kAccSumR2]; stats[1] = acc[k2::kAccNeff]; stats[2] = acc[k2::kAccNpt]; }
    return DCREG_OK;
}

int dcreg_reduce_normal_equations(dcreg_ctx* ctx, const void* d_src, const void* d_plane, int64_t n,
                                  const double pose_Rt[12], int use_weight_derivative, double out27[27],
                                  double stats[3]) {
    return reduce_common(ctx, d_src, d_plane, false, n, pose_Rt, use_weight_derivative, out27, stats);
}

int dcreg_reduce_normal_equations_f64plane(dcreg_ctx* ctx, const void* d_src, const void* d_plane, int64_t n,
                                           const double pose_Rt[12], int use_weight_derivative, double out27[27],
                                           double stats[3]) {
    return reduce_common(ctx, d_src, d_plane, true, n, pose_Rt, use_weight_derivative, out27, stats);
}

int dcreg_reduce_normal_equations_host(dcreg_ctx* ctx, const float* src4, const void* plane4, int plane_is_f64,
                                       int64_t n, const double pose_Rt[12], int use_weight_derivative,
                                       double out27[27], double stats[3]) {
    if (!ctx) return DCREG_BAD_ARG;
    if (!src4 || !plane4 || n <= 0) { ctx->err = "reduce_host: null pointer or n <= 0"; return DCREG_BAD_ARG; }
    CK(cudaSetDevice(ctx->device));
    int rc = dcreg_set_source(ctx, src4, n, 4);
    if (rc) return rc;
    if ((rc = ensure_planes(ctx, n))) return rc;
    if (plane_is_f64)
        CK(cudaMemcpyAsync(ctx->d_planes64, plane4, (size_t)n * sizeof(double4), cudaMemcpyHostToDevice, ctx->stream));
    else
        CK(cudaMemcpyAsync(ctx->d_planes32, plane4, (size_t)n * sizeof(float4), cudaMemcpyHostToDevice, ctx->stream));
    return reduce_common(ctx, ctx->d_src, plane_is_f64 ? (const void*)ctx->d_planes64 : (const void*)ctx->d_planes32,
                         plane_is_f64 != 0, n, pose_Rt, use_weight_derivative, out27, stats);
}

int dcreg_freeze_planes_f32(dcreg_ctx* ctx) {
    if (!ctx || !ctx->d_planes64 || ctx->n_src <= 0) return DCREG_BAD_ARG;
    CK(cudaSetDevice(ctx->device));
    planes_to_f32_kernel<<<(unsigned)((ctx->n_src + 255) / 256), 256, 0, ctx->stream>>>(ctx->d_planes64, ctx->n_src,
                                                                                        ctx->d_planes32);
    ctx->launches++;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(ctx->stream));
    return DCREG_OK;
}

int dcreg_time_reduce(dcreg_ctx* ctx, int plane_is_f64, const double pose_Rt[12], int use_weight_derivative,
                      int reps, int flush_l2, float* ms_per_launch) {
    if (!ctx || !pose_Rt || reps <= 0 || !ms_per_launch) return DCREG_BAD_ARG;
    if (!ctx->d_src || !ctx->d_planes64) { ctx->err = "time_reduce: no source/planes on the context"; return DCREG_BAD_ARG; }
    CK(cudaSetDevice(ctx->device));
    k1::Pose P;
    for (int i = 0; i < 9; ++i) P.R[i] = pose_Rt[i];
    for (int i = 0; i < 3; ++i) P.t[i] = pose_Rt[9 + i];
    if (flush_l2 && !ctx->d_flush) {
        ctx->flush_n = (256ll << 20) / sizeof(float4);   // 256 MiB > 126 MB L2
        CK(cudaMalloc(&ctx->d_flush, (size_t)ctx->flush_n * sizeof(float4)));
    }
    const void* plane = plane_is_f64 ? (const void*)ctx->d_planes64 : (const void*)ctx->d_planes32;
    int rc = DCREG_OK;
    double total = 0.0;
    if (!flush_l2) {
        // one event pair around the whole batch of back-to-back launches (inputs larger than L2 need no flush)
        cudaEvent_t b0, b1;
        CK(cudaEventCreate(&b0)); CK(cudaEventCreate(&b1));
        CK(cudaEventRecord(b0, ctx->stream));
        for (int i = 0; i < reps && rc == DCREG_OK; ++i) {
            rc = launch_reduce(ctx, ctx->d_src, plane, plane_is_f64 != 0, ctx->n_src, &P, use_weight_derivative);
            if (rc == DCREG_OK) rc = nccl_allreduce_acc(ctx);      // sharded: the 32-double all-reduce is part of the step
        }
        CK(cudaEventRecord(b1, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        float ms = 0.f;
        cudaEventElapsedTime(&ms, b0, b1);
        total = ms;
        cudaEventDestroy(b0); cudaEventDestroy(b1);
    } else {
        std::vector<cudaEvent_t> e0(reps), e1(reps);
        for (int i = 0; i < reps; ++i) { CK(cudaEventCreate(&e0[i])); CK(cudaEventCreate(&e1[i])); }
        for (int i = 0; i < reps && rc == DCREG_OK; ++i) {
            flush_l2_kernel<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(ctx->d_flush, ctx->flush_n, (float)i);
            ctx->launches++;
            CK(cudaEventRecord(e0[i], ctx->stream));
            rc = launch_reduce(ctx, ctx->d_src, plane, plane_is_f64 != 0, ctx->n_src, &P, use_weight_derivative);
            if (rc == DCREG_OK) rc = nccl_allreduce_acc(ctx);
            CK(cudaEventRecord(e1[i], ctx->stream));
        }
        CK(cudaStreamSynchronize(ctx->stream));
        for (int i = 0; i < reps; ++i) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, e0[i], e1[i]);
            total += ms;
            cudaEventDestroy(e0[i]); cudaEventDestroy(e1[i]);
        }
    }
    *ms_per_launch = (float)(total / reps);
    return rc;
}

int dcreg_iteration_counters(dcreg_ctx* ctx, int enable, uint64_t out[2]) {
    if (!ctx || !out) return DCREG_BAD_ARG;
    CK(cudaSetDevice(ctx->device));
    out[0] = out[1] = 0;
    if (ctx->d_iter_stats) {
        unsigned int h[2] = {0, 0};
        CK(cudaMemcpyAsync(h, ctx->d_iter_stats, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        out[0] = h[0]; out[1] = h[1];
    }
    if (enable && !ctx->d_iter_stats) CK(cudaMalloc(&ctx->d_iter_stats, 2 * sizeof(unsigned int)));
    if (!enable && ctx->d_iter_stats) { cudaFree(ctx->d_iter_stats); ctx->d_iter_stats = nullptr; }
    if (ctx->d_iter_stats) CK(cudaMemsetAsync(ctx->d_iter_stats, 0, 2 * sizeof(unsigned int), ctx->stream));
    return DCREG_OK;
}

int dcreg_time_iteration(dcreg_ctx* ctx, const dcreg_icp_params* params, const double T[16], int what, int reps,
                         float* ms_per_body) {
    if (!ctx || !params || !T || reps <= 0 || !ms_per_body) return DCREG_BAD_ARG;
    if (!ctx->d_src || !ctx->has_grid) { ctx->err = "time_iteration: set source and target first"; return DCREG_BAD_ARG; }
    CK(cudaSetDevice(ctx->device));
    dcreg_icp_params prm = *params;
    prm.fixed_iterations = 1;
    prm.max_iterations = reps + 8;
    int rc;
    if ((rc = init_state(ctx, T))) return rc;
    const float4* src_iter = ctx->d_src;
    if ((rc = sort_source_by_cell(ctx, T, &src_iter))) return rc;
    ctx->force_coherent = (what == 0);                                     // fixed pose: measure the record-reusing mode
    LoopPlan L;
    rc = plan_iteration(ctx, &prm, src_iter, nullptr, 1, nullptr, 0, what == 1, &L);
    ctx->force_coherent = false;
    if (rc) return rc;
    for (int warm = 0; warm < 2; ++warm)                                   // instruction caches, lazy module load
        if ((rc = launch_body(ctx, L, &prm, nullptr, 0, false))) return rc;
    cudaEvent_t b0, b1;
    CK(cudaEventCreate(&b0)); CK(cudaEventCreate(&b1));
    CK(cudaEventRecord(b0, ctx->stream));
    for (int i = 0; i < reps; ++i)
        if ((rc = launch_body(ctx, L, &prm, nullptr, 0, what == 1))) return rc;
    CK(cudaEventRecord(b1, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, b0, b1);
    cudaEventDestroy(b0); cudaEventDestroy(b1);
    *ms_per_body = ms / reps;
    return DCREG_OK;
}

int dcreg_iteration_timeline(dcreg_ctx* ctx, const dcreg_icp_params* params, const double T[16], int iters, uint64_t* out,
                             int out_cap_blocks, int* n_blocks) {
    if (!ctx || !params || !T || iters < 1 || !out || !n_blocks) return DCREG_BAD_ARG;
    if (!ctx->d_src || !ctx->has_grid) { ctx->err = "iteration_timeline: set source and target first"; return DCREG_BAD_ARG; }
    CK(cudaSetDevice(ctx->device));
    dcreg_icp_params prm = *params;
    prm.fixed_iterations = 1;
    prm.max_iterations = iters + 8;
    int rc;
    if ((rc = init_state(ctx, T))) return rc;
    const float4* src_iter = ctx->d_src;
    if ((rc = sort_source_by_cell(ctx, T, &src_iter))) return rc;
    LoopPlan L;
    if ((rc = plan_iteration(ctx, &prm, src_iter, nullptr, 1, nullptr, 0, true, &L))) return rc;
    if (!L.fused2) { ctx->err = "iteration_timeline: needs the dense-grid loop kernel"; return DCREG_BAD_ARG; }
    *n_blocks = L.grid_x;
    if (out_cap_blocks < L.grid_x + 1) { ctx->err = "iteration_timeline: output too small"; return DCREG_BAD_ARG; }
    const size_t bytes = (size_t)(L.grid_x + 1) * kStampSlots * sizeof(unsigned long long);
    unsigned long long* d_st = nullptr;
    CK(cudaMalloc(&d_st, bytes));
    CK(cudaMemsetAsync(d_st, 0, bytes, ctx->stream));
    for (int i = 0; i + 1 < iters && rc == DCREG_OK; ++i) rc = launch_body(ctx, L, &prm, nullptr, 0, true);
    L.b.stamps = d_st;
    if (rc == DCREG_OK) rc = launch_body(ctx, L, &prm, nullptr, 0, true);
    if (rc == DCREG_OK) {
        cudaMemcpyAsync(out, d_st, bytes, cudaMemcpyDeviceToHost, ctx->stream);
        if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) { ctx->err = "iteration_timeline: stream error"; rc = DCREG_CUDA_ERROR; }
    }
    cudaFree(d_st);
    return rc;
}

int dcreg_analyze_and_solve(dcreg_ctx* ctx, const double H27[27], const dcreg_icp_params* params,
                            dcreg_analysis* out, double dx[6]) {
    if (!ctx) return DCREG_BAD_ARG;
    if (!H27 || !params || !out || !dx) { ctx->err = "analyze_and_solve: null pointer"; return DCREG_BAD_ARG; }
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(ctx->d_small, H27, 27 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    k2_analyze_kernel<<<1, 32, 0, ctx->stream>>>(ctx->d_small, *params, ctx->d_analysis, ctx->d_small + 32);
    ctx->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, ctx->d_analysis, sizeof(dcreg_analysis), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(dx, ctx->d_small + 32, 6 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < 6; ++i)
        if (!isfinite(dx[i])) return DCREG_NONFINITE_UPDATE;
    return DCREG_OK;
}

int dcreg_solve_pcg(dcreg_ctx* ctx, const double A[36], const double b[6], const double P[36], int max_iterations,
                    double tolerance, double x[6], int* iterations) {
    if (!ctx) return DCREG_BAD_ARG;
    if (!A || !b || !P || !x) { ctx->err = "solve_pcg: null pointer"; return DCREG_BAD_ARG; }
    CK(cudaSetDevice(ctx->device));
    double* d = ctx->d_small;
    CK(cudaMemcpyAsync(d, A, 36 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d + 36, b, 6 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d + 48, P, 36 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    pcg_kernel<<<1, 32, 0, ctx->stream>>>(d, d + 36, d + 48, max_iterations, tolerance, d + 96, (int*)(d + 128));
    ctx->launches++;
    CK(cudaGetLastError());
    int it = 0;
    CK(cudaMemcpyAsync(x, d + 96, 6 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&it, d + 128, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (iterations) *iterations = it;
    return DCREG_OK;
}

// FNV-1a over the bytes that define a captured chunk of the loop
static void key_bytes(std::vector<unsigned char>& k, const void* p, size_t n) {
    const unsigned char* c = (const unsigned char*)p;
    k.insert(k.end(), c, c + n);
}

// Enqueue `iters` loop bodies.  The bodies are identical launches (pose, mode flags and the done flag live on the
// device), so a chunk is captured once into a CUDA graph and replayed: one host call per chunk instead of one or two
// launches per iteration - what keeps 8 independent ranks from queueing behind the host (round 1: 0.887 weak scaling
// at 8 GPUs with nothing shared between the ranks).  Falls back to plain launches if capture is unavailable.
static int enqueue_iterations(dcreg_ctx* ctx, LoopPlan& L, const dcreg_icp_params* prm, dcreg_iter_log* dlog, int log_cap, int iters) {
    static int use_graph = -1;
    if (use_graph < 0) use_graph = getenv("DCREG_NO_GRAPH") ? 0 : 1;
    const bool graphable = use_graph && !ctx->graph_off && L.fused2 && !L.b.force && iters > 1 &&
                           (L.fold_k2 || !(ctx->comm && !ctx->peer_ok));          // no NCCL call inside a capture
    if (graphable) {
        std::vector<unsigned char> key;
        Iter2Args kb = L.b;
        kb.use_seeds = 0;
        key_bytes(key, &kb, sizeof(kb));
        const int meta[4] = {L.grid_x, L.trials, L.use_wd ? 1 : 0, iters};
        key_bytes(key, meta, sizeof(meta));
        key_bytes(key, prm, sizeof(*prm));
        cudaGraphExec_t exec = nullptr;
        for (size_t gi = 0; gi < ctx->graphs.size(); ++gi)
            if (ctx->graphs[gi].key == key) {
                if (gi != 0) std::swap(ctx->graphs[gi], ctx->graphs[0]);
                exec = ctx->graphs[0].exec;
                break;
            }
        if (!exec) {
            cudaGraph_t graph = nullptr;
            const bool nn_valid0 = ctx->nn_valid;
            const long long launches0 = ctx->launches;
            cudaError_t e = cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeRelaxed);
            int rc = DCREG_OK;
            if (e == cudaSuccess) {
                for (int k = 0; k < iters && rc == DCREG_OK; ++k) rc = launch_body(ctx, L, prm, dlog, log_cap, true);
                e = cudaStreamEndCapture(ctx->stream, &graph);
            }
            ctx->nn_valid = nn_valid0; ctx->launches = launches0;      // nothing has run yet
            if (e == cudaSuccess && rc == DCREG_OK && graph) e = cudaGraphInstantiate(&exec, graph, 0);
            if (graph) cudaGraphDestroy(graph);
            if (e != cudaSuccess || rc != DCREG_OK || !exec) {
                cudaGetLastError();                                    // clear; run without a graph from now on
                exec = nullptr; ctx->graph_off = true;
            } else {
                if (ctx->graphs.size() >= 4) { cudaGraphExecDestroy(ctx->graphs.back().exec); ctx->graphs.pop_back(); }
                ctx->graphs.insert(ctx->graphs.begin(), dcreg_ctx::LoopGraph{key, exec});
            }
        }
        if (exec) {
            CK(cudaGraphLaunch(exec, ctx->stream));
            ctx->nn_valid = true;
            ctx->launches += (long long)iters * (L.fold_k2 ? 1 : 2); ctx->graph_launches++;
            return DCREG_OK;
        }
    }
    for (int k = 0; k < iters; ++k) {
        const int rc = launch_body(ctx, L, prm, dlog, log_cap, true);
        if (rc) return rc;
    }
    return DCREG_OK;
}

// The loop for `trials` registrations of the context's source (or of the scans of `scans`, one per trial) against its
// target, side by side.  fetch = false: enqueue only (no host synchronisation at all: no peek between chunks, no read-back)
static int run_loop(dcreg_ctx* ctx, const dcreg_icp_params* params, int trials, const double* T_init, double* T_out,
                    dcreg_iter_log* log, int log_cap, int* n_iterations, int* converged, int* status, bool fetch = true,
                    const ScanSet* scans = nullptr) {
    int rc;
    if (log && log_cap > 0 && (rc = ensure_log(ctx, (long long)trials * log_cap))) return rc;
    dcreg_iter_log* dlog = (log && log_cap > 0) ? ctx->d_log : nullptr;
    if (dlog) CK(cudaMemsetAsync(dlog, 0, (size_t)trials * log_cap * sizeof(dcreg_iter_log), ctx->stream));   // aborted iterations leave fields untouched
    if ((rc = init_state(ctx, T_init, trials, scans ? scans->off : nullptr))) return rc;
    const float4* src_iter = ctx->d_src;
    if (scans) rc = sort_scans_by_cell(ctx, *scans, &src_iter);
    else rc = sort_source_by_cell(ctx, T_init, &src_iter);                    // locality only: any pose of the batch will do
    if (rc) return rc;
    LoopPlan L;
    if ((rc = plan_iteration(ctx, params, src_iter, nullptr, trials, dlog, dlog ? log_cap : 0, true, &L, scans))) return rc;
    if ((rc = ensure_pinned(ctx, (size_t)trials * sizeof(IcpState)))) return rc;
    // fixed iteration count: the whole run is one chunk; otherwise chunks of 16 with a peek at the number of running
    // trials in between (the only host sync inside a run; iterations past convergence exit at once on the device)
    const int chunk = params->fixed_iterations ? (params->max_iterations < 64 ? params->max_iterations : 64) : 16;
    int issued = 0;
    while (issued < params->max_iterations) {
        int todo = params->max_iterations - issued;
        if (todo > chunk) todo = chunk;
        // a captured chunk is always `chunk` bodies long (one graph per run shape); bodies past max_iterations exit at once
        const int bodies = (todo < chunk && issued > 0) ? chunk : todo;
        if ((rc = enqueue_iterations(ctx, L, params, dlog, dlog ? log_cap : 0, bodies))) return rc;
        issued += bodies;
        if (fetch && issued < params->max_iterations && !params->fixed_iterations) {
            unsigned int* flag = (unsigned int*)ctx->h_pinned;       // trials still running (every solve step that finishes one decrements it)
            CK(cudaMemcpyAsync(flag, ctx->d_n_active, sizeof(unsigned int), cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            if (*flag == 0u) break;
        }
    }
    if (dlog) {
        log_fill_kernel<<<dim3((log_cap + 31) / 32, trials), 32, 0, ctx->stream>>>(dlog, log_cap, ctx->d_state, *params);
        ctx->launches++;
    }
    if (!fetch) return DCREG_OK;
    return read_results(ctx, trials, T_out, log, log_cap, n_iterations, converged, status);
}

static int check_target_and_params(dcreg_ctx* ctx, const dcreg_icp_params* params) {
    if (!ctx->has_grid) { ctx->err = "[ICP Error] Target index is not set up in context."; return DCREG_BAD_ARG; }
    if (params->max_iterations < 0) { ctx->err = "icp_run: max_iterations < 0"; return DCREG_BAD_ARG; }
    if (!(params->weight_slope > 0.0) || !(params->weight_gate >= 0.0) || !(params->weight_gate < 1.0)) {
        ctx->err = "icp_run: weight_slope must be > 0 and weight_gate in [0, 1)";
        return DCREG_BAD_ARG;
    }
    return DCREG_OK;
}

static int check_run_args(dcreg_ctx* ctx, const dcreg_icp_params* params) {
    if (!ctx->d_src || ctx->n_src <= 0) { ctx->err = "[ICP Error] Input measure cloud is null or empty."; return DCREG_BAD_ARG; }
    return check_target_and_params(ctx, params);
}

int dcreg_icp_run(dcreg_ctx* ctx, const dcreg_icp_params* params, const double T_init[16], double T_out[16],
                  dcreg_iter_log* log, int log_cap, int* n_iterations, int* converged) {
    if (!ctx) return DCREG_BAD_ARG;
    if (!params || !T_init || !T_out) { ctx->err = "icp_run: null pointer"; return DCREG_BAD_ARG; }
    int rc = check_run_args(ctx, params);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    int status = DCREG_OK;
    if ((rc = run_loop(ctx, params, 1, T_init, T_out, log, log_cap, n_iterations, converged, &status))) return rc;
    return status;
}

int dcreg_icp_enqueue(dcreg_ctx* ctx, const dcreg_icp_params* params, const double T_init[16]) {
    if (!ctx) return DCREG_BAD_ARG;
    if (!params || !T_init) { ctx->err = "icp_enqueue: null pointer"; return DCREG_BAD_ARG; }
    int rc = check_run_args(ctx, params);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    return run_loop(ctx, params, 1, T_init, nullptr, nullptr, 0, nullptr, nullptr, nullptr, false);
}

int dcreg_icp_fetch(dcreg_ctx* ctx, double T_out[16], int* n_iterations, int* converged) {
    if (!ctx) return DCREG_BAD_ARG;
    if (!T_out) { ctx->err = "icp_fetch: null pointer"; return DCREG_BAD_ARG; }
    CK(cudaSetDevice(ctx->device));
    int status = DCREG_OK;
    const int rc = read_results(ctx, 1, T_out, nullptr, 0, n_iterations, converged, &status);
    return rc ? rc : status;
}

int dcreg_icp_run_batch(dcreg_ctx* ctx, const dcreg_icp_params* params, int n_trials, const double* T_init,
                        double* T_out, int* n_iterations, int* converged, int* status, dcreg_iter_log* log, int log_cap) {
    if (!ctx) return DCREG_BAD_ARG;
    if (!params || !T_init || !T_out || n_trials <= 0) { ctx->err = "icp_run_batch: null pointer or n_trials <= 0"; return DCREG_BAD_ARG; }
    if (ctx->comm) { ctx->err = "icp_run_batch: trials are independent - distribute them over ranks, do not shard them"; return DCREG_BAD_ARG; }
    int rc = check_run_args(ctx, params);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    std::vector<int> st_local;
    if (!status) { st_local.resize(n_trials); status = st_local.data(); }
    return run_loop(ctx, params, n_trials, T_init, T_out, log, log_cap, n_iterations, converged, status);
}

int dcreg_icp_run_scans(dcreg_ctx* ctx, const dcreg_icp_params* params, int n_scans, const float* xyz, int stride,
                        const int64_t* scan_offsets, const double* T_init, double* T_out, int* n_iterations, int* converged,
                        int* status, dcreg_iter_log* log, int log_cap) {
    if (!ctx) return DCREG_BAD_ARG;
    if (!params || !xyz || !scan_offsets || !T_init || !T_out) { ctx->err = "icp_run_scans: null pointer"; return DCREG_BAD_ARG; }
    if (n_scans < 1 || n_scans > 65535) { ctx->err = "icp_run_scans: n_scans must be in [1, 65535]"; return DCREG_BAD_ARG; }
    if (stride < 3) { ctx->err = "icp_run_scans: stride < 3"; return DCREG_BAD_ARG; }
    if (scan_offsets[0] != 0) { ctx->err = "icp_run_scans: scan_offsets[0] must be 0"; return DCREG_BAD_ARG; }
    long long largest = 0;
    for (int s = 0; s < n_scans; ++s) {
        const long long ns = (long long)scan_offsets[s + 1] - (long long)scan_offsets[s];
        if (ns <= 0) {
            ctx->err = "icp_run_scans: scan " + std::to_string(s) + " is empty (scan_offsets must strictly increase)";
            return DCREG_BAD_ARG;
        }
        if (ns > largest) largest = ns;
    }
    const long long total = scan_offsets[n_scans];
    if (total > 0x1fffffffLL) { ctx->err = "icp_run_scans: more than 0x1fffffff points in all scans together"; return DCREG_BAD_ARG; }
    if (ctx->comm) { ctx->err = "icp_run_scans: scans are independent - distribute them over ranks, do not shard them"; return DCREG_BAD_ARG; }
    int rc = check_target_and_params(ctx, params);
    if (rc) return rc;
    if (!ctx->grid.dense) {
        ctx->err = "batched trials need the dense target grid (target bounding box / cell size too large for it)";
        return DCREG_BAD_ARG;
    }
    CK(cudaSetDevice(ctx->device));
    if ((rc = ensure_buffer(ctx, &ctx->d_scan, &ctx->scan_cap, total)) ||
        (rc = ensure_buffer(ctx, &ctx->d_scan_sorted, &ctx->scan_sorted_cap, total)) ||
        (rc = ensure_buffer(ctx, &ctx->d_scan_keys, &ctx->scan_keys_cap, 2 * total)) ||
        (rc = ensure_buffer(ctx, &ctx->d_scan_slots, &ctx->scan_slots_cap, 2 * total)) ||
        (rc = ensure_buffer(ctx, &ctx->d_scan_off, &ctx->scan_off_cap, (long long)n_scans + 1)) ||
        (rc = ensure_buffer(ctx, &ctx->d_scan_radius, &ctx->scan_radius_cap, (long long)n_scans)))
        return rc;
    CK(cudaMemcpyAsync(ctx->d_scan_off, scan_offsets, ((size_t)n_scans + 1) * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
    if ((rc = upload_points(ctx, xyz, total, stride, ctx->d_scan, ctx->d_scan_radius, ctx->d_scan_off, n_scans))) return rc;
    const ScanSet S{ctx->d_scan, ctx->d_scan_off, ctx->d_scan_radius, n_scans, total, largest};
    std::vector<int> st_local;
    if (!status) { st_local.resize(n_scans); status = st_local.data(); }
    return run_loop(ctx, params, n_scans, T_init, T_out, log, log_cap, n_iterations, converged, status, true, &S);
}

int dcreg_icp_run_host_planes(dcreg_ctx* ctx, const dcreg_icp_params* params, const double T_init[16],
                              dcreg_plane_callback cb, void* user, double T_out[16], dcreg_iter_log* log,
                              int log_cap, int* n_iterations, int* converged) {
    if (!ctx) return DCREG_BAD_ARG;
    if (!params || !T_init || !T_out || !cb) { ctx->err = "icp_run_host_planes: null pointer"; return DCREG_BAD_ARG; }
    if (!ctx->d_src || ctx->n_src <= 0) { ctx->err = "[ICP Error] Input measure cloud is null or empty."; return DCREG_BAD_ARG; }
    CK(cudaSetDevice(ctx->device));
    int rc;
    if (log && log_cap > 0 && (rc = ensure_log(ctx, log_cap))) return rc;
    dcreg_iter_log* dlog = (log && log_cap > 0) ? ctx->d_log : nullptr;
    if (dlog) CK(cudaMemsetAsync(dlog, 0, (size_t)log_cap * sizeof(dcreg_iter_log), ctx->stream));
    if ((rc = ensure_planes(ctx, ctx->n_src))) return rc;
    if ((rc = ensure_pinned(ctx, sizeof(IcpState) + (size_t)ctx->n_src * sizeof(double4)))) return rc;
    IcpState* hs = (IcpState*)ctx->h_pinned;
    double* hplanes = (double*)((char*)ctx->h_pinned + sizeof(IcpState));
    if ((rc = init_state(ctx, T_init))) return rc;
    double T[16];
    memcpy(T, T_init, sizeof(T));
    for (int it = 0; it < params->max_iterations; ++it) {
        int64_t npt = -1;
        if (cb(user, T, hplanes, &npt) != 0) { ctx->err = "plane callback failed"; return DCREG_BAD_ARG; }
        CK(cudaMemcpyAsync(ctx->d_planes64, hplanes, (size_t)ctx->n_src * sizeof(double4), cudaMemcpyHostToDevice,
                           ctx->stream));
        k1::Pose P;                                   // the host holds the current pose in this mode
        for (int r = 0; r < 3; ++r) {
            for (int c = 0; c < 3; ++c) P.R[r * 3 + c] = T[r * 4 + c];
            P.t[r] = T[r * 4 + 3];
        }
        // n_corr_pt is the caller's count (5th neighbour inside the radius, BEFORE the plane gates:
        // icp_test_runner.cpp:1726-1731, 1856), not the number of non-zero planes K1 sees
        if ((rc = launch_reduce(ctx, ctx->d_src, ctx->d_planes64, true, ctx->n_src, &P, params->use_weight_derivative,
                                params->weight_slope, params->weight_gate, npt >= 0 ? (double)npt : -1.0)))
            return rc;
        if ((rc = nccl_allreduce_acc(ctx))) return rc;
        if ((rc = launch_k2(ctx, params, dlog, log_cap))) return rc;
        CK(cudaMemcpyAsync(hs, ctx->d_state, sizeof(IcpState), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        for (int r = 0; r < 3; ++r) {
            for (int c = 0; c < 3; ++c) T[r * 4 + c] = hs->R[r * 3 + c];
            T[r * 4 + 3] = hs->t[r];
        }
        if (hs->done) break;
    }
    int status = DCREG_OK;
    if (dlog) {
        log_fill_kernel<<<dim3((log_cap + 31) / 32, 1), 32, 0, ctx->stream>>>(dlog, log_cap, ctx->d_state, *params);
        ctx->launches++;
    }
    if ((rc = read_results(ctx, 1, T_out, log, log_cap, n_iterations, converged, &status))) return rc;
    return status;
}

int dcreg_last_covariance(dcreg_ctx* ctx, double cov[36]) {
    if (!ctx || !cov) return DCREG_BAD_ARG;
    CK(cudaSetDevice(ctx->device));
    covariance_kernel<<<1, 32, 0, ctx->stream>>>(ctx->d_state, ctx->d_small + 256);
    ctx->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(cov, ctx->d_small + 256, 36 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return DCREG_OK;
}

int dcreg_last_covariances(dcreg_ctx* ctx, int n_trials, double* cov) {
    if (!ctx) return DCREG_BAD_ARG;
    if (!cov) { ctx->err = "last_covariances: null pointer"; return DCREG_BAD_ARG; }
    if (n_trials < 1 || n_trials > ctx->last_trials) {
        ctx->err = "last_covariances: n_trials must be in [1, " + std::to_string(ctx->last_trials) + "], the trial count of the last run";
        return DCREG_BAD_ARG;
    }
    CK(cudaSetDevice(ctx->device));
    if (ctx->cov_cap < n_trials) {
        if (ctx->d_cov) cudaFree(ctx->d_cov);
        ctx->d_cov = nullptr; ctx->cov_cap = 0;
        CK(cudaMalloc(&ctx->d_cov, (size_t)n_trials * 36 * sizeof(double)));
        ctx->cov_cap = n_trials;
    }
    covariance_kernel<<<n_trials, 32, 0, ctx->stream>>>(ctx->d_state, ctx->d_cov);
    ctx->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(cov, ctx->d_cov, (size_t)n_trials * 36 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return DCREG_OK;
}

int dcreg_comm_unique_id(dcreg_ctx* ctx, uint8_t id_out[128]) {
    if (!ctx || !id_out) return DCREG_BAD_ARG;
    if (!g_nccl.load(ctx->err)) return DCREG_NCCL_ERROR;
    ncclUniqueId id;
    int r = g_nccl.GetUniqueId(&id);
    if (r != 0) { ctx->err = "ncclGetUniqueId failed"; return DCREG_NCCL_ERROR; }
    memcpy(id_out, id.internal, 128);
    return DCREG_OK;
}

// Map every rank's mailbox into this process (cudaIpc handles carried by one ncclAllGather): afterwards the sum over
// ranks runs inside the reducing kernels (peer_reduce.cuh) and NCCL is not on the data path any more.  Any failure
// leaves peer_ok = false: the NCCL all-reduce fallback stays in place.
static void setup_peer_mailboxes(dcreg_ctx* ctx) {
    ctx->peer_ok = false;
    if (ctx->nranks < 2 || ctx->nranks > peer::kMaxRanks || !g_nccl.AllGather || getenv("DCREG_NO_PEER")) return;
    cudaIpcMemHandle_t mine;
    unsigned char* d_handles = nullptr;
    std::vector<cudaIpcMemHandle_t> all(ctx->nranks);
    bool ok = cudaMalloc(&ctx->d_mailbox, sizeof(peer::Mailbox)) == cudaSuccess &&
              cudaMemset(ctx->d_mailbox, 0, sizeof(peer::Mailbox)) == cudaSuccess &&
              cudaIpcGetMemHandle(&mine, ctx->d_mailbox) == cudaSuccess &&
              cudaMalloc(&d_handles, sizeof(mine) * ctx->nranks) == cudaSuccess;
    // every rank takes part in the collectives below even if its own setup failed (flag travels with the handle)
    unsigned char blob[sizeof(cudaIpcMemHandle_t)];
    memset(blob, 0, sizeof(blob));
    if (ok) memcpy(blob, &mine, sizeof(mine));
    unsigned char* d_mine = nullptr;
    if (cudaMalloc(&d_mine, sizeof(blob)) != cudaSuccess) { ok = false; }
    if (!d_handles || !d_mine) {          // cannot even run the collective coherently: give up on every rank the same way
        if (d_handles) cudaFree(d_handles);
        if (d_mine) cudaFree(d_mine);
        if (ctx->d_mailbox) { cudaFree(ctx->d_mailbox); ctx->d_mailbox = nullptr; }
        cudaGetLastError();
        return;
    }
    cudaMemcpyAsync(d_mine, blob, sizeof(blob), cudaMemcpyHostToDevice, ctx->stream);
    int r = g_nccl.AllGather(d_mine, d_handles, sizeof(blob), kNcclInt8, ctx->comm, ctx->stream);
    if (r == 0) {
        cudaMemcpyAsync(all.data(), d_handles, sizeof(mine) * ctx->nranks, cudaMemcpyDeviceToHost, ctx->stream);
        if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) r = 1;
    }
    if (r != 0) ok = false;
    peer::View v{};
    v.nranks = ctx->nranks; v.rank = ctx->rank;
    for (int q = 0; q < ctx->nranks && ok; ++q) {
        static const unsigned char zero[sizeof(cudaIpcMemHandle_t)] = {0};
        if (memcmp(&all[q], zero, sizeof(zero)) == 0) { ok = false; break; }      // that rank could not export
        if (q == ctx->rank) { v.box[q] = ctx->d_mailbox; continue; }
        void* ptr = nullptr;
        if (cudaIpcOpenMemHandle(&ptr, all[q], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { ok = false; break; }
        ctx->peer_ptr[q] = ptr;
        v.box[q] = (peer::Mailbox*)ptr;
    }
    // agree: peer mode only if EVERY rank mapped everything (one more tiny collective: min over ranks)
    double* d_flag = ctx->d_small + 700;
    const double flag = ok ? 1.0 : 0.0;
    cudaMemcpyAsync(d_flag, &flag, sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
    // sum of the flags == nranks  <=>  all ok
    double total = 0.0;
    if (g_nccl.AllReduce(d_flag, d_flag, 1, kNcclFloat64, kNcclSum, ctx->comm, ctx->stream) == 0) {
        cudaMemcpyAsync(&total, d_flag, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
        cudaStreamSynchronize(ctx->stream);
    }
    cudaFree(d_handles); cudaFree(d_mine);
    if (total > (double)ctx->nranks - 0.5) {
        ctx->peer_view = v;
        ctx->peer_ok = true;
    } else {
        for (int q = 0; q < peer::kMaxRanks; ++q)
            if (ctx->peer_ptr[q]) { cudaIpcCloseMemHandle(ctx->peer_ptr[q]); ctx->peer_ptr[q] = nullptr; }
        if (ctx->d_mailbox) { cudaFree(ctx->d_mailbox); ctx->d_mailbox = nullptr; }
        cudaGetLastError();
    }
}

int dcreg_comm_init(dcreg_ctx* ctx, const uint8_t nccl_unique_id[128], int rank, int nranks) {
    if (!ctx || !nccl_unique_id || nranks < 1 || rank < 0 || rank >= nranks) return DCREG_BAD_ARG;
    if (!g_nccl.load(ctx->err)) return DCREG_NCCL_ERROR;
    CK(cudaSetDevice(ctx->device));
    ncclUniqueId id;
    memcpy(id.internal, nccl_unique_id, 128);
    int r = g_nccl.CommInitRank(&ctx->comm, nranks, id, rank);
    if (r != 0) {
        ctx->comm = nullptr;
        ctx->err = std::string("ncclCommInitRank: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "error");
        return DCREG_NCCL_ERROR;
    }
    ctx->rank = rank; ctx->nranks = nranks;
    setup_peer_mailboxes(ctx);
    ctx->drop_graphs();
    return DCREG_OK;
}

int dcreg_comm_mode(const dcreg_ctx* ctx) {
    if (!ctx || !ctx->comm) return 0;
    return ctx->peer_ok ? 2 : 1;
}

int dcreg_comm_destroy(dcreg_ctx* ctx) {
    if (!ctx) return DCREG_BAD_ARG;
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (int q = 0; q < peer::kMaxRanks; ++q)
        if (ctx->peer_ptr[q]) { cudaIpcCloseMemHandle(ctx->peer_ptr[q]); ctx->peer_ptr[q] = nullptr; }
    if (ctx->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(ctx->comm);     // (a collective: peers are still alive here)
    if (ctx->d_mailbox) { cudaFree(ctx->d_mailbox); ctx->d_mailbox = nullptr; }
    ctx->peer_ok = false; ctx->peer_view = peer::View{};
    ctx->comm = nullptr; ctx->rank = 0; ctx->nranks = 1;
    ctx->drop_graphs();
    return DCREG_OK;
}

}  // extern "C"
