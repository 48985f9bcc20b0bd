// corr.cuh - device correspondence stage: uniform-grid exact 5-NN within radius + 5x3 plane fit.
//
// Replaces (reference file:line):
//   ICPContext::setTargetCloud kd-tree build           DCReg/include/utils.hpp:393-424
//   kdtree.nearestKSearch(q, 5) + 5th-NN radius gate   DCReg/src/icp_test_runner.cpp:1720-1726
//   5x3 colPivHouseholderQr plane fit + gates          icp_test_runner.cpp:1727-1773
//
// The reference's accept rule is "the 5th nearest neighbour is closer than the search radius".
// With cubic cells of edge = radius, every point closer than the radius to q lies in the 27 cells
// around q's cell, so an exact 5-NN over those cells reproduces the accept set of the kd-tree
// (SURVEY.md §7 step 6).  Distances are float32 sums of float32 squared differences, as in FLANN's
// L2_Simple functor that PCL's KdTreeFLANN uses; ties are broken by original point index.
//
// Layout in HBM: target points grouped by cell (float4: x, y, z, bit-cast original index).
//   dense mode : cells of the target's bounding box in x-fastest linear order + cell_start[ncells + 1];
//                the 3 x-adjacent cells of a row are ONE contiguous point range, so a query scans 9 ranges.
//   hash mode  : open-addressing table keyed by the packed cell coordinates (fallback when the bounding box
//                has more than kMaxDenseCells cells); a query probes 27 cells.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "small_la.cuh"

namespace corr {

constexpr unsigned long long kEmptyKey = ~0ull;
constexpr long long kMaxDenseCells = 1ll << 27;

struct Grid {
    float4* pts;                // n target points grouped by cell
    int* pos_of;                // [n] position in pts of the point with original index i (inverse of pts[j].w)
    int n;
    int dense;                  // 1: dense mode, 0: hash mode
    int rings;                  // ceil(search radius / cell edge): cells per direction a query must look at
    double inv_cell;            // 1 / cell edge
    // dense mode
    int ox, oy, oz;             // cell coordinates of the bounding box's minimum corner
    int nx, ny, nz;
    int* cell_start;            // [nx*ny*nz + 1]
    // hash mode
    unsigned long long* keys;   // capacity entries, kEmptyKey = free
    int* hstart;                // capacity
    int* hcount;                // capacity
    unsigned int mask;          // capacity - 1 (capacity is a power of two)
};

__host__ __device__ __forceinline__ int cell_coord(float v, double inv_cell) {
    return (int)floor((double)v * inv_cell);
}

__host__ __device__ __forceinline__ unsigned long long pack_key(int ix, int iy, int iz) {
    const long long B = 1ll << 20;
    return ((unsigned long long)(ix + B) << 42) | ((unsigned long long)(iy + B) << 21) | (unsigned long long)(iz + B);
}

__host__ __device__ __forceinline__ unsigned int hash_key(unsigned long long k) {
    k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
    return (unsigned int)k;
}

__device__ __forceinline__ int dense_index(const Grid& g, int cx, int cy, int cz) {
    return ((cz - g.oz) * g.ny + (cy - g.oy)) * g.nx + (cx - g.ox);
}

// ---- build -----------------------------------------------------------------------------------
// bounds[0..2] = min cell coords, bounds[3..5] = max cell coords (initialised to +-2^30 by the host)
__global__ void grid_bounds_kernel(const float4* __restrict__ pts, int n, double inv_cell, int* __restrict__ bounds) {
    int lo[3] = {1 << 30, 1 << 30, 1 << 30}, hi[3] = {-(1 << 30), -(1 << 30), -(1 << 30)};
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float4 p = pts[i];
        const int c[3] = {cell_coord(p.x, inv_cell), cell_coord(p.y, inv_cell), cell_coord(p.z, inv_cell)};
        for (int k = 0; k < 3; ++k) { lo[k] = min(lo[k], c[k]); hi[k] = max(hi[k], c[k]); }
    }
    for (int k = 0; k < 3; ++k) {
        for (int off = 16; off > 0; off >>= 1) {
            lo[k] = min(lo[k], __shfl_xor_sync(0xffffffffu, lo[k], off));
            hi[k] = max(hi[k], __shfl_xor_sync(0xffffffffu, hi[k], off));
        }
        if ((threadIdx.x & 31) == 0) { atomicMin(&bounds[k], lo[k]); atomicMax(&bounds[3 + k], hi[k]); }
    }
}

// cell id of a point: dense linear index (clamped into the box when `clamp`), or hash slot (insert mode)
__global__ void grid_count_dense_kernel(const float4* __restrict__ pts, int n, Grid g, int* __restrict__ pt_cell,
                                        int* __restrict__ counts) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 p = pts[i];
    const int c = dense_index(g, cell_coord(p.x, g.inv_cell), cell_coord(p.y, g.inv_cell), cell_coord(p.z, g.inv_cell));
    pt_cell[i] = c;
    atomicAdd(&counts[c], 1);
}

__global__ void grid_insert_hash_kernel(const float4* __restrict__ pts, int n, Grid g, int* __restrict__ pt_slot) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 p = pts[i];
    const unsigned long long key = pack_key(cell_coord(p.x, g.inv_cell), cell_coord(p.y, g.inv_cell),
                                            cell_coord(p.z, g.inv_cell));
    unsigned int slot = hash_key(key) & g.mask;
    while (true) {
        const unsigned long long prev = atomicCAS(&g.keys[slot], kEmptyKey, key);
        if (prev == kEmptyKey || prev == key) break;
        slot = (slot + 1) & g.mask;
    }
    pt_slot[i] = (int)slot;
    atomicAdd(&g.hcount[slot], 1);
}

// exclusive scan of an int array, three phases (tile sums, scan of tile sums, tile rescan)
constexpr int kScanTile = 2048;   // 256 threads x 8
__global__ void scan_tile_sums_kernel(const int* __restrict__ in, int n, int* __restrict__ tile_sums) {
    __shared__ int sh[256];
    const long long base = (long long)blockIdx.x * kScanTile;
    int s = 0;
    for (int k = 0; k < 8; ++k) {
        const long long idx = base + threadIdx.x * 8 + k;
        if (idx < n) s += in[idx];
    }
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int off = 128; off > 0; off >>= 1) {
        if (threadIdx.x < off) sh[threadIdx.x] += sh[threadIdx.x + off];
        __syncthreads();
    }
    if (threadIdx.x == 0) tile_sums[blockIdx.x] = sh[0];
}
__global__ void scan_tile_offsets_kernel(int* tile_sums, int ntiles) {   // single block, 1024 threads
    __shared__ int sh[1024];
    __shared__ int carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < ntiles; base += 1024) {
        const int idx = base + threadIdx.x;
        const int v = idx < ntiles ? tile_sums[idx] : 0;
        sh[threadIdx.x] = v;
        __syncthreads();
        for (int off = 1; off < 1024; off <<= 1) {
            const int t = threadIdx.x >= off ? sh[threadIdx.x - off] : 0;
            __syncthreads();
            sh[threadIdx.x] += t;
            __syncthreads();
        }
        if (idx < ntiles) tile_sums[idx] = carry + sh[threadIdx.x] - v;   // exclusive
        __syncthreads();
        if (threadIdx.x == 1023) carry += sh[1023];
        __syncthreads();
    }
}
__global__ void scan_tile_apply_kernel(const int* __restrict__ in, int n, const int* __restrict__ tile_offsets,
                                       int* __restrict__ out) {
    __shared__ int sh[256];
    const long long base = (long long)blockIdx.x * kScanTile;
    int loc[8];
    int s = 0;
    for (int k = 0; k < 8; ++k) {
        const long long idx = base + threadIdx.x * 8 + k;
        loc[k] = idx < n ? in[idx] : 0;
        s += loc[k];
    }
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int off = 1; off < 256; off <<= 1) {
        const int t = threadIdx.x >= off ? sh[threadIdx.x - off] : 0;
        __syncthreads();
        sh[threadIdx.x] += t;
        __syncthreads();
    }
    int run = tile_offsets[blockIdx.x] + sh[threadIdx.x] - s;
    for (int k = 0; k < 8; ++k) {
        const long long idx = base + threadIdx.x * 8 + k;
        if (idx < n) out[idx] = run;
        run += loc[k];
    }
}

// scatter points into their cell's range; `start` is the exclusive scan of the per-cell counts
__global__ void grid_scatter_kernel(const float4* __restrict__ pts, int n, const int* __restrict__ pt_cell,
                                    const int* __restrict__ start, int* __restrict__ fill, float4* __restrict__ out,
                                    int keep_w) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int c = pt_cell[i];
    const int pos = start[c] + atomicAdd(&fill[c], 1);
    float4 p = pts[i];
    if (!keep_w) p.w = __int_as_float(i);
    out[pos] = p;
}

// Deterministic order inside every cell: ascending original index.  The scatter above fills a cell in atomic-arrival
// order; this pass moves every point to (cell start + number of points of its cell with a smaller index).  One thread
// per point, O(points in its cell) reads of a range its neighbours read too - parallel over POINTS, so a cell with
// thousands of points (dense map, cell = search radius) no longer serialises on one thread the way a per-cell insertion
// sort does.  `cell_of` is indexed by the original point index (p.w): dense cell id or hash slot.
__global__ void grid_rank_cells_kernel(const float4* __restrict__ in, int n, const int* __restrict__ cell_of,
                                       const int* __restrict__ start, const int* __restrict__ count,
                                       float4* __restrict__ out, int* __restrict__ pos_of) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const float4 p = in[j];
    const int me = __float_as_int(p.w);
    const int c = cell_of[me];
    const int s = start[c];
    const int e = count ? s + count[c] : start[c + 1];
    int rank = 0;
    for (int k = s; k < e; ++k) rank += (__float_as_int(__ldg(&in[k].w)) < me) ? 1 : 0;
    out[s + rank] = p;
    if (pos_of) pos_of[me] = s + rank;
}

// dense cell of T*p (T: row-major 4x4, first three rows read), clamped into the target box
__device__ __forceinline__ int source_cell(const float4 p, const Grid& g, const double* __restrict__ T) {
    const double px = p.x, py = p.y, pz = p.z;
    const float qx = (float)(T[0] * px + T[1] * py + T[2] * pz + T[3]);
    const float qy = (float)(T[4] * px + T[5] * py + T[6] * pz + T[7]);
    const float qz = (float)(T[8] * px + T[9] * py + T[10] * pz + T[11]);
    const int cx = min(max(cell_coord(qx, g.inv_cell) - g.ox, 0), g.nx - 1);
    const int cy = min(max(cell_coord(qy, g.inv_cell) - g.oy, 0), g.ny - 1);
    const int cz = min(max(cell_coord(qz, g.inv_cell) - g.oz, 0), g.nz - 1);
    return (cz * g.ny + cy) * g.nx + cx;
}

// cell of a (transformed) source point for the spatial sort of the source cloud
__global__ void source_cell_kernel(const float4* __restrict__ src, int n, Grid g, const double* __restrict__ T,
                                   int* __restrict__ pt_cell, int* __restrict__ counts) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int c = source_cell(src[i], g, T);
    pt_cell[i] = c;
    atomicAdd(&counts[c], 1);
}

// Scan s of a scan set = slots [off[s], off[s+1]) (off strictly increasing, off[0] = 0): the s with off[s] <= i < off[s+1].
__device__ __forceinline__ int scan_of(const long long* __restrict__ off, int n_scans, long long i) {
    int lo = 0, hi = n_scans - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(&off[mid]) <= i) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// Sort keys of a scan set: (scan << 32) | target cell of T_s * p with T = [n_scans][16]; value = slot.  A stable radix sort
// on these keys keeps every scan contiguous and, inside a cell, the input order - for one scan exactly the order of the
// counting sort above (source_cell_kernel + grid_scatter_kernel + grid_rank_cells_kernel).
__global__ void scan_cell_keys_kernel(const float4* __restrict__ src, int n, const long long* __restrict__ off, int n_scans,
                                      Grid g, const double* __restrict__ T, unsigned long long* __restrict__ keys,
                                      int* __restrict__ slots) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int s = scan_of(off, n_scans, i);
    keys[i] = ((unsigned long long)s << 32) | (unsigned)source_cell(src[i], g, T + (size_t)s * 16);
    slots[i] = i;
}

// sorted[j] = src[slot[j]] (w keeps the point's slot in the unsorted buffer)
__global__ void gather_points_kernel(const float4* __restrict__ src, int n, const int* __restrict__ slot, float4* __restrict__ out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) out[j] = src[slot[j]];
}

// ---- query -----------------------------------------------------------------------------------
// The five best so far, ascending.  key = (bits of the squared distance) << 32 | original index: squared distances are
// non-negative floats, whose bit patterns order like unsigned integers, so ONE 64-bit unsigned compare is the (distance,
// then index) rule of the reference's tie handling - two instructions instead of four per compare in the insertion that
// dominates the per-thread search (ncu, lean iterations: 30 % of all warp instructions on that compare).
// The list carries no positions: a neighbour's position in g.pts is looked up from its index once, when the search is
// over (Grid::pos_of) - one register and two moves per insertion step less.
struct Knn5 {
    unsigned long long key[5];
};

__device__ __forceinline__ unsigned long long knn_key(float d2, int idx) {
    return ((unsigned long long)__float_as_uint(d2) << 32) | (unsigned long long)(unsigned)idx;
}
__device__ __forceinline__ float knn_d2(const Knn5& k, int i) { return __uint_as_float((unsigned)(k.key[i] >> 32)); }
// positions of the five (-1 where the list still holds a sentinel): five independent loads, one round trip
__device__ __forceinline__ void knn_positions(const Grid& g, const Knn5& k, int (&pos)[5]) {
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        const int idx = (int)(unsigned)(k.key[i] & 0xffffffffull);
        pos[i] = idx == 0x7fffffff ? -1 : __ldg(&g.pos_of[idx]);
    }
}

__device__ __forceinline__ void knn_init(Knn5& k) {
#pragma unroll
    for (int i = 0; i < 5; ++i) k.key[i] = knn_key(3.0e38f, 0x7fffffff);
}

__device__ __forceinline__ void knn_insert(Knn5& k, unsigned long long key) {
    k.key[4] = key;
#pragma unroll
    for (int i = 4; i > 0; --i) {
        if (k.key[i] < k.key[i - 1]) { const unsigned long long tk = k.key[i]; k.key[i] = k.key[i - 1]; k.key[i - 1] = tk; }
    }
}

// FLANN L2_Simple: float differences, float accumulation, x then y then z (no FMA contraction)
__device__ __forceinline__ float dist2(float qx, float qy, float qz, const float4& p) {
    const float ex = __fsub_rn(qx, p.x), ey = __fsub_rn(qy, p.y), ez = __fsub_rn(qz, p.z);
    return __fadd_rn(__fadd_rn(__fmul_rn(ex, ex), __fmul_rn(ey, ey)), __fmul_rn(ez, ez));
}

__device__ __forceinline__ void knn_scan_range(const float4* __restrict__ pts, int s, int e, float qx, float qy,
                                               float qz, Knn5& k) {
    int j = s;
#pragma unroll 1
    for (; j + 3 < e; j += 4) {                       // four candidates per trip: four loads in flight (the scan is one
        const float4 p0 = __ldg(&pts[j]), p1 = __ldg(&pts[j + 1]), p2 = __ldg(&pts[j + 2]), p3 = __ldg(&pts[j + 3]);   // thread's latency chain)
        const unsigned long long k0 = knn_key(dist2(qx, qy, qz, p0), __float_as_int(p0.w)), k1 = knn_key(dist2(qx, qy, qz, p1), __float_as_int(p1.w));
        const unsigned long long k2 = knn_key(dist2(qx, qy, qz, p2), __float_as_int(p2.w)), k3 = knn_key(dist2(qx, qy, qz, p3), __float_as_int(p3.w));
        if (k0 < k.key[4]) knn_insert(k, k0);
        if (k1 < k.key[4]) knn_insert(k, k1);
        if (k2 < k.key[4]) knn_insert(k, k2);
        if (k3 < k.key[4]) knn_insert(k, k3);
    }
#pragma unroll 1
    for (; j < e; ++j) {
        const float4 p0 = __ldg(&pts[j]);
        const unsigned long long k0 = knn_key(dist2(qx, qy, qz, p0), __float_as_int(p0.w));
        if (k0 < k.key[4]) knn_insert(k, k0);
    }
}

__device__ __forceinline__ void knn_search(const Grid& g, float qx, float qy, float qz, Knn5& k) {
    const int cx = cell_coord(qx, g.inv_cell), cy = cell_coord(qy, g.inv_cell), cz = cell_coord(qz, g.inv_cell);
    if (g.dense) {
        // K = ceil(radius / cell) rings of cells cover the search radius (K = 1 when cell = radius; a finer grid,
        // cell = radius / 2, K = 2, scans ~3x fewer candidates because most cells are pruned by their box distance).
        // Rows (dy, dz) are visited in rings of growing max(|dy|, |dz|); inside a row the own column first, then
        // outwards.  A row / cell is skipped only when its box distance exceeds the current 5th-best distance
        // (strictly, with a 1e-5 relative margin for the float arithmetic of the bound), so the search stays exact.
        // Loops are deliberately NOT unrolled: one copy of the scan loop keeps the kernel inside the instruction
        // cache (the fully unrolled version stalled on instruction fetch, profiles/icp_iteration_r1).
        const int K = g.rings;
        const float cell = (float)(1.0 / g.inv_cell);
        const int lx = cx - g.ox, ly = cy - g.oy, lz = cz - g.oz;
        if (lx + K < 0 || lx - K >= g.nx) return;
        // position inside the own cell, in [0, cell) up to float rounding of cx * cell: every gap below is shrunk
        // by an absolute eps that covers that rounding, so a bound can only be too small (never prunes a hit)
        const float eps = 2e-6f * (fabsf(qx) + fabsf(qy) + fabsf(qz) + cell);
        const float fx = qx - (float)cx * cell, fy = qy - (float)cy * cell, fz = qz - (float)cz * cell;
        if (K == 1) {
            // cell = search radius (the usual set-up): 9 rows of 3 cells.  Same rows, same pruning tests and the same
            // own / left / right order as the general loop below, but a row's FOUR cell boundaries are fetched together
            // (one memory round trip per visited row instead of up to six dependent ones: the lanes of a warp prune
            // differently, so a warp walks nearly all 27 cells and every dependent load is on its critical path).
            const float gl = fmaxf(fx - eps, 0.0f), gr = fmaxf((cell - fx) - eps, 0.0f);
            const float gl2 = gl * gl * 0.99999f, gr2 = gr * gr * 0.99999f;
            const int xa = min(max(lx - 1, 0), g.nx), xb = min(max(lx, 0), g.nx), xc = min(max(lx + 1, 0), g.nx), xd = min(max(lx + 2, 0), g.nx);
#pragma unroll 1
            for (int r = 0; r < 9; ++r) {
                // own row first, then the ring: (dz, dy) = (-1,-1) (-1,0) (-1,1) (0,-1) (0,1) (1,-1) (1,0) (1,1)
                const int q = r == 0 ? 4 : (r <= 4 ? r - 1 : r);
                const int dz = q / 3 - 1, dy = q % 3 - 1;
                const int zz = lz + dz, yy = ly + dy;
                if (zz < 0 || zz >= g.nz || yy < 0 || yy >= g.ny) continue;
                const float gz = dz == 0 ? 0.0f : fmaxf((dz < 0 ? fz : cell - fz) - eps, 0.0f);
                const float gy = dy == 0 ? 0.0f : fmaxf((dy < 0 ? fy : cell - fy) - eps, 0.0f);
                const float row_lb = (gy * gy + gz * gz) * 0.99999f;
                if (row_lb > knn_d2(k, 4)) continue;
                const int* rowp = g.cell_start + (size_t)(zz * g.ny + yy) * g.nx;
                const int b0 = __ldg(rowp + xa), b1 = __ldg(rowp + xb), b2 = __ldg(rowp + xc), b3 = __ldg(rowp + xd);
                knn_scan_range(g.pts, b1, b2, qx, qy, qz, k);
                if (row_lb + gl2 <= knn_d2(k, 4)) knn_scan_range(g.pts, b0, b1, qx, qy, qz, k);
                if (row_lb + gr2 <= knn_d2(k, 4)) knn_scan_range(g.pts, b2, b3, qx, qy, qz, k);
            }
            return;
        }
#pragma unroll 1
        for (int ring = 0; ring <= K; ++ring) {
            // a whole ring is at least (ring - 1) * cell + (distance to the own cell's nearest face) away
            if (ring > 1) {
                const float m = fmaxf(fminf(fminf(fy, cell - fy), fminf(fz, cell - fz)) + (float)(ring - 1) * cell - eps, 0.0f);
                if (m * m * 0.99999f > knn_d2(k, 4)) break;
            }
#pragma unroll 1
            for (int dz = -ring; dz <= ring; ++dz) {
                const int zz = lz + dz;
                if (zz < 0 || zz >= g.nz) continue;
                const float gz = dz == 0 ? 0.0f : fmaxf((dz < 0 ? fz + (float)(-dz - 1) * cell : (cell - fz) + (float)(dz - 1) * cell) - eps, 0.0f);
                const int stepy = (dz == -ring || dz == ring) ? 1 : 2 * ring;     // only the ring's boundary rows
#pragma unroll 1
                for (int dy = -ring; dy <= ring; dy += (stepy > 0 ? stepy : 1)) {
                    const int yy = ly + dy;
                    if (yy < 0 || yy >= g.ny) continue;
                    const float gy = dy == 0 ? 0.0f : fmaxf((dy < 0 ? fy + (float)(-dy - 1) * cell : (cell - fy) + (float)(dy - 1) * cell) - eps, 0.0f);
                    const float row_lb = (gy * gy + gz * gz) * 0.99999f;
                    if (row_lb > knn_d2(k, 4)) continue;
                    const int* rowp = g.cell_start + (size_t)(zz * g.ny + yy) * g.nx;
                    // own column, then +-1, +-2, ... : stop a side once its gap bound exceeds the 5th-best distance
                    {
                        const int x0 = min(max(lx, 0), g.nx), x1 = min(max(lx + 1, 0), g.nx);
                        knn_scan_range(g.pts, __ldg(rowp + x0), __ldg(rowp + x1), qx, qy, qz, k);
                    }
#pragma unroll 1
                    for (int dx = 1; dx <= K; ++dx) {
                        const float gl = fmaxf(fx + (float)(dx - 1) * cell - eps, 0.0f);
                        const float gr = fmaxf((cell - fx) + (float)(dx - 1) * cell - eps, 0.0f);
                        const bool left = (row_lb + gl * gl * 0.99999f) <= knn_d2(k, 4);
                        if (left) {
                            const int x0 = min(max(lx - dx, 0), g.nx), x1 = min(max(lx - dx + 1, 0), g.nx);
                            knn_scan_range(g.pts, __ldg(rowp + x0), __ldg(rowp + x1), qx, qy, qz, k);
                        }
                        const bool right = (row_lb + gr * gr * 0.99999f) <= knn_d2(k, 4);
                        if (right) {
                            const int x0 = min(max(lx + dx, 0), g.nx), x1 = min(max(lx + dx + 1, 0), g.nx);
                            knn_scan_range(g.pts, __ldg(rowp + x0), __ldg(rowp + x1), qx, qy, qz, k);
                        }
                        if (!left && !right) break;
                    }
                }
            }
        }
    } else {
        const int K = g.rings;
        for (int dz = -K; dz <= K; ++dz)
            for (int dy = -K; dy <= K; ++dy)
                for (int dx = -K; dx <= K; ++dx) {
                    const unsigned long long key = pack_key(cx + dx, cy + dy, cz + dz);
                    unsigned int slot = hash_key(key) & g.mask;
                    int start = 0, cnt = 0;
                    while (true) {
                        const unsigned long long kk = __ldg(&g.keys[slot]);
                        if (kk == key) { start = __ldg(&g.hstart[slot]); cnt = __ldg(&g.hcount[slot]); break; }
                        if (kk == kEmptyKey) break;
                        slot = (slot + 1) & g.mask;
                    }
                    knn_scan_range(g.pts, start, start + cnt, qx, qy, qz, k);
                }
    }
}

// ---- bounded exact M-NN with a gap certificate (dense grid, one thread per query) ----------------------------------
// Same traversal as knn_search, three differences:
//   * it keeps the kSeeds (7) nearest, not 5: the first five are the answer, the extra two widen the certificate below;
//   * the list starts as sentinels at the caller's bound B (any value >= the true 7th squared distance keeps the
//     search exact: a candidate with d2 == B and a real index still beats a sentinel), so rows / cells / candidates
//     beyond B are never touched;
//   * lb collects a lower bound on the squared distance of every target point that does NOT end up in the list:
//     the d2 of every rejected or evicted candidate and the box distance of everything pruned.  The caller uses it
//     to prove, in later iterations, that the seven still contain the five nearest without searching
//     (icp_iter2_kernel).
constexpr int kSeeds = 7;

struct KnnM {                 // as Knn5: key = (bits of the squared distance) << 32 | original index, ascending
    unsigned long long key[kSeeds];
    int pos[kSeeds];
};
__device__ __forceinline__ float knn_d2(const KnnM& k, int i) { return __uint_as_float((unsigned)(k.key[i] >> 32)); }

__device__ __forceinline__ void knnm_insert(KnnM& k, unsigned long long key, int pos) {
    k.key[kSeeds - 1] = key; k.pos[kSeeds - 1] = pos;
#pragma unroll
    for (int i = kSeeds - 1; i > 0; --i) {
        if (k.key[i] < k.key[i - 1]) {
            const unsigned long long tk = k.key[i]; k.key[i] = k.key[i - 1]; k.key[i - 1] = tk;
            const int tp = k.pos[i]; k.pos[i] = k.pos[i - 1]; k.pos[i - 1] = tp;
        }
    }
}

__device__ __forceinline__ void knn_scan_range_lb(const float4* __restrict__ pts, int s, int e, float qx, float qy,
                                                  float qz, KnnM& k, float& lb) {
    constexpr int L = kSeeds - 1;
    int j = s;
#pragma unroll 1
    for (; j + 1 < e; j += 2) {                       // two candidates per trip: both loads in flight
        const float4 p0 = __ldg(&pts[j]), p1 = __ldg(&pts[j + 1]);
        const float a0 = dist2(qx, qy, qz, p0), a1 = dist2(qx, qy, qz, p1);
        const unsigned long long k0 = knn_key(a0, __float_as_int(p0.w)), k1 = knn_key(a1, __float_as_int(p1.w));
        if (k0 < k.key[L]) { lb = fminf(lb, knn_d2(k, L)); knnm_insert(k, k0, j); }
        else lb = fminf(lb, a0);                      // rejected candidates and evicted entries bound the outside
        if (k1 < k.key[L]) { lb = fminf(lb, knn_d2(k, L)); knnm_insert(k, k1, j + 1); }
        else lb = fminf(lb, a1);
    }
    if (j < e) {
        const float4 p0 = __ldg(&pts[j]);
        const float a0 = dist2(qx, qy, qz, p0);
        const unsigned long long k0 = knn_key(a0, __float_as_int(p0.w));
        if (k0 < k.key[L]) { lb = fminf(lb, knn_d2(k, L)); knnm_insert(k, k0, j); }
        else lb = fminf(lb, a0);
    }
}

__device__ __forceinline__ void knn_search_lb(const Grid& g, float qx, float qy, float qz, float B, KnnM& k, float& lb) {
    constexpr int L = kSeeds - 1;
#pragma unroll
    for (int i = 0; i < kSeeds; ++i) { k.key[i] = knn_key(B, 0x7fffffff); k.pos[i] = -1; }
    const int cx = cell_coord(qx, g.inv_cell), cy = cell_coord(qy, g.inv_cell), cz = cell_coord(qz, g.inv_cell);
    const int K = g.rings;
    const float cell = (float)(1.0 / g.inv_cell);
    const int lx = cx - g.ox, ly = cy - g.oy, lz = cz - g.oz;
    if (lx + K < 0 || lx - K >= g.nx) return;
    const float eps = 2e-6f * (fabsf(qx) + fabsf(qy) + fabsf(qz) + cell);
    const float fx = qx - (float)cx * cell, fy = qy - (float)cy * cell, fz = qz - (float)cz * cell;
#pragma unroll 1
    for (int ring = 0; ring <= K; ++ring) {
        if (ring > 1) {
            const float m = fmaxf(fminf(fminf(fy, cell - fy), fminf(fz, cell - fz)) + (float)(ring - 1) * cell - eps, 0.0f);
            if (m * m * 0.99999f > knn_d2(k, L)) { lb = fminf(lb, m * m * 0.99999f); break; }
        }
#pragma unroll 1
        for (int dz = -ring; dz <= ring; ++dz) {
            const int zz = lz + dz;
            if (zz < 0 || zz >= g.nz) continue;
            const float gz = dz == 0 ? 0.0f : fmaxf((dz < 0 ? fz + (float)(-dz - 1) * cell : (cell - fz) + (float)(dz - 1) * cell) - eps, 0.0f);
            const int stepy = (dz == -ring || dz == ring) ? 1 : 2 * ring;     // only the ring's boundary rows
#pragma unroll 1
            for (int dy = -ring; dy <= ring; dy += (stepy > 0 ? stepy : 1)) {
                const int yy = ly + dy;
                if (yy < 0 || yy >= g.ny) continue;
                const float gy = dy == 0 ? 0.0f : fmaxf((dy < 0 ? fy + (float)(-dy - 1) * cell : (cell - fy) + (float)(dy - 1) * cell) - eps, 0.0f);
                const float row_lb = (gy * gy + gz * gz) * 0.99999f;
                if (row_lb > knn_d2(k, L)) { lb = fminf(lb, row_lb); continue; }
                const int* rowp = g.cell_start + (size_t)(zz * g.ny + yy) * g.nx;
                {
                    const int x0 = min(max(lx, 0), g.nx), x1 = min(max(lx + 1, 0), g.nx);
                    knn_scan_range_lb(g.pts, __ldg(rowp + x0), __ldg(rowp + x1), qx, qy, qz, k, lb);
                }
                bool left = true, right = true;
#pragma unroll 1
                for (int dx = 1; dx <= K; ++dx) {
                    if (left) {
                        const float gl = fmaxf(fx + (float)(dx - 1) * cell - eps, 0.0f);
                        const float b = row_lb + gl * gl * 0.99999f;
                        if (b <= knn_d2(k, L)) {
                            const int x0 = min(max(lx - dx, 0), g.nx), x1 = min(max(lx - dx + 1, 0), g.nx);
                            knn_scan_range_lb(g.pts, __ldg(rowp + x0), __ldg(rowp + x1), qx, qy, qz, k, lb);
                        } else { lb = fminf(lb, b); left = false; }
                    }
                    if (right) {
                        const float gr = fmaxf((cell - fx) + (float)(dx - 1) * cell - eps, 0.0f);
                        const float b = row_lb + gr * gr * 0.99999f;
                        if (b <= knn_d2(k, L)) {
                            const int x0 = min(max(lx + dx, 0), g.nx), x1 = min(max(lx + dx + 1, 0), g.nx);
                            knn_scan_range_lb(g.pts, __ldg(rowp + x0), __ldg(rowp + x1), qx, qy, qz, k, lb);
                        } else { lb = fminf(lb, b); right = false; }
                    }
                    if (!left && !right) break;
                }
            }
        }
    }
}


// ---- one query, one warp (dense grid) -----------------------------------------------------------------------------
// Same contract as knn_search_lb, executed by all 32 lanes for ONE query: used when only a few slots of a warp need a
// search, where the sequential search of one lane would keep the other 31 waiting for ~15 us.  Lanes set up the cell
// rows in parallel, walk every row with stride 32 (coalesced), compact the candidates with d2 <= B into a 64-entry
// shared buffer and rank them ((d2, index) order): ranks 0..6 are the list, everything else feeds lb.
// Returns false (nothing usable) when more than 64 candidates survive the bound; the caller then searches sequentially.
constexpr int kWarpKnnCap = 64;

struct WarpKnnSmem {
    int rs[81], re[81];                              // point range per cell row (empty when pruned)
    int pref[82];                                    // exclusive prefix sums of the row lengths (+ total)
    unsigned long long key[kWarpKnnCap];             // candidates inside the bound: knn_key(d2, index), ...
    int pos[kWarpKnnCap];                            // ... and their position
    unsigned long long okey[kSeeds];                 // the list, ascending
    int opos[kSeeds];
};

// One row (r of (2K+1)^2, x-fastest over (dy, dz)) of a bounded query's set-up: the point range of the row's cells that can
// hold something within the squared bound B, and `lb`, a lower bound on the squared distance of everything it dropped
// (3e38: dropped nothing).  A tile's searches have their rows set up by ALL its threads at once before the warps start
// (icp_iter2_kernel): one memory round trip for the whole tile instead of one at the head of every search.
struct RowRange { int s, e; float lb; };

__device__ __forceinline__ RowRange knn_row_range(const Grid& g, float qx, float qy, float qz, float B, int r) {
    const int K = g.rings, W = 2 * K + 1;
    const float cell = (float)(1.0 / g.inv_cell);
    const int cx = cell_coord(qx, g.inv_cell), cy = cell_coord(qy, g.inv_cell), cz = cell_coord(qz, g.inv_cell);
    const int lx = cx - g.ox, ly = cy - g.oy, lz = cz - g.oz;
    const float eps = 2e-6f * (fabsf(qx) + fabsf(qy) + fabsf(qz) + cell);
    const float fx = qx - (float)cx * cell, fy = qy - (float)cy * cell, fz = qz - (float)cz * cell;
    RowRange out{0, 0, 3.0e38f};
    const int rz = r / W;
    const int dz = rz - K, dy = r - rz * W - K;
    const int zz = lz + dz, yy = ly + dy;
    if (zz >= 0 && zz < g.nz && yy >= 0 && yy < g.ny) {
        const float gz = dz == 0 ? 0.0f : fmaxf((dz < 0 ? fz + (float)(-dz - 1) * cell : (cell - fz) + (float)(dz - 1) * cell) - eps, 0.0f);
        const float gy = dy == 0 ? 0.0f : fmaxf((dy < 0 ? fy + (float)(-dy - 1) * cell : (cell - fy) + (float)(dy - 1) * cell) - eps, 0.0f);
        const float row_lb = (gy * gy + gz * gz) * 0.99999f;
        if (row_lb <= B) {
            int xa = lx - K, xb = lx + K;                  // drop end cells whose box distance exceeds the bound
#pragma unroll 1
            for (; xa < lx; ++xa) {
                const float gl = fmaxf(fx + (float)(lx - xa - 1) * cell - eps, 0.0f);
                const float b = row_lb + gl * gl * 0.99999f;
                if (b <= B) break;
                out.lb = fminf(out.lb, b);
            }
#pragma unroll 1
            for (; xb > lx; --xb) {
                const float gr = fmaxf((cell - fx) + (float)(xb - lx - 1) * cell - eps, 0.0f);
                const float b = row_lb + gr * gr * 0.99999f;
                if (b <= B) break;
                out.lb = fminf(out.lb, b);
            }
            xa = max(xa, 0); xb = min(xb, g.nx - 1);
            if (xa <= xb) {
                const int* rowp = g.cell_start + (size_t)(zz * g.ny + yy) * g.nx;
                out.s = __ldg(rowp + xa); out.e = __ldg(rowp + xb + 1);
            }
        } else {
            out.lb = row_lb;
        }
    }
    return out;
}

// prof (profiling only, may be null): [0] += cycles of the row set-up, [1] += prefix + candidate scan, [2] += selection,
// [3] += searches, [4] += candidates scanned
__device__ __forceinline__ bool knn_warp_search(const Grid& g, float qx, float qy, float qz, float B, WarpKnnSmem& S,
                                                KnnM& out, float& lb, long long* prof = nullptr, const RowRange* pre = nullptr) {
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    long long tc0 = 0, tc1 = 0, tc2 = 0;
    if (prof) tc0 = clock64();
    const int K = g.rings, W = 2 * K + 1, nrows = W * W;
    float lbl = lb;                                   // lane-local lower bound of everything this lane drops
    if (lane < kSeeds) { S.okey[lane] = knn_key(B, 0x7fffffff); S.opos[lane] = -1; }
#pragma unroll 1
    for (int r = lane; r < nrows; r += 32) {
        const RowRange rr = pre ? pre[r] : knn_row_range(g, qx, qy, qz, B, r);
        lbl = fminf(lbl, rr.lb);
        S.rs[r] = rr.s; S.re[r] = rr.e;
    }
    __syncwarp();
    if (prof) tc1 = clock64();
    // Candidates of ALL rows as one flat list (prefix sums of the row lengths): lane l takes candidates l, l + 32, ...
    // wherever their rows are, so the point loads of different rows are independent and in flight together (walking
    // the rows one after the other costs one dependent memory round trip per row: 9 for cell = radius, up to 81).
    int total = 0;
#pragma unroll 1
    for (int base = 0; base < nrows; base += 32) {
        const int r = base + lane;
        const int len = r < nrows ? S.re[r] - S.rs[r] : 0;
        int incl = len;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const int t = __shfl_up_sync(full, incl, off);
            if (lane >= off) incl += t;
        }
        if (r < nrows) S.pref[r] = total + incl - len;
        total += __shfl_sync(full, incl, 31);
    }
    if (lane == 0) S.pref[nrows] = total;
    __syncwarp();
    int cnt = 0;
    bool overflow = false;
    int row = 0;                                      // row of this lane's current candidate (candidates ascend per lane)
    // cell = radius (9 rows): the prefix sums in registers, so a candidate's row is nine compares instead of a walk
    // through shared memory with one dependent load per step
    const bool few_rows = nrows <= 9;
    int pr[9];
#pragma unroll
    for (int r = 0; r < 9; ++r) pr[r] = (few_rows && r < nrows) ? S.pref[r + 1] : 0x7fffffff;
    constexpr int kU = 4;                             // candidates per lane and trip: that many loads in flight
#pragma unroll 1
    for (int c0 = 0; c0 < total; c0 += 32 * kU) {
        int jj[kU];
        bool in[kU];
        float4 pp[kU];
#pragma unroll
        for (int u = 0; u < kU; ++u) {
            const int c = c0 + u * 32 + lane;
            in[u] = c < total;
            jj[u] = 0;
            if (in[u]) {
                if (few_rows) {
                    row = 0;
#pragma unroll
                    for (int r = 0; r < 8; ++r) row += (c >= pr[r]) ? 1 : 0;
                } else {
                    while (c >= S.pref[row + 1]) ++row;
                }
                jj[u] = S.rs[row] + (c - S.pref[row]);
                pp[u] = __ldg(&g.pts[jj[u]]);
            }
        }
#pragma unroll
        for (int u = 0; u < kU; ++u) {
            if (c0 + u * 32 >= total) break;          // (uniform) nothing left for this and the following slots
            bool hit = false;
            float d = 0.0f;
            int pi = 0;
            if (in[u]) {
                d = dist2(qx, qy, qz, pp[u]);
                pi = __float_as_int(pp[u].w);
                hit = d <= B;
                if (!hit) lbl = fminf(lbl, d);
            }
            const unsigned bits = __ballot_sync(full, hit);
            const int slot = cnt + __popc(bits & ((1u << lane) - 1u));
            if (hit && slot < kWarpKnnCap) { S.key[slot] = knn_key(d, pi); S.pos[slot] = jj[u]; }
            cnt += __popc(bits);
        }
        if (cnt > kWarpKnnCap) { overflow = true; break; }
    }
    __syncwarp();
    if (overflow) return false;
    if (prof) tc2 = clock64();
    // Rank of every candidate inside the bound = number of candidates that precede it in (d2, index) order; ranks 0..6 are
    // the list.  All-pairs over the (few: ~20 of ~45 scanned) hits with broadcast shared-memory reads: the iterations
    // are independent, so unrolled they pipeline (~500 cycles).  Measured alternatives on the C2 loop (clock64 per
    // phase, tools/timeline.py): seven warp-wide minimum extractions with REDUX 2200-2900 cycles (a serial chain of
    // collectives), this loop not unrolled ~2000.
#pragma unroll 1
    for (int en = lane; en < cnt; en += 32) {
        const unsigned long long ke = S.key[en];
        int rank = 0;
#pragma unroll 4
        for (int f = 0; f < cnt; ++f) rank += (S.key[f] < ke) ? 1 : 0;
        if (rank < kSeeds) { S.okey[rank] = ke; S.opos[rank] = S.pos[en]; }
        else lbl = fminf(lbl, __uint_as_float((unsigned)(ke >> 32)));
    }
    lbl = __uint_as_float(__reduce_min_sync(full, __float_as_uint(lbl)));      // lbl >= 0: bit patterns order like the values
    __syncwarp();
#pragma unroll
    for (int i = 0; i < kSeeds; ++i) { out.key[i] = S.okey[i]; out.pos[i] = S.opos[i]; }
    lb = lbl;
    __syncwarp();
    if (prof && lane == 0) {
        const long long tc3 = clock64();
        prof[0] += tc1 - tc0; prof[1] += tc2 - tc1; prof[2] += tc3 - tc2; prof[3] += 1; prof[4] += total;
    }
    return true;
}

// ---- exact 1-NN (post-run point-to-point metrics, DCReg/include/utils.hpp:538-589) ---------------------------
// Nearest target point of q in a dense grid: rings of cells of growing Chebyshev radius around q's cell, clipped to
// the grid box, until the best distance found is no larger than the distance to the next ring.  FLANN-style float32
// squared distances.  Returns the squared distance (3e38 if the grid is empty).
__device__ __forceinline__ float nn1_search(const Grid& g, float qx, float qy, float qz) {
    const float cell = (float)(1.0 / g.inv_cell);
    const int lx = cell_coord(qx, g.inv_cell) - g.ox, ly = cell_coord(qy, g.inv_cell) - g.oy, lz = cell_coord(qz, g.inv_cell) - g.oz;
    // first ring that can touch the box, last ring that still does
    const int ox = lx < 0 ? -lx : (lx >= g.nx ? lx - g.nx + 1 : 0);
    const int oy = ly < 0 ? -ly : (ly >= g.ny ? ly - g.ny + 1 : 0);
    const int oz = lz < 0 ? -lz : (lz >= g.nz ? lz - g.nz + 1 : 0);
    const int r0 = max(ox, max(oy, oz));
    const int r1 = max(max(lx, g.nx - 1 - lx), max(max(ly, g.ny - 1 - ly), max(lz, g.nz - 1 - lz)));
    float best = 3.0e38f;
#pragma unroll 1
    for (int r = r0; r <= r1; ++r) {
        if (r > 0) {
            const float lb = (float)(r - 1) * cell * 0.99999f;      // every point of ring r is at least this far
            if (lb * lb > best) break;
        }
        const int z0 = max(-r, -lz), z1 = min(r, g.nz - 1 - lz);
        const int y0 = max(-r, -ly), y1 = min(r, g.ny - 1 - ly);
#pragma unroll 1
        for (int dz = z0; dz <= z1; ++dz) {
#pragma unroll 1
            for (int dy = y0; dy <= y1; ++dy) {
                const int* rowp = g.cell_start + (size_t)((lz + dz) * g.ny + (ly + dy)) * g.nx;
                const bool shell = (dz == -r) || (dz == r) || (dy == -r) || (dy == r);
                if (shell) {                                         // whole x-span of the ring, one contiguous range
                    const int xa = max(lx - r, 0), xb = min(lx + r, g.nx - 1);
                    if (xa > xb) continue;
                    const int s = __ldg(rowp + xa), e = __ldg(rowp + xb + 1);
                    for (int j = s; j < e; ++j) best = fminf(best, dist2(qx, qy, qz, __ldg(&g.pts[j])));
                } else {                                             // interior row: only the two end cells dx = +-r
                    for (int sgn = -1; sgn <= 1; sgn += 2) {
                        const int xx = lx + sgn * r;
                        if (xx < 0 || xx >= g.nx) continue;
                        const int s = __ldg(rowp + xx), e = __ldg(rowp + xx + 1);
                        for (int j = s; j < e; ++j) best = fminf(best, dist2(qx, qy, qz, __ldg(&g.pts[j])));
                    }
                }
            }
        }
    }
    return best;
}

// per-block partial sums: [0] sum of distances, [1] sum of squared distances below the threshold, [2] count below it.
// When T != nullptr the query is fl32(T p) (pcl::transformPointCloud: FP64 math, float32 store), else p itself.
__global__ void nn1_metrics_kernel(const float4* __restrict__ q, long long n, const double* __restrict__ T, Grid g,
                                   double threshold, double* __restrict__ partials) {
    __shared__ double sh[3][8];
    double sd = 0.0, ssq = 0.0, cnt = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float4 p = __ldg(&q[i]);
        float x = p.x, y = p.y, z = p.z;
        if (T) {
            const double px = p.x, py = p.y, pz = p.z;
            x = (float)(T[0] * px + T[1] * py + T[2] * pz + T[3]);
            y = (float)(T[4] * px + T[5] * py + T[6] * pz + T[7]);
            z = (float)(T[8] * px + T[9] * py + T[10] * pz + T[11]);
        }
        const float d2 = nn1_search(g, x, y, z);
        const double dist = sqrt((double)d2);
        sd += dist;
        if (dist < threshold) { ssq += (double)d2; cnt += 1.0; }
    }
    for (int off = 16; off > 0; off >>= 1) {
        sd += __shfl_down_sync(0xffffffffu, sd, off);
        ssq += __shfl_down_sync(0xffffffffu, ssq, off);
        cnt += __shfl_down_sync(0xffffffffu, cnt, off);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { sh[0][warp] = sd; sh[1][warp] = ssq; sh[2][warp] = cnt; }
    __syncthreads();
    if (threadIdx.x < 3) {
        double s = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += sh[threadIdx.x][w];
        partials[blockIdx.x * 3 + threadIdx.x] = s;
    }
}

// transform + float32 store of a cloud (aligned copy for the backward Chamfer pass)
__global__ void transform_points_kernel(const float4* __restrict__ in, long long n, const double* __restrict__ T,
                                        float4* __restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 p = in[i];
    const double px = p.x, py = p.y, pz = p.z;
    out[i] = make_float4((float)(T[0] * px + T[1] * py + T[2] * pz + T[3]), (float)(T[4] * px + T[5] * py + T[6] * pz + T[7]),
                         (float)(T[8] * px + T[9] * py + T[10] * pz + T[11]), p.w);
}

// ---- point-to-point metrics for many poses (dcreg_point_to_point_metrics_batch) ---------------------------------
// Pose records: 16 doubles each, [0..11] the top three rows of T, [12] margin, [13] shrink (p2p_bound.hpp).
constexpr int kPoseRec = 16;

// fl32(T p): the expression of nn1_metrics_kernel / transform_points_kernel, so every point lands on the same float
__device__ __forceinline__ float3 posed_point(const double* __restrict__ T, const float4 p) {
    const double px = p.x, py = p.y, pz = p.z;
    return make_float3((float)(T[0] * px + T[1] * py + T[2] * pz + T[3]), (float)(T[4] * px + T[5] * py + T[6] * pz + T[7]),
                       (float)(T[8] * px + T[9] * py + T[10] * pz + T[11]));
}

// cell coordinate of an FP64 position, clamped so a far query cannot overflow int (a clamped cell is nearer to the
// grid box than the true one, so the ring bounds below stay lower bounds)
__device__ __forceinline__ int cell_coord_clamped(double v, double inv_cell) {
    return (int)fmin(fmax(floor(v * inv_cell), -1073741824.0), 1073741824.0);
}

__device__ __forceinline__ float posed_scan_range(const Grid& g, const double* __restrict__ T, int s, int e, float yx,
                                                  float yy, float yz, float best) {
#pragma unroll 1
    for (int j = s; j < e; ++j) {
        const float3 a = posed_point(T, __ldg(&g.pts[j]));
        best = fminf(best, dist2(yx, yy, yz, make_float4(a.x, a.y, a.z, 0.f)));
    }
    return best;
}

// Smallest float d2(y, fl32(T p)) over the source points p of a dense grid built in the source's own frame: the
// value nn1_search returns for y over a grid built on the aligned copy.  Same ring walk around q' = R^T (y - t);
// a ring is skipped by the bound (*) of p2p_bound.hpp, which keeps the minimum exact.
__device__ __forceinline__ float nn1_search_posed(const Grid& g, const double* __restrict__ T, float yx, float yy, float yz) {
    const double vx = (double)yx - T[3], vy = (double)yy - T[7], vz = (double)yz - T[11];
    const double qx = T[0] * vx + T[4] * vy + T[8] * vz, qy = T[1] * vx + T[5] * vy + T[9] * vz, qz = T[2] * vx + T[6] * vy + T[10] * vz;
    const double margin = T[12], shrink = T[13];
    const double cell = 1.0 / g.inv_cell;
    const int lx = cell_coord_clamped(qx, g.inv_cell) - g.ox, ly = cell_coord_clamped(qy, g.inv_cell) - g.oy,
              lz = cell_coord_clamped(qz, g.inv_cell) - g.oz;
    const int ox = lx < 0 ? -lx : (lx >= g.nx ? lx - g.nx + 1 : 0);
    const int oy = ly < 0 ? -ly : (ly >= g.ny ? ly - g.ny + 1 : 0);
    const int oz = lz < 0 ? -lz : (lz >= g.nz ? lz - g.nz + 1 : 0);
    const int r0 = max(ox, max(oy, oz));
    const int r1 = max(max(lx, g.nx - 1 - lx), max(max(ly, g.ny - 1 - ly), max(lz, g.nz - 1 - lz)));
    float best = 3.0e38f;
#pragma unroll 1
    for (int r = r0; r <= r1; ++r) {
        if (r > 0) {
            const double l = (double)(r - 1) * cell * 0.99999 - margin;
            if (l > 0.0 && l * l * shrink > (double)best) break;
        }
        const int z0 = max(-r, -lz), z1 = min(r, g.nz - 1 - lz);
        const int y0 = max(-r, -ly), y1 = min(r, g.ny - 1 - ly);
#pragma unroll 1
        for (int dz = z0; dz <= z1; ++dz) {
#pragma unroll 1
            for (int dy = y0; dy <= y1; ++dy) {
                const int* rowp = g.cell_start + (size_t)((lz + dz) * g.ny + (ly + dy)) * g.nx;
                const bool shell = (dz == -r) || (dz == r) || (dy == -r) || (dy == r);
                if (shell) {                                         // whole x-span of the ring, one contiguous range
                    const int xa = max(lx - r, 0), xb = min(lx + r, g.nx - 1);
                    if (xa > xb) continue;
                    best = posed_scan_range(g, T, __ldg(rowp + xa), __ldg(rowp + xb + 1), yx, yy, yz, best);
                } else {                                             // interior row: only the two end cells dx = +-r
                    for (int sgn = -1; sgn <= 1; sgn += 2) {
                        const int xx = lx + sgn * r;
                        if (xx < 0 || xx >= g.nx) continue;
                        best = posed_scan_range(g, T, __ldg(rowp + xx), __ldg(rowp + xx + 1), yx, yy, yz, best);
                    }
                }
            }
        }
    }
    return best;
}

// Forward pass, blockIdx.y = pose: nn1_metrics_kernel's decomposition and per-block partials for each pose.
__global__ void nn1_metrics_poses_kernel(const float4* __restrict__ q, long long n, const double* __restrict__ poses, Grid g,
                                         double threshold, double* __restrict__ partials) {
    __shared__ double sh[3][8];
    const double* T = poses + (size_t)blockIdx.y * kPoseRec;
    double sd = 0.0, ssq = 0.0, cnt = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float3 a = posed_point(T, __ldg(&q[i]));
        const float d2 = nn1_search(g, a.x, a.y, a.z);
        const double dist = sqrt((double)d2);
        sd += dist;
        if (dist < threshold) { ssq += (double)d2; cnt += 1.0; }
    }
    for (int off = 16; off > 0; off >>= 1) {
        sd += __shfl_down_sync(0xffffffffu, sd, off);
        ssq += __shfl_down_sync(0xffffffffu, ssq, off);
        cnt += __shfl_down_sync(0xffffffffu, cnt, off);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { sh[0][warp] = sd; sh[1][warp] = ssq; sh[2][warp] = cnt; }
    __syncthreads();
    if (threadIdx.x < 3) {
        double s = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += sh[threadIdx.x][w];
        partials[((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 3 + threadIdx.x] = s;
    }
}

// Backward (Chamfer) pass, blockIdx.y = pose: target point -> nearest aligned source point through the source-frame
// grid; per-block sum of distances in nn1_metrics_kernel's order.
__global__ void nn1_chamfer_poses_kernel(const float4* __restrict__ tgt, long long m, const double* __restrict__ poses,
                                         Grid gs, double* __restrict__ partials) {
    __shared__ double sh[8];
    const double* T = poses + (size_t)blockIdx.y * kPoseRec;
    double sd = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (long long)gridDim.x * blockDim.x) {
        const float4 y = __ldg(&tgt[i]);
        sd += sqrt((double)nn1_search_posed(gs, T, y.x, y.y, y.z));
    }
    for (int off = 16; off > 0; off >>= 1) sd += __shfl_down_sync(0xffffffffu, sd, off);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) sh[warp] = sd;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += sh[w];
        partials[(size_t)blockIdx.y * gridDim.x + blockIdx.x] = s;
    }
}

// One thread per pose: the host sums of dcreg_point_to_point_metrics (block order 0..grid-1), then
// out = { sqrt(sum_sq / n), count / n, (sum_f / n + sum_b / m) / 2, count }.
__global__ void p2p_finish_kernel(const double* __restrict__ pf, int gridf, const double* __restrict__ pb, int gridb,
                                  int n_poses, long long n, long long m, double* __restrict__ out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_poses) return;
    double sum_fwd = 0, sum_sq = 0, valid = 0, sum_bwd = 0;
    const double* f = pf + (size_t)k * gridf * 3;
    for (int b = 0; b < gridf; ++b) { sum_fwd += f[3 * b]; sum_sq += f[3 * b + 1]; valid += f[3 * b + 2]; }
    const double* bb = pb + (size_t)k * gridb;
    for (int b = 0; b < gridb; ++b) sum_bwd += bb[b];
    out[4 * k + 0] = sqrt(sum_sq / (double)n);
    out[4 * k + 1] = valid / (double)n;
    out[4 * k + 2] = 0.5 * (sum_fwd / (double)n + sum_bwd / (double)m);
    out[4 * k + 3] = valid;
}

// Plane through the 5 neighbours: least squares of [nb] x = -1, n = x/|x|, d = 1/|x|, gates
// |x| >= min_norm and max_j (n.nb_j + d)^2 < thickness^2 (icp_test_runner.cpp:1727-1773).
// Returns true and (n, d) when a valid plane exists.
__device__ __forceinline__ bool fit_plane(const Grid& g, const int (&kpos)[5], double min_norm, double thickness,
                                          double& nx, double& ny, double& nz, double& d) {
    double A[15], b[5], x[3];
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        const float4 p = __ldg(&g.pts[kpos[j]]);
        A[j * 3 + 0] = (double)p.x;
        A[j * 3 + 1] = (double)p.y;
        A[j * 3 + 2] = (double)p.z;
        b[j] = -1.0;
    }
    dla::colpiv_qr_solve<5, 3>(A, b, x);
    const double ps = sqrt(x[0] * x[0] + x[1] * x[1] + x[2] * x[2]);
    if (!(ps >= min_norm)) return false;                 // :1752 (also rejects NaN)
    nx = x[0] / ps; ny = x[1] / ps; nz = x[2] / ps; d = 1.0 / ps;
    double worst = 0.0;
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        const float4 p = __ldg(&g.pts[kpos[j]]);          // re-read (L1 hit) instead of holding 15 more doubles
        double e = nx * (double)p.x + ny * (double)p.y + nz * (double)p.z + d;
        e *= e;
        worst = fmax(worst, e);
    }
    return worst < thickness * thickness;                // :1772-1773
}

// The same fit with the register-resident QR (small_la.cuh: same operations in the same order, bit-identical results).  A
// separate function with its own register allocation: it is called from the fit work list of the loop kernel, where
// almost nothing is live across the call (inlined into a loop body full of live state it spills; measured 3.7x slower
// there).  Measured and rejected (round 2): a variant of the QR with hardware reciprocal / rsqrt seeds instead of the
// ~30 IEEE divisions and square roots on the fit's dependent chain) makes a fit 7 -> 6 us, but on exactly rank-deficient
// neighbourhoods (collinear lattice points) its 1-ulp differences flip the pivoted QR's rank decision, and the loop then
// disagrees with the generic fit by one correspondence (tests/test_gpu_parity.py, lattice scene).
__device__ __noinline__ bool fit_plane_reg(const Grid& g, const int (&kpos)[5], double min_norm, double thickness,
                                           double& nx, double& ny, double& nz, double& d) {
    double A[5][3], b[5], x[3];
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        const float4 p = __ldg(&g.pts[kpos[j]]);
        A[j][0] = (double)p.x;
        A[j][1] = (double)p.y;
        A[j][2] = (double)p.z;
        b[j] = -1.0;
    }
    dla::colpiv_qr_solve_reg<5, 3>(A, b, x);
    const double ps = sqrt(x[0] * x[0] + x[1] * x[1] + x[2] * x[2]);
    if (!(ps >= min_norm)) return false;                 // :1752 (also rejects NaN)
    nx = x[0] / ps; ny = x[1] / ps; nz = x[2] / ps; d = 1.0 / ps;
    double worst = 0.0;
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        const float4 p = __ldg(&g.pts[kpos[j]]);
        double e = nx * (double)p.x + ny * (double)p.y + nz * (double)p.z + d;
        e *= e;
        worst = fmax(worst, e);
    }
    return worst < thickness * thickness;                // :1772-1773
}

}  // namespace corr
