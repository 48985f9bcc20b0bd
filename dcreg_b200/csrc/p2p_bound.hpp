// p2p_bound.hpp - pruning bound of the batched Chamfer pass (host logic, no CUDA).
//
// dcreg_point_to_point_metrics_batch finds, for a target point y and a pose (R, t), the nearest ALIGNED source point
// a = fl32(R p + t) (the float32 store of pcl::transformPointCloud, evaluated in FP64) with the FLANN float32 squared
// distance d2(y, a), exactly as the single call does over a grid built on the aligned copy.  It searches instead one
// grid over the source in its own frame, around q' = R^T (y - t) (FP64), in rings of cells of growing Chebyshev
// radius.  A ring whose points are all at least L from q' (source frame) is skipped when
//
//         (L - margin)^2 * shrink > best                                                                      (*)
//
// with best the smallest float d2 found so far.  Derivation, for a source point p with |p - q'| >= L, b = R p + t:
//   1. |a - b| <= E_a = (2^-24 + 2^-50) (|R|_F pmax + |t|): one float32 rounding (relative 2^-24 per component) of
//      a 4-term FP64 dot product (error below 2^-50 of the sum of the magnitudes of its terms).
//   2. q' is R^T (y - t) up to E_q = 2^-50 |R|_F (ymax + |t|) (one subtraction and a 3-term dot product in FP64).
//   3. b - y = R (p - q'') + (R R^T - I)(y - t), q'' = R^T (y - t) exactly.  With e >= ||R^T R - I||_F (R as given,
//      not necessarily orthonormal: poses read back from 8-decimal text are not), sigma_min(R) >= sqrt(1 - e) and
//      sigma_max(R) <= sqrt(1 + e), so |b - y| >= sqrt(1 - e) (L - E_q) - e (ymax + |t|).
//   4. Hence the exact distance D = |a - y| >= sqrt(1 - e) (L - margin) + 1e-18 with
//      margin = (E_a + sqrt(1 + e) E_q + e (ymax + |t|) + 1e-18) / sqrt(1 - e) (rounded up by a factor 1 + 1e-6).
//   5. The float d2 = fl(fl(ex^2 + ey^2) + ez^2), ex = fl(y_x - a_x), carries at most 5 relative roundings of 2^-24,
//      so d2 >= D^2 (1 - 5 * 2^-24) while no square underflows; D > 1e-18 keeps the largest square normal and the
//      absolute subnormal error of the others (< 2^-149) below 1e-9 of D^2.  The FP64 evaluation of (*) itself adds
//      three roundings of 2^-53.  c = 8 covers all of it: shrink = (1 - e)(1 - 8 * 2^-24).
//   6. L: q' lies in cell floor(q' / cell), a ring-r cell is r cells away on some axis, so every point of ring r is
//      at least (r - 1) cell away; the FP64 cell-coordinate roundings are below 2^-21 cells inside the +-2^19-cell
//      range of the grid, and the device takes L = (r - 1) cell 0.99999, the bound nn1_search uses.
// Every point of a skipped ring thus has float d2 >= best, so the minimum (and every sum built on it) equals the
// exhaustive one.  If R is far from a rotation (e >= 1) nothing is skipped: the search is exhaustive, still exact.
#pragma once
#include <cmath>
#include <limits>

namespace p2p_bound {

struct Bound {
    double margin;   // source-frame distance subtracted from a ring's lower bound
    double shrink;   // factor on the squared bound before it is compared with the best float d2
};

// T: row-major 4x4 pose; pmax >= max |p| over the source, ymax >= max |y| over the target (Euclidean norms)
inline Bound backward_bound(const double* T, double pmax, double ymax) {
    double fr2 = 0.0, e2 = 0.0;
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            fr2 += T[4 * i + j] * T[4 * i + j];
            double s = i == j ? -1.0 : 0.0;
            for (int k = 0; k < 3; ++k) s += T[4 * k + i] * T[4 * k + j];
            e2 += s * s;
        }
    const double e = std::sqrt(e2) * (1.0 + 1e-6) + 1e-15;    // + the rounding of R^T R - I itself
    const double fr = std::sqrt(fr2) * (1.0 + 1e-6);
    const double tn = std::sqrt(T[3] * T[3] + T[7] * T[7] + T[11] * T[11]) * (1.0 + 1e-6);
    if (!(e < 1.0) || !std::isfinite(fr + tn + pmax + ymax)) return {std::numeric_limits<double>::infinity(), 0.0};
    const double Ea = (0x1p-24 + 0x1p-50) * (fr * pmax + tn);
    const double Eq = 0x1p-50 * fr * (ymax + tn);
    const double m0 = Ea + std::sqrt(1.0 + e) * Eq + e * (ymax + tn) + 1e-18;
    return {m0 / std::sqrt(1.0 - e) * (1.0 + 1e-6), (1.0 - e) * (1.0 - 8.0 * 0x1p-24)};
}

}  // namespace p2p_bound
