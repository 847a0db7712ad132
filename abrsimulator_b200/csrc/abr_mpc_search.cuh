// Pieces of the MPC search shared by the search kernels of abr_mpc.cu (SPEC §5.1-5.6) and the scenario kernel of
// abr_mpc_scen.cu (SPEC §5.7): the interior step of the rollout, the branch-and-bound bound and its tables, and the
// (value, linear index) comparison of the argmin.
#pragma once
#include "abr_common.cuh"

namespace abr {
namespace {

struct SearchOut { double q; int idx; };

// Interior step i of mpc.py:144-156 (+ next_buffer, mpc.py:111-118) on the running state.
template <bool CLAMP>
__device__ __forceinline__ void interior(double& vq, double& qv, double& rt, double& b, const double u,
                                         const double absdu, const double rbv, const double dlv, const double L,
                                         const double B) {
    vq = dadd(vq, u);
    qv = dadd(qv, absdu);
    const double d = dsub(rbv, b);
    rt = dadd(rt, CLAMP ? max0(d) : d);
    const double t = max0(dsub(b, dlv));
    const double tl = dadd(t, L);
    const double w = max0(dsub(tl, B));
    b = max0(dsub(tl, w));
}

// ---- branch and bound: what the levels still to come can add at best, and the bound built from it ----
// After action a at the level before,
//   g5[a]  = max over a5 of U5[a5] - vw |U5[a5] - U5[a]|                       (the last level)
//   g45[a] = max over a4 of U4[a4] - vw |U4[a4] - U4[a]| + g5[a4]              (the last two levels)
// (rebuffering still to come is bounded by zero).  These combine utility and smoothness, which the objective
// accumulates in separate sums, so a bound built from them holds in real arithmetic only; the slack in prune_bound
// covers the rounding of the dozen operations in between a million times over.  Lanes a < A of every warp of the
// session compute the same entries.
__device__ __forceinline__ void bound_tables(const double* __restrict__ sU, const int A, const int h, const double vw,
                                             double* __restrict__ g5, double* __restrict__ g45, const int lane) {
    const int i4 = h - 2, i5 = h - 1;
    if (lane < A) {
        double m = __longlong_as_double(0xfff0000000000000ll);
        for (int a5 = 0; a5 < A; ++a5) {
            const double x = sU[i5 * A + a5] - vw * fabs(sU[i5 * A + a5] - sU[i5 * A + lane]);
            m = x > m ? x : m;
        }
        g5[lane] = m;
    }
    __syncwarp();
    if (lane < A) {
        double m = __longlong_as_double(0xfff0000000000000ll);
        for (int a4 = 0; a4 < A; ++a4) {
            const double x = sU[i4 * A + a4] - vw * fabs(sU[i4 * A + a4] - sU[i4 * A + lane]) + g5[a4];
            m = x > m ? x : m;
        }
        g45[lane] = m;
    }
    __syncwarp();
}

// upper bound of the value of every completion, from the sums so far and the best still to come (g5 / g45 entry)
template <bool VW1>
__device__ __forceinline__ double prune_bound(const double vq, const double qv, const double rt, const double g,
                                              const double vw, const double rw) {
    const double sq = VW1 ? qv : dmul(vw, qv), sr = dmul(rw, rt);
    const double slack = 1e-9 * (fabs(vq) + sq + sr + fabs(g) + 1.0);
    return (dsub(dsub(vq, sq), sr) + g) + slack;
}

__device__ __forceinline__ void better(double& q, int& idx, const double oq, const int oi) {
    if (oq > q || (oq == q && oi < idx)) { q = oq; idx = oi; }
}

}  // namespace
}  // namespace abr
