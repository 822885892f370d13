// st_deform.cuh -- the per-triangle arithmetic that k_deform (st_deform.cu) and the coarse-graining kernels
// (st_deform_scale.cu) share, so that both spell every sum in the oracle's order from one definition; the gather of
// an f8 position and the histogram bin rule, shared with the pair-dispersion kernel (st_disperse.cu) as well.
#pragma once
#include "st_kernels.h"

namespace st {

__device__ __forceinline__ pt ld_ro_pt(const pt* __restrict__ a, int i)
{
    const double2 v = __ldg(reinterpret_cast<const double2*>(a + i));
    pt r; r.y = v.x; r.x = v.y; return r;
}

// bin of v on ascending edges e[0..ne): searchsorted(e, v, side="right"), so ne + 1 bins with underflow and overflow
__device__ __forceinline__ int bin_right(const double* __restrict__ e, int ne, double v)
{
    if (v != v) return ne;                                      // NaN sorts last, as numpy's searchsorted
    int lo = 0, hi = ne;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (e[mid] <= v) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// 2A = (X0 Y1 - X1 Y0) + (X1 Y2 - X2 Y1) + (X2 Y0 - X0 Y2), left to right
__device__ __forceinline__ double twice_area(double X0, double X1, double X2, double Y0, double Y1, double Y2)
{
    const double t01 = __dsub_rn(__dmul_rn(X0, Y1), __dmul_rn(X1, Y0));
    const double t12 = __dsub_rn(__dmul_rn(X1, Y2), __dmul_rn(X2, Y1));
    const double t20 = __dsub_rn(__dmul_rn(X2, Y0), __dmul_rn(X0, Y2));
    return __dadd_rn(__dadd_rn(t01, t12), t20);
}

// sum over the edges 0->1, 1->2, 2->0 of (F_{i+1} + F_i)(Z_{i+1} - Z_i), left to right
__device__ __forceinline__ double edge_sum(double F0, double F1, double F2, double Z0, double Z1, double Z2)
{
    const double e01 = __dmul_rn(__dadd_rn(F1, F0), __dsub_rn(Z1, Z0));
    const double e12 = __dmul_rn(__dadd_rn(F2, F1), __dsub_rn(Z2, Z1));
    const double e20 = __dmul_rn(__dadd_rn(F0, F2), __dsub_rn(Z0, Z2));
    return __dadd_rn(__dadd_rn(e01, e12), e20);
}

}  // namespace st
