// st_sample.cu -- SI3 T-cell fields sampled along the buoy trajectories: the host cell's value, or a bilinear
// interpolation between the four T-points around the buoy, at every sampled row.
//
// Definitions (DESIGN.md section 15, oracle/sample_ref.py).  Per buoy p of a row: its cell (jT, iT) from the state
// (bit 31 stripped), its f8 position P from the row, its row mask m.  m == 0, or a cell outside 1..Nj-2 x 1..Ni-2,
// gives FillValue in every field.  Otherwise:
//   cell:      F[jT,iT] (an exact f4 copy);
//   bilinear:  the T-quad on P's side of the grid lines S->N and W->E through T[jT,iT] (a tie goes to the higher
//              index); (xi, eta) by the closed-form inverse bilinear map (k2 == 0: the parallelogram's linear root),
//              each clamped to [0,1]; the corners SW, SE, NE, NW weighted (1-xi)(1-eta), xi(1-eta), xi eta, (1-xi) eta,
//              a corner with tmask 0 or a non-finite value dropped, the rest renormalised; no corner kept: the cell
//              value.  In f8, spelled with __d*_rn so that nothing is contracted into an FMA, rounded once to f4.
// A non-finite result gives FillValue.  The stencil reaches T[jT+-1, iT+-1]: inside the grid for every cell that is
// sampled (DESIGN.md section 15 shows that every masked-1 row a step writes has such a cell).
//
// Kernel, on the caller's stream: k_sample<MODE>, one thread per buoy over one wave of resident blocks.  The cell word,
// the mask and, for a buoy that is sampled in bilinear mode, the position stream through (touch once); T-points, tmask
// and the field planes are gathered through the read-only path with the L2 evict_last policy, so the grid and the
// fields stay resident in L2; one coalesced f4 store per field into out (nF, nP).
#include "st_kernels.h"

namespace st {

constexpr int SP_BLOCK = 256;

__device__ __forceinline__ float sp_fill(float v) { return isfinite(v) ? v : (float)ST_FILL; }
__device__ __forceinline__ double sp_clamp01(double v) { return v > 0.0 ? (v < 1.0 ? v : 1.0) : 0.0; }
// (B.x - A.x)(P.y - A.y) - (B.y - A.y)(P.x - A.x): > 0 when P lies left of A->B
__device__ __forceinline__ double sp_orient(pt A, pt B, pt P)
{
    return __dsub_rn(__dmul_rn(__dsub_rn(B.x, A.x), __dsub_rn(P.y, A.y)),
                     __dmul_rn(__dsub_rn(B.y, A.y), __dsub_rn(P.x, A.x)));
}
__device__ __forceinline__ double sp_cross(double ux, double uy, double vx, double vy)
{
    return __dsub_rn(__dmul_rn(ux, vy), __dmul_rn(uy, vx));
}
__device__ __forceinline__ float sp_ld(const float* __restrict__ a, long long i)
{
    float r;
    asm("ld.global.nc.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(r) : "l"(a + i), "l"(l2_keep_policy()));
    return r;
}

template <int MODE>
__global__ void __launch_bounds__(SP_BLOCK) k_sample(long long nP, int Nj, int Ni, const int2* __restrict__ cell,
                                                     const int8_t* __restrict__ mask, const pt* __restrict__ yx,
                                                     const pt* __restrict__ T, const int8_t* __restrict__ tmask,
                                                     const float* __restrict__ F, long long stride, int nF,
                                                     float* __restrict__ out)
{
    for (long long p = (long long)blockIdx.x * SP_BLOCK + threadIdx.x; p < nP; p += (long long)gridDim.x * SP_BLOCK) {
        const int2 cw = __ldcs(cell + p);
        const int8_t m = __ldcs(mask + p);
        const int jT = cw.x & 0x7fffffff, iT = cw.y;
        if (m == 0 || jT < 1 || jT > Nj - 2 || iT < 1 || iT > Ni - 2) {
            for (int f = 0; f < nF; ++f) __stcs(out + f * nP + p, (float)ST_FILL);
            continue;
        }
        const int c = jT * Ni + iT;
        ST_CHECK_CELL(c, Ni + 1, Nj, Ni);
        if (MODE == 0) {
#pragma unroll 4
            for (int f = 0; f < nF; ++f) __stcs(out + f * nP + p, sp_fill(sp_ld(F, f * stride + c)));
            continue;
        }
        // 1. the T-quad: P's side of S->N gives i0, of W->E gives j0 (a right-handed grid: sample.tpoints checks it).
        // The position is streamed only for the buoys that are sampled, issued with the pick's four gathers.
        const pt P = ld_stream_pt(yx + p);
        const pt S = ldg_pt(T, c - Ni), N = ldg_pt(T, c + Ni), W = ldg_pt(T, c - 1), E = ldg_pt(T, c + 1);
        const int a = c - (sp_orient(W, E, P) < 0.0 ? Ni : 0) - (sp_orient(S, N, P) > 0.0 ? 1 : 0);   // SW corner
        // its corners and their land flags, gathered together (three of the four T-points were just read)
        const pt pa = ldg_pt(T, a), pb = ldg_pt(T, a + 1), pc = ldg_pt(T, a + Ni + 1), pd = ldg_pt(T, a + Ni);
        const bool la = __ldg(tmask + a) != 0, lb = __ldg(tmask + a + 1) != 0, lc = __ldg(tmask + a + Ni + 1) != 0,
                   ld = __ldg(tmask + a + Ni) != 0;
        // 2. inverse bilinear coordinates
        const double ex = __dsub_rn(pb.x, pa.x), ey = __dsub_rn(pb.y, pa.y);
        const double fx = __dsub_rn(pd.x, pa.x), fy = __dsub_rn(pd.y, pa.y);
        const double gx = __dsub_rn(__dadd_rn(__dsub_rn(pa.x, pb.x), pc.x), pd.x);
        const double gy = __dsub_rn(__dadd_rn(__dsub_rn(pa.y, pb.y), pc.y), pd.y);
        const double hx = __dsub_rn(P.x, pa.x), hy = __dsub_rn(P.y, pa.y);
        const double k2 = sp_cross(gx, gy, fx, fy);
        const double k1 = __dadd_rn(sp_cross(ex, ey, fx, fy), sp_cross(hx, hy, gx, gy));
        const double k0 = sp_cross(hx, hy, ex, ey);
        double eta;
        if (k2 == 0.0) {
            eta = __ddiv_rn(-k0, k1);                                          // a parallelogram: linear
        } else {
            double disc = __dsub_rn(__dmul_rn(k1, k1), __dmul_rn(__dmul_rn(4.0, k0), k2));
            if (disc < 0.0) disc = 0.0;
            const double q = __dmul_rn(-0.5, __dadd_rn(k1, copysign(__dsqrt_rn(disc), k1)));
            eta = __ddiv_rn(k0, q);
        }
        const double dx = __dadd_rn(ex, __dmul_rn(gx, eta)), dy = __dadd_rn(ey, __dmul_rn(gy, eta));
        double xi = fabs(dx) >= fabs(dy) ? __ddiv_rn(__dsub_rn(hx, __dmul_rn(fx, eta)), dx)
                                         : __ddiv_rn(__dsub_rn(hy, __dmul_rn(fy, eta)), dy);
        xi = sp_clamp01(xi);
        eta = sp_clamp01(eta);
        // 3. weights SW, SE, NE, NW
        const double xm = __dsub_rn(1.0, xi), em = __dsub_rn(1.0, eta);
        const double w0 = __dmul_rn(xm, em), w1 = __dmul_rn(xi, em), w2 = __dmul_rn(xi, eta), w3 = __dmul_rn(xm, eta);
        for (int f = 0; f < nF; ++f) {
            const float* Ff = F + f * stride;
            const double v0 = sp_ld(Ff, a), v1 = sp_ld(Ff, a + 1), v2 = sp_ld(Ff, a + Ni + 1), v3 = sp_ld(Ff, a + Ni);
            double num = 0.0, den = 0.0;
            if (la && isfinite(v0)) { num = __dadd_rn(num, __dmul_rn(w0, v0)); den = __dadd_rn(den, w0); }
            if (lb && isfinite(v1)) { num = __dadd_rn(num, __dmul_rn(w1, v1)); den = __dadd_rn(den, w1); }
            if (lc && isfinite(v2)) { num = __dadd_rn(num, __dmul_rn(w2, v2)); den = __dadd_rn(den, w2); }
            if (ld && isfinite(v3)) { num = __dadd_rn(num, __dmul_rn(w3, v3)); den = __dadd_rn(den, w3); }
            // 4. no weight kept: the cell value
            const float r = den > 0.0 ? __double2float_rn(__ddiv_rn(num, den)) : sp_ld(Ff, c);
            __stcs(out + f * nP + p, sp_fill(r));
        }
    }
}

template <int MODE>
static cudaError_t launch_sample_mode(long long nP, int Nj, int Ni, const int2* cell, const int8_t* mask, const pt* yx,
                                      const pt* T, const int8_t* tmask, const float* F, long long stride, int nF,
                                      float* out, cudaStream_t st)
{
    // one wave of resident blocks, grid-strided
    cudaError_t e;
    int dev = 0, nsm = 0, per_sm = 0;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess ||
        (e = cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess ||
        (e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_sample<MODE>, SP_BLOCK, 0)) != cudaSuccess)
        return e;
    const long long tiles = (nP + SP_BLOCK - 1) / SP_BLOCK, wave = (long long)nsm * (per_sm < 1 ? 1 : per_sm);
    const int grid = (int)(tiles < wave ? tiles : wave);
    k_sample<MODE><<<grid, SP_BLOCK, 0, st>>>(nP, Nj, Ni, cell, mask, yx, T, tmask, F, stride, nF, out);
    return cudaGetLastError();
}

cudaError_t launch_sample(long long nP, int Nj, int Ni, const int2* cell, const int8_t* mask, const pt* yx,
                          const pt* T, const int8_t* tmask, const float* F, long long stride, int nF, int interp,
                          float* out, cudaStream_t st)
{
    if (nP < 1) return cudaSuccess;
    return interp == 0 ? launch_sample_mode<0>(nP, Nj, Ni, cell, mask, yx, T, tmask, F, stride, nF, out, st)
                       : launch_sample_mode<1>(nP, Nj, Ni, cell, mask, yx, T, tmask, F, stride, nF, out, st);
}

}  // namespace st
