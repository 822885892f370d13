// st_deform.cu -- strain rates of buoy triangles between two trajectory rows (RGPS-style sea-ice
// deformation: divergence, shear, vorticity), one thread per triangle.
//
// Definitions (DESIGN.md section 10, oracle/deform_ref.py): mid-time positions X = (x0+x1)/2, Y = (y0+y1)/2 and
// velocities U = (x1-x0)/dt, V = (y1-y0)/dt of the three vertices; the velocity gradient is the line integral
// over the three directed edges i -> i+1 (Green's theorem, Lindsay & Stern 2003):
//   2A = sum X_i Y_{i+1} - X_{i+1} Y_i,   ux = sum (U_{i+1}+U_i)(Y_{i+1}-Y_i) / 2A,   uy = -sum (U_{i+1}+U_i)(X_{i+1}-X_i) / 2A
// (vx, vy the same with V).  Every sum is spelled left to right in the oracle's order with __d*_rn, so the
// outputs are bit-identical to it.
//
// Traffic: 12 B of indices and 24 B of outputs per triangle, streamed (ld/st.global.cs, whole sectors: a block
// stages its 256 index triples through shared memory with 16-byte loads); positions and masks are gathered
// through the read-only path.  The caller sorts the triangles by their smallest vertex once, so that a warp's
// gathers stay within a few lines of a cell-major cloud.
#include "st_deform.cuh"

namespace st {

constexpr int DEF_BLOCK = 256;

// out: six (nT) f4 planes [divergence | shear | vorticity | area | y_ctr | x_ctr]
__global__ void __launch_bounds__(DEF_BLOCK) k_deform(long long nT, const int* __restrict__ tri,
                                                      const pt* __restrict__ yx0, const int8_t* __restrict__ m0,
                                                      const pt* __restrict__ yx1, const int8_t* __restrict__ m1,
                                                      double dt, float* __restrict__ out)
{
    __shared__ int4 s_tri[DEF_BLOCK * 3 / 4];
    const long long t0 = (long long)blockIdx.x * DEF_BLOCK;
    const long long t = t0 + threadIdx.x;
    if (t0 + DEF_BLOCK <= nT) {
        if (threadIdx.x < DEF_BLOCK * 3 / 4)
            s_tri[threadIdx.x] = __ldcs(reinterpret_cast<const int4*>(tri + 3 * t0) + threadIdx.x);
    } else {                                                      // the last, partial block
        int* s = reinterpret_cast<int*>(s_tri);
        for (int k = threadIdx.x; k < 3 * (nT - t0); k += DEF_BLOCK) s[k] = __ldcs(tri + 3 * t0 + k);
    }
    __syncthreads();
    if (t >= nT) return;
    const int* s = reinterpret_cast<const int*>(s_tri) + 3 * threadIdx.x;      // stride 3 words: no bank conflict
    const int i0 = s[0], i1 = s[1], i2 = s[2];

    // all twelve gathers are issued together (one memory round trip), masks and positions alike
    const int8_t k00 = __ldg(m0 + i0), k01 = __ldg(m0 + i1), k02 = __ldg(m0 + i2);
    const int8_t k10 = __ldg(m1 + i0), k11 = __ldg(m1 + i1), k12 = __ldg(m1 + i2);
    const pt a0 = ld_ro_pt(yx0, i0), a1 = ld_ro_pt(yx0, i1), a2 = ld_ro_pt(yx0, i2);
    const pt b0 = ld_ro_pt(yx1, i0), b1 = ld_ro_pt(yx1, i1), b2 = ld_ro_pt(yx1, i2);
    float r[6];
    bool ok = k00 != 0 && k01 != 0 && k02 != 0 && k10 != 0 && k11 != 0 && k12 != 0;
    if (ok) {
        const double X0 = __dmul_rn(0.5, __dadd_rn(a0.x, b0.x)), Y0 = __dmul_rn(0.5, __dadd_rn(a0.y, b0.y));
        const double X1 = __dmul_rn(0.5, __dadd_rn(a1.x, b1.x)), Y1 = __dmul_rn(0.5, __dadd_rn(a1.y, b1.y));
        const double X2 = __dmul_rn(0.5, __dadd_rn(a2.x, b2.x)), Y2 = __dmul_rn(0.5, __dadd_rn(a2.y, b2.y));
        const double U0 = __ddiv_rn(__dsub_rn(b0.x, a0.x), dt), V0 = __ddiv_rn(__dsub_rn(b0.y, a0.y), dt);
        const double U1 = __ddiv_rn(__dsub_rn(b1.x, a1.x), dt), V1 = __ddiv_rn(__dsub_rn(b1.y, a1.y), dt);
        const double U2 = __ddiv_rn(__dsub_rn(b2.x, a2.x), dt), V2 = __ddiv_rn(__dsub_rn(b2.y, a2.y), dt);
        const double A2 = twice_area(X0, X1, X2, Y0, Y1, Y2);
        const double area = __dmul_rn(0.5, A2);
        // valid: anticlockwise at both ends and at mid-time
        ok = twice_area(a0.x, a1.x, a2.x, a0.y, a1.y, a2.y) > 0.0 &&
             twice_area(b0.x, b1.x, b2.x, b0.y, b1.y, b2.y) > 0.0 && area > 0.0;
        if (ok) {
            const double ux = __ddiv_rn(edge_sum(U0, U1, U2, Y0, Y1, Y2), A2);
            const double uy = -__ddiv_rn(edge_sum(U0, U1, U2, X0, X1, X2), A2);
            const double vx = __ddiv_rn(edge_sum(V0, V1, V2, Y0, Y1, Y2), A2);
            const double vy = -__ddiv_rn(edge_sum(V0, V1, V2, X0, X1, X2), A2);
            const double d = __dsub_rn(ux, vy), e = __dadd_rn(uy, vx);
            r[0] = __double2float_rn(__dadd_rn(ux, vy));
            r[1] = __double2float_rn(__dsqrt_rn(__dadd_rn(__dmul_rn(d, d), __dmul_rn(e, e))));
            r[2] = __double2float_rn(__dsub_rn(vx, uy));
            r[3] = __double2float_rn(area);
            r[4] = __double2float_rn(__ddiv_rn(__dadd_rn(__dadd_rn(Y0, Y1), Y2), 3.0));
            r[5] = __double2float_rn(__ddiv_rn(__dadd_rn(__dadd_rn(X0, X1), X2), 3.0));
        }
    }
    if (!ok) {
#pragma unroll
        for (int j = 0; j < 6; ++j) r[j] = (float)ST_FILL;
    }
#pragma unroll
    for (int j = 0; j < 6; ++j) __stcs(out + j * nT + t, r[j]);
}

cudaError_t launch_deform(long long nT, const int32_t* tri, const pt* yx0, const int8_t* m0, const pt* yx1,
                          const int8_t* m1, double dt, float* out, cudaStream_t st)
{
    if (nT > 0)
        k_deform<<<(unsigned)((nT + DEF_BLOCK - 1) / DEF_BLOCK), DEF_BLOCK, 0, st>>>(nT, tri, yx0, m0, yx1, m1, dt, out);
    return cudaGetLastError();
}

}  // namespace st
