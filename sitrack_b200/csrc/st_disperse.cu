// st_disperse.cu -- two-particle (pair) dispersion of buoys over time lags, and per-(lag, class) statistics of it,
// reduced on the device (Rampal et al. 2008; Girard et al. 2009).
//
// Definitions (DESIGN.md section 13, oracle/dispersion_ref.py).  Per pair (a, b) and (origin row, closing row) pair,
// valid when both buoys have mask != 0 in both rows; in f8, in this order:
//   dy0 = y_a - y_b, dx0 = x_a - x_b, r0 = sqrt(dy0*dy0 + dx0*dx0)   (origin row; dy1, dx1, r1 at the closing row)
//   dr = r1 - r0,  dD2 = (dy1-dy0)*(dy1-dy0) + (dx1-dx0)*(dx1-dx0),  s = |dr| / (r0 * tau),  tau = lag * dt_days
// class = bin_right(r_edges, r0), stretch bin = bin_right(bins, s).  Statistics per (lag, class): counts of s per bin
// (shared-memory int counters, then integer atomics: exact) and the sums of r0, dr, dr^2, dD2 (per-warp butterflies by
// class, warps added in order into per-block accumulators, block partials summed in a fixed order by k_disp_final).
// The launch grid depends on nQ only, and each origin row is reduced on its own, so the sums are bit-identical run
// to run and between one fused call over several origins and one call per origin.
//
// Kernels, all on the caller's stream: k_disperse (one thread per pair, grid-strided over tiles of DS_BLOCK pairs;
// the closing row's gathers once per pair, then each active origin's gathers issued together), k_disp_final.
#include "st_deform.cuh"

namespace st {

constexpr int DS_BLOCK = 256;
constexpr int DS_WARPS = DS_BLOCK / 32;
constexpr int DS_GRID = 1184;          // fixed (not the SM count): block partials, hence their sums, are the same on
                                       // every device

int disp_grid(long long nQ)
{
    const long long g = (nQ + DS_BLOCK - 1) / DS_BLOCK;
    return (int)(g < 1 ? 1 : g > DS_GRID ? DS_GRID : g);
}

// shared memory: class edges (ncedge f8), bins (nedge f8), per-block sums acc[nact][C][4] f8, warp partials
// wp[2][DS_WARPS][C][4] f8 (two so that one barrier per origin separates their writes and reads), then the counters
// cnt[nact][C][nbin] int
size_t disp_smem(int nact, int ncedge, int nedge)
{
    const size_t C = (size_t)ncedge + 1, nbin = (size_t)nedge + 1;
    return ((size_t)ncedge + nedge + (size_t)nact * C * 4 + 2 * DS_WARPS * C * 4) * sizeof(double) +
           (size_t)nact * C * nbin * sizeof(int);
}

__global__ void __launch_bounds__(DS_BLOCK) k_disperse(DispOrigins og, long long nQ, const int2* __restrict__ pairs,
                                                       const pt* __restrict__ yx1, const int8_t* __restrict__ m1,
                                                       double dt, int ncedge, const double* __restrict__ r_edges,
                                                       int nedge, const double* __restrict__ bins,
                                                       double* __restrict__ part, unsigned long long* __restrict__ hist,
                                                       double* __restrict__ out)
{
    extern __shared__ double s_dyn[];
    const int C = ncedge + 1, nbin = nedge + 1, nact = og.nact, C4 = 4 * C;
    double* ce = s_dyn;
    double* be = ce + ncedge;
    double* acc = be + nedge;
    double* wp = acc + nact * C4;
    int* cnt = reinterpret_cast<int*>(wp + 2 * DS_WARPS * C4);
    for (int k = threadIdx.x; k < ncedge; k += DS_BLOCK) ce[k] = r_edges[k];
    for (int k = threadIdx.x; k < nedge; k += DS_BLOCK) be[k] = bins[k];
    for (int k = threadIdx.x; k < nact * C4; k += DS_BLOCK) acc[k] = 0.0;
    for (int k = threadIdx.x; k < nact * C * nbin; k += DS_BLOCK) cnt[k] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int par = 0;
    for (long long base = (long long)blockIdx.x * DS_BLOCK; base < nQ; base += (long long)gridDim.x * DS_BLOCK) {
        const long long i = base + threadIdx.x;
        const bool in = i < nQ;
        int a = 0, b = 0;
        if (in) { const int2 q = __ldcs(pairs + i); a = q.x; b = q.y; }
        // the closing row: once per pair
        int8_t k1a = 0, k1b = 0;
        pt p1a = {0.0, 0.0}, p1b = {0.0, 0.0};
        if (in) { k1a = __ldg(m1 + a); k1b = __ldg(m1 + b); p1a = ld_ro_pt(yx1, a); p1b = ld_ro_pt(yx1, b); }
        const double dy1 = __dsub_rn(p1a.y, p1b.y), dx1 = __dsub_rn(p1a.x, p1b.x);
        const double r1 = __dsqrt_rn(__dadd_rn(__dmul_rn(dy1, dy1), __dmul_rn(dx1, dx1)));
        for (int o = 0; o < nact; ++o) {
            // the origin's four gathers, issued together
            int8_t k0a = 0, k0b = 0;
            pt p0a = {0.0, 0.0}, p0b = {0.0, 0.0};
            if (in) {
                k0a = __ldg(og.m[o] + a); k0b = __ldg(og.m[o] + b);
                p0a = ld_ro_pt(og.yx[o], a); p0b = ld_ro_pt(og.yx[o], b);
            }
            const bool ok = in && k0a != 0 && k0b != 0 && k1a != 0 && k1b != 0;
            const double dy0 = __dsub_rn(p0a.y, p0b.y), dx0 = __dsub_rn(p0a.x, p0b.x);
            const double r0 = __dsqrt_rn(__dadd_rn(__dmul_rn(dy0, dy0), __dmul_rn(dx0, dx0)));
            const double dr = __dsub_rn(r1, r0);
            const double ey = __dsub_rn(dy1, dy0), ex = __dsub_rn(dx1, dx0);
            const double dD2 = __dadd_rn(__dmul_rn(ey, ey), __dmul_rn(ex, ex));
            int c = -1;
            if (ok) {
                const double tau = __dmul_rn((double)og.lag[o], dt);
                const double s = __ddiv_rn(fabs(dr), __dmul_rn(r0, tau));
                c = bin_right(ce, ncedge, r0);
                atomicAdd(cnt + (o * C + c) * nbin + bin_right(be, nedge, s), 1);
            }
            if (out && in) {
                const double F = ST_FILL;
                out[i] = ok ? r0 : F;
                out[nQ + i] = ok ? r1 : F;
                out[2 * nQ + i] = ok ? dr : F;
                out[3 * nQ + i] = ok ? dD2 : F;
            }
            // warp partials by class: one xor butterfly per class present in the warp
            double* w = wp + (par * DS_WARPS + warp) * C4;
            for (int k = lane; k < C4; k += 32) w[k] = 0.0;
            __syncwarp();
            const double v[4] = {r0, dr, __dmul_rn(dr, dr), dD2};
            unsigned rem = __ballot_sync(0xffffffffu, c >= 0);
            while (rem) {
                const int cc = __shfl_sync(0xffffffffu, c, __ffs(rem) - 1);
                const bool mine = c == cc;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    double x = mine ? v[q] : 0.0;
#pragma unroll
                    for (int sh = 16; sh > 0; sh >>= 1) x = __dadd_rn(x, __shfl_xor_sync(0xffffffffu, x, sh));
                    if (lane == 0) w[4 * cc + q] = x;
                }
                rem &= ~__ballot_sync(0xffffffffu, mine);
            }
            __syncthreads();
            // the warps' partials into the block's sums, in warp order
            const double* wb = wp + par * DS_WARPS * C4;
            for (int k = threadIdx.x; k < C4; k += DS_BLOCK) {
                double s = acc[o * C4 + k];
                for (int ww = 0; ww < DS_WARPS; ++ww) s = __dadd_rn(s, wb[ww * C4 + k]);
                acc[o * C4 + k] = s;
            }
            par ^= 1;
        }
    }
    __syncthreads();
    for (int k = threadIdx.x; k < nact * C4; k += DS_BLOCK)
        part[((long long)blockIdx.x * nact + k / C4) * C4 + k % C4] = acc[k];
    for (int k = threadIdx.x; k < nact * C * nbin; k += DS_BLOCK)
        if (cnt[k]) {
            const int o = k / (C * nbin);
            atomicAdd(hist + (long long)(og.lag[o] - 1) * C * nbin + k % (C * nbin), (unsigned long long)cnt[k]);
        }
}

// One block per (active origin, class): the blocks' partials summed in a fixed order -> sums[lag-1][class][4].
__global__ void __launch_bounds__(DS_BLOCK) k_disp_final(DispOrigins og, int C, int nblk, const double* __restrict__ part,
                                                         double* __restrict__ sums)
{
    __shared__ double s_r[4][DS_BLOCK];
    const int o = blockIdx.x / C, c = blockIdx.x % C, nact = og.nact;
    double a[4] = {0.0, 0.0, 0.0, 0.0};
    for (int b = threadIdx.x; b < nblk; b += DS_BLOCK) {
        const double* p = part + (((long long)b * nact + o) * C + c) * 4;
#pragma unroll
        for (int q = 0; q < 4; ++q) a[q] = __dadd_rn(a[q], p[q]);
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) s_r[q][threadIdx.x] = a[q];
    __syncthreads();
    for (int w = DS_BLOCK / 2; w > 0; w >>= 1) {
        if (threadIdx.x < w) {
#pragma unroll
            for (int q = 0; q < 4; ++q) s_r[q][threadIdx.x] = __dadd_rn(s_r[q][threadIdx.x], s_r[q][threadIdx.x + w]);
        }
        __syncthreads();
    }
    if (threadIdx.x < 4) sums[((long long)(og.lag[o] - 1) * C + c) * 4 + threadIdx.x] = s_r[threadIdx.x][0];
}

long long disp_scratch_bytes(long long nQ, int lags, int ncedge)
{
    return (long long)disp_grid(nQ) * lags * (ncedge + 1) * 4 * (long long)sizeof(double);
}

cudaError_t launch_dispersion(const DispOrigins& og, long long nQ, const int32_t* pairs, const pt* yx1,
                              const int8_t* m1, double dt, int lags, int ncedge, const double* r_edges, int nedge,
                              const double* bins, void* scratch, int64_t* hist, double* sums, double* out,
                              cudaStream_t st)
{
    const int C = ncedge + 1, nbin = nedge + 1, grid = disp_grid(nQ);
    cudaError_t e = cudaMemsetAsync(hist, 0, sizeof(int64_t) * (size_t)lags * C * nbin, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(sums, 0, sizeof(double) * (size_t)lags * C * 4, st);
    if (e != cudaSuccess) return e;
    const size_t smem = disp_smem(og.nact, ncedge, nedge);
    if (smem > 48 * 1024 &&
        (e = cudaFuncSetAttribute(k_disperse, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess)
        return e;
    k_disperse<<<grid, DS_BLOCK, smem, st>>>(og, nQ, reinterpret_cast<const int2*>(pairs), yx1, m1, dt, ncedge, r_edges,
                                              nedge, bins, static_cast<double*>(scratch),
                                              reinterpret_cast<unsigned long long*>(hist), out);
    k_disp_final<<<og.nact * C, DS_BLOCK, 0, st>>>(og, C, grid, static_cast<const double*>(scratch), sums);
    return cudaGetLastError();
}

}  // namespace st
