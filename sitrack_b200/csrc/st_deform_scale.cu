// st_deform_scale.cu -- buoy-triangle deformation coarse-grained over a hierarchy of material boxes, and per-scale
// statistics of it (spatial scaling of sea-ice deformation, Marsan et al. 2004), reduced on the device.
//
// Definitions (DESIGN.md section 11, oracle/deform_scale_ref.py).  The triangles come sorted by the Morton code of
// their level-1 box, so every box of every level is a contiguous range of them.  Per valid triangle, in f8 (invalid
// triangles contribute +0.0):
//   a2 = 2A,  Nux = edge_sum(U,Y),  Nuy = -edge_sum(U,X),  Nvx = edge_sum(V,Y),  Nvy = -edge_sum(V,X),  NY = a2 Yc,  NX = a2 Xc
// and a box's rates are its sums over a2's sum (Green's theorem: interior edges cancel).  Summation order, fixed
// so that the oracle reproduces it bit for bit (no floating-point atomics):
//   level 1: one warp per box; lane l sums the triangles l, l+32, ... left to right from +0.0, then an xor
//            butterfly with offsets 16, 8, 4, 2, 1 (p = p + p[l^o]);
//   level s+1: ((c0 + c1) + c2) + c3 over the children that exist, in Morton order, from +0.0.
// Statistics: per scale (0 = the triangles with their own k_deform rates) histograms of eps_tot, |div| and shear
// through shared-memory int counters and integer atomics (exact), and moment sums through per-block partials and
// one fixed-order reduction (bit-identical run to run; the grid shape depends on the hierarchy only).
//
// Kernels, all on the caller's stream: k_scale_l1 (level-1 box sums + scale-0 statistics), k_scale_parent (one
// launch per coarser level), k_scale_stats (box outputs, validity, statistics of every level), k_scale_final.
// DEV = false: box counts from the ScalePlan (material boxes, built on the host).  DEV = true: box counts from device
// memory (dnbox, Eulerian boxes segmented on the device, st_deform_grid.cu); the ScalePlan then holds upper bounds of
// them, so launch grids, box record layout and moment partials depend on the bounds only.
#include "st_deform.cuh"

namespace st {

constexpr int SC_BLOCK = 256;
constexpr int SC_WARPS = SC_BLOCK / 32;
constexpr int SC_GRID = 1184;          // fixed (not the SM count): the moment partials, hence their sums, are the
                                       // same on every device
constexpr int SC_BOX = 8;              // doubles per box record: a2, ux, uy, vx, vy, NY, NX sums + padding

// rates of a sum record -> eps_tot, |div|, shear (the statistics' three variables), f8 as the oracle
struct Rates { double div, shear, vort, tot; };
__device__ __forceinline__ Rates rates_of(double ux, double uy, double vx, double vy)
{
    Rates r;
    const double D = __dadd_rn(ux, vy), d = __dsub_rn(ux, vy), e = __dadd_rn(uy, vx);
    r.div = D;
    r.shear = __dsqrt_rn(__dadd_rn(__dmul_rn(d, d), __dmul_rn(e, e)));
    r.vort = __dsub_rn(vx, uy);
    r.tot = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(D, D), __dmul_rn(d, d)), __dmul_rn(e, e)));
    return r;
}

struct StatAcc {
    double m[4];                       // sums of L_eff, eps_tot, eps_tot^2, eps_tot^3
    __device__ void zero() { m[0] = m[1] = m[2] = m[3] = 0.0; }
    __device__ void add(double Leff, double tot)
    {
        const double t2 = __dmul_rn(tot, tot);
        m[0] = __dadd_rn(m[0], Leff); m[1] = __dadd_rn(m[1], tot);
        m[2] = __dadd_rn(m[2], t2);   m[3] = __dadd_rn(m[3], __dmul_rn(t2, tot));
    }
};

__device__ __forceinline__ void count(int* cnt, int nbin, const double* e, int ne, const Rates& r)
{
    atomicAdd(cnt + bin_right(e, ne, r.tot), 1);
    atomicAdd(cnt + nbin + bin_right(e, ne, fabs(r.div)), 1);
    atomicAdd(cnt + 2 * nbin + bin_right(e, ne, r.shear), 1);
}

// shared memory: edges (ne f8), then 3 * nbin int counters
__device__ __forceinline__ void stats_smem_init(const double* __restrict__ edges, int ne, int nbin, double*& e, int*& cnt)
{
    extern __shared__ double s_dyn[];
    e = s_dyn;
    cnt = reinterpret_cast<int*>(s_dyn + ne);
    for (int k = threadIdx.x; k < ne; k += SC_BLOCK) e[k] = edges[k];
    for (int k = threadIdx.x; k < 3 * nbin; k += SC_BLOCK) cnt[k] = 0;
    __syncthreads();
}

// the block's moment partial (fixed order: warp butterfly, then warp 0 over the warps) and its histogram counts
__device__ __forceinline__ void stats_flush(StatAcc a, int blk, int scale, int nbin, const int* cnt,
                                            double* __restrict__ part, unsigned long long* __restrict__ hist)
{
    __shared__ double s_m[4][SC_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) a.m[q] = __dadd_rn(a.m[q], __shfl_xor_sync(0xffffffffu, a.m[q], o));
        if (lane == 0) s_m[q][warp] = a.m[q];
    }
    __syncthreads();
    if (threadIdx.x < 4) {
        double s = 0.0;
        for (int w = 0; w < SC_WARPS; ++w) s = __dadd_rn(s, s_m[threadIdx.x][w]);
        part[4 * (long long)blk + threadIdx.x] = s;
    }
    unsigned long long* h = hist + (long long)scale * 3 * nbin;
    for (int k = threadIdx.x; k < 3 * nbin; k += SC_BLOCK)
        if (cnt[k]) atomicAdd(h + k, (unsigned long long)cnt[k]);
}

// Level-1 box sums (one warp per box, boxes grid-strided over the warps) and the scale-0 statistics.
template <bool DEV>
__global__ void __launch_bounds__(SC_BLOCK) k_scale_l1(ScalePlan p, const long long* __restrict__ tri_off,
                                                       const int* __restrict__ tri,
                                                       const pt* __restrict__ yx0, const int8_t* __restrict__ m0,
                                                       const pt* __restrict__ yx1, const int8_t* __restrict__ m1,
                                                       double dt, const double* __restrict__ edges,
                                                       double* __restrict__ box, double* __restrict__ part,
                                                       unsigned long long* __restrict__ hist,
                                                       const long long* __restrict__ dnbox)
{
    double* e; int* cnt;
    stats_smem_init(edges, p.nedge, p.nbin, e, cnt);
    const int lane = threadIdx.x & 31;
    StatAcc st; st.zero();
    const long long nbox = DEV ? dnbox[0] : p.nbox[0];
    for (long long b = (long long)blockIdx.x * SC_WARPS + (threadIdx.x >> 5); b < nbox; b += (long long)gridDim.x * SC_WARPS) {
        const long long t1 = tri_off[b + 1];
        double acc[7] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        for (long long t = tri_off[b] + lane; t < t1; t += 32) {
            const int i0 = __ldcs(tri + 3 * t), i1 = __ldcs(tri + 3 * t + 1), i2 = __ldcs(tri + 3 * t + 2);
            // all twelve gathers are issued together, as in k_deform
            const int8_t k00 = __ldg(m0 + i0), k01 = __ldg(m0 + i1), k02 = __ldg(m0 + i2);
            const int8_t k10 = __ldg(m1 + i0), k11 = __ldg(m1 + i1), k12 = __ldg(m1 + i2);
            const pt a0 = ld_ro_pt(yx0, i0), a1 = ld_ro_pt(yx0, i1), a2 = ld_ro_pt(yx0, i2);
            const pt b0 = ld_ro_pt(yx1, i0), b1 = ld_ro_pt(yx1, i1), b2 = ld_ro_pt(yx1, i2);
            // an invalid triangle adds nothing: adding +0.0 to an accumulator that starts at +0.0 is the identity
            if (k00 != 0 && k01 != 0 && k02 != 0 && k10 != 0 && k11 != 0 && k12 != 0) {
                const double X0 = __dmul_rn(0.5, __dadd_rn(a0.x, b0.x)), Y0 = __dmul_rn(0.5, __dadd_rn(a0.y, b0.y));
                const double X1 = __dmul_rn(0.5, __dadd_rn(a1.x, b1.x)), Y1 = __dmul_rn(0.5, __dadd_rn(a1.y, b1.y));
                const double X2 = __dmul_rn(0.5, __dadd_rn(a2.x, b2.x)), Y2 = __dmul_rn(0.5, __dadd_rn(a2.y, b2.y));
                const double A2 = twice_area(X0, X1, X2, Y0, Y1, Y2);
                const double area = __dmul_rn(0.5, A2);
                if (twice_area(a0.x, a1.x, a2.x, a0.y, a1.y, a2.y) > 0.0 &&
                    twice_area(b0.x, b1.x, b2.x, b0.y, b1.y, b2.y) > 0.0 && area > 0.0) {
                    const double U0 = __ddiv_rn(__dsub_rn(b0.x, a0.x), dt), V0 = __ddiv_rn(__dsub_rn(b0.y, a0.y), dt);
                    const double U1 = __ddiv_rn(__dsub_rn(b1.x, a1.x), dt), V1 = __ddiv_rn(__dsub_rn(b1.y, a1.y), dt);
                    const double U2 = __ddiv_rn(__dsub_rn(b2.x, a2.x), dt), V2 = __ddiv_rn(__dsub_rn(b2.y, a2.y), dt);
                    const double Nux = edge_sum(U0, U1, U2, Y0, Y1, Y2), Nuy = -edge_sum(U0, U1, U2, X0, X1, X2);
                    const double Nvx = edge_sum(V0, V1, V2, Y0, Y1, Y2), Nvy = -edge_sum(V0, V1, V2, X0, X1, X2);
                    acc[0] = __dadd_rn(acc[0], A2);
                    acc[1] = __dadd_rn(acc[1], Nux);
                    acc[2] = __dadd_rn(acc[2], Nuy);
                    acc[3] = __dadd_rn(acc[3], Nvx);
                    acc[4] = __dadd_rn(acc[4], Nvy);
                    acc[5] = __dadd_rn(acc[5], __dmul_rn(A2, __ddiv_rn(__dadd_rn(__dadd_rn(Y0, Y1), Y2), 3.0)));
                    acc[6] = __dadd_rn(acc[6], __dmul_rn(A2, __ddiv_rn(__dadd_rn(__dadd_rn(X0, X1), X2), 3.0)));
                    // scale 0: the triangle's own rates, exactly k_deform's f8 values
                    const Rates r = rates_of(__ddiv_rn(Nux, A2), __ddiv_rn(Nuy, A2), __ddiv_rn(Nvx, A2), __ddiv_rn(Nvy, A2));
                    st.add(__dsqrt_rn(area), r.tot);
                    count(cnt, p.nbin, e, p.nedge, r);
                }
            }
        }
        double w = 0.0;
#pragma unroll
        for (int k = 0; k < 7; ++k) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) acc[k] = __dadd_rn(acc[k], __shfl_xor_sync(0xffffffffu, acc[k], o));
            if (lane == k) w = acc[k];
        }
        if (lane < 7) box[SC_BOX * b + lane] = w;
    }
    __syncthreads();
    stats_flush(st, p.blk0[0] + blockIdx.x, 0, p.nbin, cnt, part, hist);
}

// Level s+1 from level s: thread per parent box, ((c0 + c1) + c2) + c3 over its children in Morton order.
template <bool DEV>
__global__ void __launch_bounds__(SC_BLOCK) k_scale_parent(long long n, const long long* __restrict__ coff,
                                                           const double* __restrict__ child, double* __restrict__ parent,
                                                           const long long* __restrict__ dn)
{
    const long long i = (long long)blockIdx.x * SC_BLOCK + threadIdx.x;
    if (i >= (DEV ? *dn : n)) return;
    double acc[7] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    const long long c1 = coff[i + 1];
    for (long long c = coff[i]; c < c1; ++c) {
#pragma unroll
        for (int k = 0; k < 7; ++k) acc[k] = __dadd_rn(acc[k], child[SC_BOX * c + k]);
    }
#pragma unroll
    for (int k = 0; k < 7; ++k) parent[SC_BOX * i + k] = acc[k];
}

// Box outputs, validity and statistics of every level >= 1; the blocks [blk0[s], blk0[s+1]) serve scale s.
// out (optional): seven f4 planes over all boxes [divergence | shear | vorticity | total | L_eff | y_ctr | x_ctr].
template <bool DEV>
__global__ void __launch_bounds__(SC_BLOCK) k_scale_stats(ScalePlan p, const double* __restrict__ box,
                                                          const double* __restrict__ edges, double* __restrict__ part,
                                                          unsigned long long* __restrict__ hist, float* __restrict__ out,
                                                          long long nbox_all, const long long* __restrict__ dnbox)
{
    double* e; int* cnt;
    stats_smem_init(edges, p.nedge, p.nbin, e, cnt);
    const int gb = p.blk0[1] + blockIdx.x;
    int s = 1;
    while (s < p.levels && gb >= p.blk0[s + 1]) ++s;
    const int lv = s - 1;
    const long long nb = DEV ? dnbox[lv] : p.nbox[lv], first = p.box0[lv];
    const long long stride = (long long)(p.blk0[s + 1] - p.blk0[s]) * SC_BLOCK;
    const double thr = p.min_area[lv];
    StatAcc st; st.zero();
    for (long long i = (long long)(gb - p.blk0[s]) * SC_BLOCK + threadIdx.x; i < nb; i += stride) {
        const double* q = box + SC_BOX * (first + i);
        const double S = q[0];
        const double ux = __ddiv_rn(q[1], S), uy = __ddiv_rn(q[2], S), vx = __ddiv_rn(q[3], S), vy = __ddiv_rn(q[4], S);
        const double area = __dmul_rn(0.5, S);
        const Rates r = rates_of(ux, uy, vx, vy);
        const double Leff = __dsqrt_rn(area);
        const bool ok = area >= thr;
        if (ok) {
            st.add(Leff, r.tot);
            count(cnt, p.nbin, e, p.nedge, r);
        }
        if (out) {
            const float F = (float)ST_FILL;
            const long long j = first + i;
            out[j] = ok ? __double2float_rn(r.div) : F;
            out[nbox_all + j] = ok ? __double2float_rn(r.shear) : F;
            out[2 * nbox_all + j] = ok ? __double2float_rn(r.vort) : F;
            out[3 * nbox_all + j] = ok ? __double2float_rn(r.tot) : F;
            out[4 * nbox_all + j] = ok ? __double2float_rn(Leff) : F;
            out[5 * nbox_all + j] = ok ? __double2float_rn(__ddiv_rn(q[5], S)) : F;
            out[6 * nbox_all + j] = ok ? __double2float_rn(__ddiv_rn(q[6], S)) : F;
        }
    }
    __syncthreads();
    stats_flush(st, gb, s, p.nbin, cnt, part, hist);
}

// One block per scale: the scale's block partials summed in a fixed order -> moments (S,4).
__global__ void __launch_bounds__(SC_BLOCK) k_scale_final(ScalePlan p, const double* __restrict__ part,
                                                          double* __restrict__ mom)
{
    __shared__ double s_r[4][SC_BLOCK];
    const int s = blockIdx.x;
    double a[4] = {0.0, 0.0, 0.0, 0.0};
    for (int i = p.blk0[s] + threadIdx.x; i < p.blk0[s + 1]; i += SC_BLOCK) {
#pragma unroll
        for (int q = 0; q < 4; ++q) a[q] = __dadd_rn(a[q], part[4 * (long long)i + q]);
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) s_r[q][threadIdx.x] = a[q];
    __syncthreads();
    for (int w = SC_BLOCK / 2; w > 0; w >>= 1) {
        if (threadIdx.x < w) {
#pragma unroll
            for (int q = 0; q < 4; ++q) s_r[q][threadIdx.x] = __dadd_rn(s_r[q][threadIdx.x], s_r[q][threadIdx.x + w]);
        }
        __syncthreads();
    }
    if (threadIdx.x < 4) mom[4 * s + threadIdx.x] = s_r[threadIdx.x][0];
}

static int grid_for(long long items, int per_block)
{
    const long long g = (items + per_block - 1) / per_block;
    return (int)(g < 1 ? 1 : g > SC_GRID ? SC_GRID : g);
}

long long scale_plan(int levels, const long long* nbox, const double* min_area, int nedge, ScalePlan* p)
{
    ScalePlan q = {};
    q.levels = levels;
    q.nedge = nedge;
    q.nbin = nedge + 1;
    long long first = 0, coff = 0;
    q.blk0[0] = 0;
    q.blk0[1] = grid_for(nbox[0], SC_WARPS);
    for (int l = 0; l < levels; ++l) {
        q.nbox[l] = nbox[l];
        q.box0[l] = first;
        q.child0[l] = l ? coff : 0;
        q.min_area[l] = min_area[l];
        first += nbox[l];
        if (l) coff += nbox[l] + 1;
        q.blk0[l + 2] = q.blk0[l + 1] + grid_for(nbox[l], SC_BLOCK);
    }
    q.nbox_all = first;
    *p = q;
    return (SC_BOX * first + 4LL * q.blk0[levels + 1]) * (long long)sizeof(double);
}

size_t scale_smem(const ScalePlan& p) { return (size_t)p.nedge * sizeof(double) + (size_t)3 * p.nbin * sizeof(int); }

template <bool DEV>
static cudaError_t launch_scales(const ScalePlan& p, const int32_t* tri, const long long* tri_off,
                                 const long long* child_off, const pt* yx0, const int8_t* m0, const pt* yx1,
                                 const int8_t* m1, double dt, const double* edges, void* scratch, double* mom,
                                 int64_t* hist, float* out, const long long* dnbox, cudaStream_t st)
{
    double* box = static_cast<double*>(scratch);
    double* part = box + SC_BOX * p.nbox_all;
    unsigned long long* h = reinterpret_cast<unsigned long long*>(hist);
    const size_t smem = scale_smem(p);
    cudaError_t e = cudaMemsetAsync(hist, 0, sizeof(int64_t) * 3 * (size_t)p.nbin * (p.levels + 1), st);
    if (e != cudaSuccess) return e;
    if (smem > 48 * 1024) {
        if ((e = cudaFuncSetAttribute(k_scale_l1<DEV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess ||
            (e = cudaFuncSetAttribute(k_scale_stats<DEV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess)
            return e;
    }
    k_scale_l1<DEV><<<p.blk0[1], SC_BLOCK, smem, st>>>(p, tri_off, tri, yx0, m0, yx1, m1, dt, edges, box, part, h, dnbox);
    for (int l = 1; l < p.levels; ++l)
        k_scale_parent<DEV><<<(unsigned)((p.nbox[l] + SC_BLOCK - 1) / SC_BLOCK), SC_BLOCK, 0, st>>>(
            p.nbox[l], child_off + p.child0[l], box + SC_BOX * p.box0[l - 1], box + SC_BOX * p.box0[l],
            DEV ? dnbox + l : nullptr);
    k_scale_stats<DEV><<<p.blk0[p.levels + 1] - p.blk0[1], SC_BLOCK, smem, st>>>(p, box, edges, part, h, out,
                                                                                 p.nbox_all, dnbox);
    k_scale_final<<<p.levels + 1, SC_BLOCK, 0, st>>>(p, part, mom);
    return cudaGetLastError();
}

cudaError_t launch_deform_scales(const ScalePlan& p, const int32_t* tri, const long long* tri_off,
                                 const long long* child_off, const pt* yx0, const int8_t* m0, const pt* yx1,
                                 const int8_t* m1, double dt, const double* edges, void* scratch, double* mom,
                                 int64_t* hist, float* out, cudaStream_t st)
{
    return launch_scales<false>(p, tri, tri_off, child_off, yx0, m0, yx1, m1, dt, edges, scratch, mom, hist, out,
                                nullptr, st);
}

cudaError_t launch_deform_scales_devcount(const ScalePlan& p, const int32_t* tri, const long long* tri_off,
                                          const long long* child_off, const pt* yx0, const int8_t* m0, const pt* yx1,
                                          const int8_t* m1, double dt, const double* edges, void* scratch, double* mom,
                                          int64_t* hist, float* out, const long long* dnbox, cudaStream_t st)
{
    return launch_scales<true>(p, tri, tri_off, child_off, yx0, m0, yx1, m1, dt, edges, scratch, mom, hist, out,
                               dnbox, st);
}

}  // namespace st
