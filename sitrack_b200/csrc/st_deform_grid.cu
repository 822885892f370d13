// st_deform_grid.cu -- buoy-triangle deformation coarse-grained over the cells of a fixed Eulerian grid, with box
// membership rebuilt every window on the device, per-scale statistics and dense per-level fields.
//
// Definitions (DESIGN.md section 12, oracle/deform_grid_ref.py).  Level-1 cell (bj, bi) covers
// [oy + bj L0, oy + (bj+1) L0) x [ox + bi L0, ox + (bi+1) L0); level s has side L0 2^(s-1) and key (bj, bi) >> (s-1).
// A triangle is binned in a window when it is valid by section 10's rule and its mid-time centroid
// Yc = ((Y0+Y1)+Y2)/3 (Xc likewise) lies in the grid: q = floor((Yc - oy) / L0) with 0 <= q < nj compared in f8
// (so NaN and inf are never binned), likewise in x.  Binned triangles are sorted stably by the Morton code of their
// level-1 key (i bits even, j bits odd), ties in the caller's triangle order; each level's boxes are the runs of that
// order, and from there st_deform_scale.cu's kernels run unchanged in their DEV = true form (box counts in device
// memory, launch grids from the bounds min(nT, nj_s ni_s)), so the sums, outputs and statistics follow section 11.
//
// Stages, all on the caller's stream, no allocation, no host synchronisation:
//   k_grid_key     one thread per triangle: validity, centroid, cell, 64-bit code (sentinel 2^(2b) when not binned)
//   SortPairs      cub::DeviceRadixSort over (code, triangle index), bits [0, 2b+1), b = ceil(log2(max(nj, ni)))
//   k_grid_gather  the binned triangles' rows in sorted order, and their count
//   per level      k_grid_mark (run heads) + DeviceScan::ExclusiveSum + k_grid_heads (ranges, codes, box count)
//   the pass       k_scale_l1 / k_scale_parent / k_scale_stats / k_scale_final <DEV = true>, box planes in scratch
//   k_grid_fill + k_grid_scatter   FillValue, then each box's seven f4 outputs at its cell
#include "st_deform.cuh"
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

namespace st {

constexpr int GR_BLOCK = 256;
constexpr int GR_ALIGN = 256;

__device__ __forceinline__ unsigned long long spread2(unsigned long long v)   // bits of v (< 2^32) to even positions
{
    v = (v | (v << 16)) & 0x0000FFFF0000FFFFull;
    v = (v | (v << 8)) & 0x00FF00FF00FF00FFull;
    v = (v | (v << 4)) & 0x0F0F0F0F0F0F0F0Full;
    v = (v | (v << 2)) & 0x3333333333333333ull;
    v = (v | (v << 1)) & 0x5555555555555555ull;
    return v;
}

__device__ __forceinline__ int compact2(unsigned long long v)                  // even bits of v -> an integer
{
    v &= 0x5555555555555555ull;
    v = (v | (v >> 1)) & 0x3333333333333333ull;
    v = (v | (v >> 2)) & 0x0F0F0F0F0F0F0F0Full;
    v = (v | (v >> 4)) & 0x00FF00FF00FF00FFull;
    v = (v | (v >> 8)) & 0x0000FFFF0000FFFFull;
    v = (v | (v >> 16)) & 0x00000000FFFFFFFFull;
    return (int)v;
}

// One thread per triangle (caller's order): the sort key and value.
__global__ void __launch_bounds__(GR_BLOCK) k_grid_key(long long nT, const int* __restrict__ tri,
                                                       const pt* __restrict__ yx0, const int8_t* __restrict__ m0,
                                                       const pt* __restrict__ yx1, const int8_t* __restrict__ m1,
                                                       double oy, double ox, double L0, int nj, int ni,
                                                       unsigned long long sentinel, unsigned long long* __restrict__ kin,
                                                       int* __restrict__ vin)
{
    const long long t = (long long)blockIdx.x * GR_BLOCK + threadIdx.x;
    if (t >= nT) return;
    const int i0 = __ldcs(tri + 3 * t), i1 = __ldcs(tri + 3 * t + 1), i2 = __ldcs(tri + 3 * t + 2);
    // all twelve gathers are issued together, as in k_deform
    const int8_t k00 = __ldg(m0 + i0), k01 = __ldg(m0 + i1), k02 = __ldg(m0 + i2);
    const int8_t k10 = __ldg(m1 + i0), k11 = __ldg(m1 + i1), k12 = __ldg(m1 + i2);
    const pt a0 = ld_ro_pt(yx0, i0), a1 = ld_ro_pt(yx0, i1), a2 = ld_ro_pt(yx0, i2);
    const pt b0 = ld_ro_pt(yx1, i0), b1 = ld_ro_pt(yx1, i1), b2 = ld_ro_pt(yx1, i2);
    unsigned long long code = sentinel;
    if (k00 != 0 && k01 != 0 && k02 != 0 && k10 != 0 && k11 != 0 && k12 != 0) {
        const double X0 = __dmul_rn(0.5, __dadd_rn(a0.x, b0.x)), Y0 = __dmul_rn(0.5, __dadd_rn(a0.y, b0.y));
        const double X1 = __dmul_rn(0.5, __dadd_rn(a1.x, b1.x)), Y1 = __dmul_rn(0.5, __dadd_rn(a1.y, b1.y));
        const double X2 = __dmul_rn(0.5, __dadd_rn(a2.x, b2.x)), Y2 = __dmul_rn(0.5, __dadd_rn(a2.y, b2.y));
        const double area = __dmul_rn(0.5, twice_area(X0, X1, X2, Y0, Y1, Y2));
        if (twice_area(a0.x, a1.x, a2.x, a0.y, a1.y, a2.y) > 0.0 &&
            twice_area(b0.x, b1.x, b2.x, b0.y, b1.y, b2.y) > 0.0 && area > 0.0) {
            const double Yc = __ddiv_rn(__dadd_rn(__dadd_rn(Y0, Y1), Y2), 3.0);
            const double Xc = __ddiv_rn(__dadd_rn(__dadd_rn(X0, X1), X2), 3.0);
            const double qj = floor(__ddiv_rn(__dsub_rn(Yc, oy), L0));
            const double qi = floor(__ddiv_rn(__dsub_rn(Xc, ox), L0));
            // in f8, before any conversion: NaN fails every comparison, and no integer overflows
            if (qj >= 0.0 && qj < (double)nj && qi >= 0.0 && qi < (double)ni)
                code = (spread2((unsigned long long)qj) << 1) | spread2((unsigned long long)qi);
        }
    }
    kin[t] = code;
    vin[t] = (int)t;
}

// The binned triangles' rows in sorted order, and their count (the sentinel sorts after every code).
__global__ void __launch_bounds__(GR_BLOCK) k_grid_gather(long long nT, const unsigned long long* __restrict__ code,
                                                          const int* __restrict__ idx, const int* __restrict__ tri,
                                                          unsigned long long sentinel, int* __restrict__ tri_h,
                                                          long long* __restrict__ nbin)
{
    const long long i = (long long)blockIdx.x * GR_BLOCK + threadIdx.x;
    if (i >= nT) return;
    const bool in = code[i] != sentinel;
    if (in) {
        const long long t = idx[i];
        tri_h[3 * i] = __ldg(tri + 3 * t); tri_h[3 * i + 1] = __ldg(tri + 3 * t + 1); tri_h[3 * i + 2] = __ldg(tri + 3 * t + 2);
        if (i + 1 == nT || code[i + 1] == sentinel) *nbin = i + 1;
    } else if (i == 0) {
        *nbin = 0;
    }
}

// Run heads of the first *n items of c >> sh; 0 beyond *n (the scan runs over the bound).
__global__ void __launch_bounds__(GR_BLOCK) k_grid_mark(long long bound, const long long* __restrict__ n,
                                                        const unsigned long long* __restrict__ c, int sh,
                                                        int* __restrict__ flag)
{
    const long long i = (long long)blockIdx.x * GR_BLOCK + threadIdx.x;
    if (i >= bound) return;
    flag[i] = i < *n && (i == 0 || (c[i] >> sh) != (c[i - 1] >> sh));
}

// Box b of the run starting at item i: its range start off[b] = i, its code c[i] >> sh; the box count and the
// closing range end off[nbox] = *n.
__global__ void __launch_bounds__(GR_BLOCK) k_grid_heads(long long bound, const long long* __restrict__ n,
                                                         const unsigned long long* __restrict__ c, int sh,
                                                         const int* __restrict__ flag, const int* __restrict__ pos,
                                                         long long* __restrict__ off,
                                                         unsigned long long* __restrict__ box_code,
                                                         long long* __restrict__ nbox)
{
    const long long i = (long long)blockIdx.x * GR_BLOCK + threadIdx.x;
    if (i >= bound) return;
    const long long nn = *n;
    if (flag[i]) {
        off[pos[i]] = i;
        box_code[pos[i]] = c[i] >> sh;
    }
    if (i + 1 == nn) {
        const long long nb = (long long)pos[i] + flag[i];
        *nbox = nb;
        off[nb] = nn;
    } else if (nn == 0 && i == 0) {
        *nbox = 0;
        off[0] = 0;
    }
}

__global__ void __launch_bounds__(GR_BLOCK) k_grid_fill(long long n, float* __restrict__ f)
{
    for (long long i = (long long)blockIdx.x * GR_BLOCK + threadIdx.x; i < n; i += (long long)gridDim.x * GR_BLOCK)
        f[i] = (float)ST_FILL;
}

// One thread per box of one level: its seven f4 outputs (k_scale_stats' planes) at its cell of the dense field.
__global__ void __launch_bounds__(GR_BLOCK) k_grid_scatter(long long bound, const long long* __restrict__ nbox,
                                                           const unsigned long long* __restrict__ code,
                                                           const float* __restrict__ planes, long long plane_stride,
                                                           int ni_s, long long cells, float* __restrict__ field)
{
    const long long i = (long long)blockIdx.x * GR_BLOCK + threadIdx.x;
    if (i >= bound || i >= *nbox) return;
    const unsigned long long k = code[i];
    const long long cell = (long long)compact2(k >> 1) * ni_s + compact2(k);
#pragma unroll
    for (int j = 0; j < 7; ++j) field[j * cells + cell] = planes[j * plane_stride + i];
}

static long long up(long long b) { return (b + GR_ALIGN - 1) / GR_ALIGN * GR_ALIGN; }
static unsigned blocks(long long n) { return (unsigned)((n + GR_BLOCK - 1) / GR_BLOCK); }

const char* grid_plan(long long nT, int levels, int nj, int ni, const double* min_area, int nedge, GridPlan* g)
{
    if (nT < 1 || nT > INT32_MAX) return "nT must be in 1..2^31-1";
    if (levels < 1 || levels > SC_MAX_LEVELS) return "levels must be in 1..20";
    if (nj < 1 || nj > GR_MAX_SIDE || ni < 1 || ni > GR_MAX_SIDE) return "nj and ni must be in 1..2^20";
    if (nedge < 1 || nedge > SC_MAX_EDGES) return "nedge must be in 1..4096";
    GridPlan q = {};
    q.nT = nT; q.levels = levels; q.nj = nj; q.ni = ni;
    int b = 0;
    while ((1 << b) < (nj > ni ? nj : ni)) ++b;
    q.end_bit = 2 * b + 1;
    long long bound[SC_MAX_LEVELS], noff = 0;
    double ma[SC_MAX_LEVELS];
    q.field0[0] = 0;
    for (int l = 0; l < levels; ++l) {
        q.nj_s[l] = ((nj - 1) >> l) + 1;
        q.ni_s[l] = ((ni - 1) >> l) + 1;
        const long long cells = (long long)q.nj_s[l] * q.ni_s[l];
        bound[l] = cells < nT ? cells : nT;
        q.field0[l + 1] = q.field0[l] + 7 * cells;
        noff += bound[l] + 1;
        ma[l] = min_area ? min_area[l] : 1.0;
    }
    const long long box_bytes = scale_plan(levels, bound, ma, nedge, &q.sp);
    const long long nall = q.sp.nbox_all;
    long long o = 0;
    q.o_box = o;    o += up(box_bytes);
    q.o_planes = o; o += up(7 * nall * (long long)sizeof(float));
    q.o_code = o;   o += up(nall * 8);
    q.o_off = o;    o += up(noff * 8);
    q.o_nbin = o;   o += up(8);
    q.o_flag = o;   o += up(nT * 4);
    q.o_pos = o;    o += up(nT * 4);
    q.o_kin = o;    o += up(nT * 8);
    q.o_kout = o;   o += up(nT * 8);
    q.o_vin = o;    o += up(nT * 4);
    q.o_vout = o;   o += up(nT * 4);
    q.o_tri = o;    o += up(3 * nT * 4);
    q.o_cub = o;
    q.bytes = o;
    *g = q;
    return nullptr;
}

cudaError_t grid_plan_cub(GridPlan* g)
{
    size_t sort_b = 0, scan_b = 0;
    cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, sort_b, (const unsigned long long*)nullptr,
                                                    (unsigned long long*)nullptr, (const int*)nullptr, (int*)nullptr,
                                                    (int)g->nT, 0, g->end_bit);
    if (e != cudaSuccess) return e;
    if ((e = cub::DeviceScan::ExclusiveSum(nullptr, scan_b, (const int*)nullptr, (int*)nullptr, (int)g->nT)) != cudaSuccess)
        return e;
    g->cub_bytes = sort_b > scan_b ? sort_b : scan_b;
    g->bytes = g->o_cub + up((long long)g->cub_bytes);
    return cudaSuccess;
}

cudaError_t launch_deform_grid(const GridPlan& g, const int32_t* tri, const pt* yx0, const int8_t* m0, const pt* yx1,
                               const int8_t* m1, double dt, double oy, double ox, double L0, const double* edges,
                               void* scratch, double* mom, int64_t* hist, float* fields, long long* nbox,
                               int upto, cudaStream_t st)
{
    char* base = static_cast<char*>(scratch);
    auto at = [&](long long o) { return base + o; };
    const ScalePlan& p = g.sp;
    const long long nT = g.nT;
    float* planes = reinterpret_cast<float*>(at(g.o_planes));
    unsigned long long* code = reinterpret_cast<unsigned long long*>(at(g.o_code));
    long long* off = reinterpret_cast<long long*>(at(g.o_off));
    long long* nbin = reinterpret_cast<long long*>(at(g.o_nbin));
    int* flag = reinterpret_cast<int*>(at(g.o_flag));
    int* pos = reinterpret_cast<int*>(at(g.o_pos));
    unsigned long long* kin = reinterpret_cast<unsigned long long*>(at(g.o_kin));
    unsigned long long* kout = reinterpret_cast<unsigned long long*>(at(g.o_kout));
    int* vin = reinterpret_cast<int*>(at(g.o_vin));
    int* vout = reinterpret_cast<int*>(at(g.o_vout));
    int* tri_h = reinterpret_cast<int*>(at(g.o_tri));
    void* tmp = at(g.o_cub);
    const unsigned long long sentinel = 1ull << (g.end_bit - 1);
    size_t tb = g.cub_bytes;
    cudaError_t e;

    k_grid_key<<<blocks(nT), GR_BLOCK, 0, st>>>(nT, tri, yx0, m0, yx1, m1, oy, ox, L0, g.nj, g.ni, sentinel, kin, vin);
    if (upto < GR_STAGE_SORT) return cudaGetLastError();
    if ((e = cub::DeviceRadixSort::SortPairs(tmp, tb, kin, kout, vin, vout, (int)nT, 0, g.end_bit, st)) != cudaSuccess)
        return e;
    if (upto < GR_STAGE_SEGMENT) return cudaGetLastError();
    k_grid_gather<<<blocks(nT), GR_BLOCK, 0, st>>>(nT, kout, vout, tri, sentinel, tri_h, nbin);
    // level 1: runs of the sorted triangles' codes; level s+1: runs of level s's codes >> 2
    long long off0 = 0;
    for (int l = 0; l < g.levels; ++l) {
        const long long items = l ? p.nbox[l - 1] : nT;
        const long long* n = l ? nbox + l - 1 : nbin;
        const unsigned long long* c = l ? code + p.box0[l - 1] : kout;
        const int sh = l ? 2 : 0;
        k_grid_mark<<<blocks(items), GR_BLOCK, 0, st>>>(items, n, c, sh, flag);
        tb = g.cub_bytes;
        if ((e = cub::DeviceScan::ExclusiveSum(tmp, tb, flag, pos, (int)items, st)) != cudaSuccess) return e;
        k_grid_heads<<<blocks(items), GR_BLOCK, 0, st>>>(items, n, c, sh, flag, pos, off + off0, code + p.box0[l],
                                                          nbox + l);
        off0 += p.nbox[l] + 1;
    }
    if (upto < GR_STAGE_ALL) return cudaGetLastError();
    // child ranges of levels >= 2 follow the level-1 ranges, as ScalePlan.child0 expects
    e = launch_deform_scales_devcount(p, tri_h, off, off + p.nbox[0] + 1, yx0, m0, yx1, m1, dt, edges, at(g.o_box),
                                      mom, hist, planes, nbox, st);
    if (e != cudaSuccess) return e;
    const long long nf = g.field0[g.levels];
    const long long fb = (nf + GR_BLOCK - 1) / GR_BLOCK;
    k_grid_fill<<<(unsigned)(fb < 4096 ? fb : 4096), GR_BLOCK, 0, st>>>(nf, fields);
    for (int l = 0; l < g.levels; ++l) {
        const long long cells = (long long)g.nj_s[l] * g.ni_s[l];
        k_grid_scatter<<<blocks(p.nbox[l]), GR_BLOCK, 0, st>>>(p.nbox[l], nbox + l, code + p.box0[l],
                                                               planes + p.box0[l], p.nbox_all, g.ni_s[l], cells,
                                                               fields + g.field0[l]);
    }
    return cudaGetLastError();
}

}  // namespace st
