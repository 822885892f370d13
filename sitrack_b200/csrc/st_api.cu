// st_api.cu -- the C ABI of include/sitrack_b200.h: context, HBM residency of the
// static grid / records / buoy state, and thin launch wrappers.  No arithmetic of
// the tracking path happens on the host in this file.
#include "../../include/sitrack_b200.h"
#include "st_kernels.h"

#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>

using namespace st;

namespace st {
cudaError_t launch_seed_locate_opt(const LocateGrid& lg, const AdvectGrid& g, const float* ic0,
                                   long long nP, const pt* SG, const pt* SC, const SeedOut& o,
                                   double rd_found_km, int max_itr, int do_survive, int do_cell, cudaStream_t st);
}

struct st_ctx {
    int device = 0;
    int Nj = 0, Ni = 0;
    AdvectGrid grid{};
    // owned device memory
    pt *F = nullptr, *U = nullptr, *V = nullptr;
    int8_t* tmask = nullptr;
    int8_t* cellbits = nullptr;
    float4* frames = nullptr;                                   // certified fast path (k_cell_frames)
    unsigned long long frame_stats[2] = {0, 0};                 // cells admitted / examined
    double *latT = nullptr, *lonT = nullptr, *resKM = nullptr;
    int *bin_start = nullptr, *bin_pts = nullptr;
    AngEntry* atab = nullptr;
    LocateGrid lg{};
    bool has_locate = false;
    // buoys
    long long nP = 0, capP = 0;
    pt* pos = nullptr; int2* cell = nullptr; int8_t* alive = nullptr;
    WalkScratch wq = {nullptr, nullptr, nullptr, nullptr};               // scratch between k_advect_cert and k_walk
    unsigned long long* n_bad_cell = nullptr;                   // buoys st_set_buoys discontinued for an out-of-range cell
    int32_t *rec_first = nullptr, *rec_last = nullptr;
    bool has_window = false;
    int variant = 0;            // st_set_kernel_variant: 0 = k_advect_warp (default), 1 = k_advect_step_v1, ...
    // row chaining (st_set_row_chain): pos_src != nullptr => the positions of the buoys that are alive live in that
    // f8 yx row (the last chained step's), pos holds them only for the discontinued ones until sync_pos()
    bool chain_on = false;
    const pt* pos_src = nullptr;
    // host-API scratch outputs
    pt *o_yx = nullptr, *o_ll = nullptr; int8_t* o_mask = nullptr; unsigned long long* o_nalive = nullptr;
    long long capOut = 0;
    // fused position all-gather over peer memory (st_gather_*)
    struct Gather {
        int rank = 0, world = 0, f4 = 0, nbuf = 0;
        long long nP_total = 0, offset = 0;
        size_t buf_bytes = 0, flags_off = 0, block_bytes = 0;
        char* base = nullptr;                 // this rank's block: nbuf gathered arrays, then the flag page
        char* peer[ST_MAX_PEERS + 1] = {};    // every rank's block as mapped here (peer[rank] == base)
        bool ipc_opened[ST_MAX_PEERS + 1] = {};
        bool connected = false;
        int mode = 0;                         // st_gather_set_mode: 0 per-thread peer stores, 1 copy engines, 2 bulk peer stores
        cudaStream_t comm = nullptr, ps[ST_MAX_PEERS] = {};
        cudaEvent_t ev_k = nullptr, ev_c[ST_MAX_PEERS] = {};
    } ga;
    // record slots
    std::vector<float*> d_rec, h_rec;
    cudaStream_t stream = nullptr;
    std::string err;
};

static thread_local std::string g_err;
extern "C" { static int sync_pos_blocking(st_ctx* c); }      // row chaining: defined with the step

static int fail(st_ctx* c, int code, const std::string& msg)
{
    if (c) c->err = msg;
    g_err = msg;
    return code;
}
static int cuda_fail(st_ctx* c, cudaError_t e, const char* what)
{
    return fail(c, e == cudaErrorMemoryAllocation ? ST_ENOMEM : ST_ECUDA,
                std::string(what) + ": " + cudaGetErrorString(e));
}
#define CU(c, call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return cuda_fail((c), e_, #call); } while (0)

// WGS84, the globe cartopy gives NorthPolarStereo by default
static const double kA = 6378137.0, kF = 1.0 / 298.257223563;

static double proj_akm1(double lat_ts_deg, double e)
{
    const double HALFPI = 1.5707963267948966;
    const double phits = fabs(lat_ts_deg) * 0.017453292519943295;
    if (fabs(phits - HALFPI) < 1e-10) return 2.0 / sqrt(pow(1.0 + e, 1.0 + e) * pow(1.0 - e, 1.0 - e));
    const double s = sin(phits), es = e * s;
    const double ts = tan(0.5 * (HALFPI - phits)) / pow((1.0 - es) / (1.0 + es), 0.5 * e);
    return cos(phits) / ts / sqrt(1.0 - es * es);
}

// Geodetic latitude as a function of t = tan(pi/4 - chi/2) on 0 <= t <= 1/2 (lat >~ 37N):
// phi - pi/2 is odd in t, so phi = pi/2 + t Q(w), w = 8 t^2 - 1 in [-1,1].  Q is analytic with its
// nearest singularity at w = -9, so its Chebyshev coefficients fall like 17.9^-k: degree 8 leaves
// 1.7e-13 rad = 1e-11 degrees (degree 11: 5e-17 rad).  Coefficient generation (host, long double), like the angle table: not tracking arithmetic.
static void fit_lat_poly(double e_, double out[ST_LAT_DEG + 1])
{
    const int N = ST_LAT_DEG + 1, M = 32;
    const long double e = e_, PI_L = 3.14159265358979323846264338327950288L;
    long double c[N] = {0};
    for (int j = 0; j < M; ++j) {
        const long double th = PI_L * (j + 0.5L) / M, w = cosl(th);
        const long double t = sqrtl((w + 1.0L) / 8.0L);
        long double phi = PI_L / 2 - 2 * atanl(t);
        for (int it = 0; it < 60; ++it) {
            const long double es = e * sinl(phi);
            phi = PI_L / 2 - 2 * atanl(t * powl((1 - es) / (1 + es), e / 2));
        }
        const long double f = (phi - PI_L / 2) / t;
        for (int k = 0; k < N; ++k) c[k] += f * cosl(k * th);
    }
    for (int k = 0; k < N; ++k) c[k] *= 2.0L / M;
    c[0] *= 0.5L;
    // Chebyshev -> monomial: T_0 = 1, T_1 = w, T_{k+1} = 2 w T_k - T_{k-1}
    long double a[N] = {0}, Tkm1[N] = {0}, Tk[N] = {0};
    Tkm1[0] = 1; Tk[1] = 1;
    a[0] += c[0];
    for (int i = 0; i < N; ++i) a[i] += c[1] * Tk[i];
    for (int k = 2; k < N; ++k) {
        long double Tn[N] = {0};
        for (int i = 0; i < N; ++i) { Tn[i] = -Tkm1[i]; if (i > 0) Tn[i] += 2 * Tk[i - 1]; }
        for (int i = 0; i < N; ++i) a[i] += c[k] * Tn[i];
        for (int i = 0; i < N; ++i) { Tkm1[i] = Tk[i]; Tk[i] = Tn[i]; }
    }
    for (int k = 0; k < N; ++k) out[k] = (double)a[k];
}

static ProjConst make_proj(double lat_ts, double lon0, double kA = ::kA, double kF = ::kF)
{
    const double es = kF * (2.0 - kF), e = sqrt(es);
    const double n = kF / (2.0 - kF), n2 = n * n, n3 = n2 * n, n4 = n3 * n, n5 = n4 * n, n6 = n5 * n;
    ProjConst p;
    p.k_t = 1000.0 / (kA * proj_akm1(lat_ts, e));
    // conformal -> geodetic latitude, series in the third flattening (Karney 2011 / GeographicLib)
    p.c[0] = 2 * n - 2. / 3 * n2 - 2 * n3 + 116. / 45 * n4 + 26. / 45 * n5 - 2854. / 675 * n6;
    p.c[1] = 7. / 3 * n2 - 8. / 5 * n3 - 227. / 45 * n4 + 2704. / 315 * n5 + 2323. / 945 * n6;
    p.c[2] = 56. / 15 * n3 - 136. / 35 * n4 - 1262. / 105 * n5 + 73814. / 2835 * n6;
    p.c[3] = 4279. / 630 * n4 - 332. / 35 * n5 - 399572. / 14175 * n6;
    p.c[4] = 4174. / 315 * n5 - 144838. / 6237 * n6;
    p.c[5] = 601676. / 22275 * n6;
    p.lon0_rad = lon0 * 0.017453292519943295;
    p.fill_lat = p.fill_lon = 0.0;
    const double R2D = 57.29577951308232, PI = 3.141592653589793;
    fit_lat_poly(e, p.lat_poly_deg);
    for (int k = 0; k <= ST_LAT_DEG; ++k) p.lat_poly_deg[k] *= R2D;
    p.w_scale = 8.0 * p.k_t * p.k_t;
    // octant tables of inv_stere_fast (st_device.cuh: folded_angle): angle = sign * (off + sg * theta)
    const double off4[4] = {0.0, PI / 2, PI, PI / 2}, sg4[4] = {1.0, -1.0, -1.0, 1.0};
    for (int o = 0; o < 8; ++o) {
        const double sgn = (o & 4) ? -1.0 : 1.0;
        p.oct_off[o] = (sgn * off4[o & 3]) * R2D + lon0;
        p.oct_sg[o] = sgn * sg4[o & 3] * R2D;
    }
    p.wrap_up = lon0 > 0.0;
    return p;
}
static ProjFwdConst make_proj_fwd(double lat_ts, double lon0, double kA = ::kA, double kF = ::kF)
{
    const double es = kF * (2.0 - kF), e = sqrt(es);
    ProjFwdConst p;
    p.a_akm1_km = kA * proj_akm1(lat_ts, e) / 1000.0;
    p.e = e;
    p.lon0_rad = lon0 * 0.017453292519943295;
    return p;
}

static int use_device(st_ctx* c, int device)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(c, ST_ECUDA, std::string("no CUDA device: ") + cudaGetErrorString(e) +
                                     " (libsitrack_b200 has no CPU fallback)");
    if (device < 0 || device >= n) return fail(c, ST_EINVAL, "device index out of range");
    CU(c, cudaSetDevice(device));
    return ST_OK;
}

template <class T>
static cudaError_t upload(T** dst, const T* src, size_t n)
{
    cudaError_t e = cudaMalloc((void**)dst, n * sizeof(T));
    if (e != cudaSuccess) return e;
    e = cudaMemcpy(*dst, src, n * sizeof(T), cudaMemcpyHostToDevice);
    // a copy from pageable memory may return once the data is staged, before the DMA has landed; the kernels
    // that follow run on non-blocking streams, which the legacy stream does not order: wait for it here
    if (e == cudaSuccess) e = cudaStreamSynchronize(cudaStreamLegacy);
    return e;
}

static bool g_coord_range_ok = true;
static cudaError_t upload_pts(pt** dst, const double* Y, const double* X, size_t n)
{
    std::vector<pt> tmp(n);
    for (size_t k = 0; k < n; ++k) {                                            // layout marshalling only
        tmp[k].y = Y[k]; tmp[k].x = X[k];
        // the branch-free divisions of the inside test rely on coordinates of ordinary magnitude
        const double ay = fabs(Y[k]), ax = fabs(X[k]);
        if (!(ay <= 16777216.0 && ax <= 16777216.0) || (ay != 0.0 && ay < 7.888609052210118e-31) ||
            (ax != 0.0 && ax < 7.888609052210118e-31)) g_coord_range_ok = false;
    }
    return upload(dst, tmp.data(), n);
}

// lat/lon of the fill point (-9999,-9999) km, computed by the device's own inverse: rows of idle
// buoys carry it (si3_part_tracker.py:493 converts every row, fill rows included)
static cudaError_t refresh_fill(st_ctx* c)
{
    double* d = nullptr;
    cudaError_t e = cudaMalloc(&d, 4 * sizeof(double));
    if (e != cudaSuccess) return e;
    const double h[2] = {ST_FILL, ST_FILL};
    double out[2] = {0, 0};
    e = cudaMemcpy(d, h, sizeof(h), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = launch_xy2latlon((const pt*)d, (pt*)(d + 2), 1, c->grid.proj, 0);
    if (e == cudaSuccess) e = cudaMemcpy(out, d + 2, sizeof(out), cudaMemcpyDeviceToHost);
    cudaFree(d);
    c->grid.proj.fill_lat = out[0]; c->grid.proj.fill_lon = out[1];
    return e;
}

static cudaError_t make_angle_table(AngEntry** dst)
{
    std::vector<AngEntry> t(ST_ANG_LAST + 1);
    for (int j = 0; j <= ST_ANG_LAST; ++j) { const double a = j / (double)ST_ANG_STEPS; t[j].alpha = asin(a); t[j].ca = sqrt(1.0 - a * a); t[j].sa = a; t[j].pad = 0.0; }
    return upload(dst, t.data(), t.size());
}

struct Scratch {                       // RAII device scratch for the host-array helpers
    std::vector<void*> p;
    ~Scratch() { for (void* q : p) cudaFree(q); }
    template <class T> cudaError_t up(T** d, const T* h, size_t n)
    { cudaError_t e = upload(d, h, n); if (e == cudaSuccess) p.push_back(*d); return e; }
    template <class T> cudaError_t alloc(T** d, size_t n)
    { cudaError_t e = cudaMalloc((void**)d, n * sizeof(T)); if (e == cudaSuccess) p.push_back(*d); return e; }
};

extern "C" {

int st_abi_version(void) { return ST_ABI_VERSION; }

const char* st_last_error(const st_ctx* ctx) { return ctx ? ctx->err.c_str() : g_err.c_str(); }

int st_create(st_ctx** out, int device, int Nj, int Ni, const double* Yf, const double* Xf,
              const double* Yu, const double* Xu, const double* Yv, const double* Xv,
              const int8_t* tmask, int uv_strategy, double rdt, double rmin_conc)
{
    if (!out) return fail(nullptr, ST_EINVAL, "st_create: out is NULL");
    *out = nullptr;
    if (Nj < 5 || Ni < 5 || (long long)Nj * Ni > 0x7fffffffLL) return fail(nullptr, ST_EINVAL, "st_create: bad grid shape");
    if (!Yf || !Xf || !tmask) return fail(nullptr, ST_EINVAL, "st_create: Yf, Xf and tmask are required");
    if (uv_strategy != 0 && uv_strategy != 1) return fail(nullptr, ST_EINVAL, "st_create: uv_strategy must be 0 or 1");
    if (uv_strategy == 1 && (!Yu || !Xu || !Yv || !Xv))
        return fail(nullptr, ST_EINVAL, "st_create: uv_strategy=1 needs the U- and V-point coordinates");
    int rc = use_device(nullptr, device);
    if (rc) return rc;
    st_ctx* c = new st_ctx();
    c->device = device; c->Nj = Nj; c->Ni = Ni;
    const size_t n = (size_t)Nj * Ni;
    g_coord_range_ok = true;
    cudaError_t e = upload_pts(&c->F, Yf, Xf, n);
    if (e == cudaSuccess && Yu) e = upload_pts(&c->U, Yu, Xu, n);
    if (e == cudaSuccess && Yv) e = upload_pts(&c->V, Yv, Xv, n);
    if (e == cudaSuccess) e = upload(&c->tmask, tmask, n);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { rc = cuda_fail(nullptr, e, "st_create"); st_destroy(c); return rc; }
    if (!g_coord_range_ok) {
        st_destroy(c);
        return fail(nullptr, ST_EINVAL, "st_create: grid coordinates must be km with 2^-100 <= |c| <= 2^24 (or 0) and finite");
    }
    c->grid.Nj = Nj; c->grid.Ni = Ni; c->grid.uv_strategy = uv_strategy; c->grid.rdt = rdt;
    c->grid.rmin_conc = rmin_conc; c->grid.F = c->F; c->grid.U = c->U; c->grid.V = c->V; c->grid.tmask = c->tmask;
    c->grid.proj = make_proj(70.0, -45.0);
    e = make_angle_table(&c->atab);
    c->grid.atab = c->atab;
    if (e == cudaSuccess) e = refresh_fill(c);
    if (e == cudaSuccess) {
        int* d_bad = nullptr; int bad = 0;
        e = cudaMalloc(&c->cellbits, n);
        if (e == cudaSuccess) e = cudaMalloc(&d_bad, sizeof(int));
        if (e == cudaSuccess) e = cudaMemsetAsync(d_bad, 0, sizeof(int), c->stream);
        if (e == cudaSuccess) e = launch_cell_bits(c->grid, c->cellbits, d_bad, c->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        cudaFree(d_bad);
        c->grid.cellbits = c->cellbits;
        // the orientation filter's error bound assumes km coordinates within 2^17 (inside_margin)
        c->grid.filter_ok = (bad == 0) && !getenv("SITRACK_B200_NO_FILTER");
    }
    if (e != cudaSuccess) { rc = cuda_fail(nullptr, e, "st_create(projection tables, cell bits)"); st_destroy(c); return rc; }
    { const char* ev = getenv("SITRACK_B200_KERNEL"); if (ev && ev[0] == 'v' && ev[1] == '1') c->variant = 1; }
    *out = c;
    return ST_OK;
}

// Frames and margins of the certified two-kernel step (variant 4, csrc/st_cert.cuh), built on first use: 32 B per cell.
static int ensure_frames(st_ctx* c)
{
    if (c->grid.frames_ok) return ST_OK;
    if (!c->grid.filter_ok) return fail(c, ST_ESTATE, "this grid has no cell frames (coordinates beyond 2^17 km, or SITRACK_B200_NO_FILTER set)");
    CU(c, cudaSetDevice(c->device));
    const size_t n = (size_t)c->Nj * c->Ni;
    unsigned long long* d_stats = nullptr;
    cudaError_t e = cudaMalloc(&c->frames, sizeof(float4) * 2 * n);
    if (e == cudaSuccess) e = cudaMalloc(&d_stats, 2 * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMemsetAsync(d_stats, 0, 2 * sizeof(unsigned long long), c->stream);
    if (e == cudaSuccess) e = launch_cell_frames(c->grid, c->frames, d_stats, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(c->frame_stats, d_stats, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    cudaFree(d_stats);
    if (e != cudaSuccess) { cudaFree(c->frames); c->frames = nullptr; return cuda_fail(c, e, "cell frames"); }
    c->grid.frames = c->frames;
    c->grid.frames_ok = 1;
    return ST_OK;
}

// scratch between k_advect_cert and k_walk, sized like the buoy arrays
static int ensure_walk_scratch(st_ctx* c)
{
    if (c->wq.P || c->capP == 0) return ST_OK;
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaMalloc(&c->wq.P, sizeof(pt) * c->capP));
    CU(c, cudaMalloc(&c->wq.maskW, sizeof(unsigned) * (c->capP / 32)));
    CU(c, cudaMalloc(&c->wq.maskX, sizeof(unsigned) * (c->capP / 32)));
    CU(c, cudaMalloc(&c->wq.maskA, sizeof(unsigned) * (c->capP / 32)));
    return ST_OK;
}

int st_set_kernel_variant(st_ctx* c, int variant)
{
#ifdef ST_EXPERIMENTS
    const bool known = variant >= 0 && variant <= 12;
#else
    const bool known = variant >= 0 && variant <= 5;
#endif
    if (!c || !known) return fail(c, ST_EINVAL, "st_set_kernel_variant: 0 = 2 warp-private with orientation filter (default), 1 v1, 3 warp-private exact, 4 certified two-kernel step, 5 default kernel with the certified U/V pick; 6-12 only in -DST_EXPERIMENTS builds");
    // a grid that does not qualify for frames (st_create: filter_ok) runs variant 4 as variant 2
    if ((variant == 4 || variant == 5) && c->grid.filter_ok) { int rc = ensure_frames(c); if (rc) return rc; }
    c->variant = variant;
    return ST_OK;
}

void st_destroy(st_ctx* c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    cudaFree(c->F); cudaFree(c->U); cudaFree(c->V); cudaFree(c->tmask); cudaFree(c->atab); cudaFree(c->cellbits); cudaFree(c->frames);
    cudaFree(c->latT); cudaFree(c->lonT); cudaFree(c->resKM); cudaFree(c->bin_start); cudaFree(c->bin_pts);
    cudaFree(c->pos); cudaFree(c->cell); cudaFree(c->alive); cudaFree(c->rec_first); cudaFree(c->rec_last); cudaFree(c->n_bad_cell);
    cudaFree(c->wq.P); cudaFree(c->wq.maskW); cudaFree(c->wq.maskX); cudaFree(c->wq.maskA);
    cudaFree(c->o_yx); cudaFree(c->o_ll); cudaFree(c->o_mask); cudaFree(c->o_nalive);
    for (float* p : c->d_rec) cudaFree(p);
    for (float* p : c->h_rec) cudaFreeHost(p);
    st_gather_destroy(c);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

int st_set_projection(st_ctx* c, double lat_ts_deg, double lon0_deg)
{
    if (!c) return fail(nullptr, ST_EINVAL, "ctx is NULL");
    c->grid.proj = make_proj(lat_ts_deg, lon0_deg);
    CU(c, cudaSetDevice(c->device));
    CU(c, refresh_fill(c));
    return ST_OK;
}

// ---- seeding ---------------------------------------------------------------------------
int st_set_locate_grid(st_ctx* c, const double* latT, const double* lonT, const double* resKM)
{
    if (!c || !latT || !lonT) return fail(c, ST_EINVAL, "st_set_locate_grid: latT/lonT required");
    CU(c, cudaSetDevice(c->device));
    const size_t n = (size_t)c->Nj * c->Ni;
    cudaFree(c->latT); cudaFree(c->lonT); cudaFree(c->resKM); cudaFree(c->bin_start); cudaFree(c->bin_pts);
    c->latT = c->lonT = c->resKM = nullptr; c->bin_start = c->bin_pts = nullptr; c->has_locate = false;
    CU(c, upload(&c->latT, latT, n));
    CU(c, upload(&c->lonT, lonT, n));
    if (resKM) CU(c, upload(&c->resKM, resKM, n));
    CU(c, locate_build(c->Nj, c->Ni, c->latT, c->lonT, c->resKM, &c->lg, &c->bin_start, &c->bin_pts, c->stream));
    c->has_locate = true;
    return ST_OK;
}

int st_seed_locate_dev(st_ctx* c, int64_t nP, const double* SG, const double* SC, const float* ic0,
                       int32_t* cell, int32_t* nearest, int8_t* keep, void* stream)
{
    if (!c) return fail(nullptr, ST_EINVAL, "ctx is NULL");
    if (!c->has_locate) return fail(c, ST_ESTATE, "st_seed_locate: call st_set_locate_grid first");
    if (nP < 0 || !SG || !SC || !ic0) return fail(c, ST_EINVAL, "st_seed_locate: SG, SC and ic0 are required");
    CU(c, cudaSetDevice(c->device));
    SeedOut o{(int2*)cell, (int2*)nearest, keep, nullptr};
    CU(c, launch_seed_locate(c->lg, c->grid, ic0, nP, (const pt*)SG, (const pt*)SC, o, 1, 1, (cudaStream_t)stream));
    return ST_OK;
}

int st_seed_compact_dev(st_ctx* c, int64_t nP, const double* pos, const int32_t* cell, const int8_t* keep,
                        double* out_pos, int32_t* out_cell, int64_t* n_out, void* stream)
{
    if (!c) return fail(nullptr, ST_EINVAL, "ctx is NULL");
    if (nP < 0 || !pos || !cell || !keep || !out_pos || !out_cell || !n_out) return fail(c, ST_EINVAL, "st_seed_compact_dev: NULL argument");
    CU(c, cudaSetDevice(c->device));
    long long* d_n = nullptr;
    CU(c, cudaMalloc(&d_n, sizeof(long long)));
    cudaError_t e = seed_compact(nP, (const pt*)pos, (const int2*)cell, keep, (pt*)out_pos, (int2*)out_cell, d_n, (cudaStream_t)stream);
    long long n = 0;
    if (e == cudaSuccess) e = cudaMemcpy(&n, d_n, sizeof(n), cudaMemcpyDeviceToHost);
    cudaFree(d_n);
    if (e != cudaSuccess) return cuda_fail(c, e, "st_seed_compact_dev");
    *n_out = n;
    return ST_OK;
}

int st_seed_locate_ex(st_ctx* c, int64_t nP, const double* SG, const double* SC, const float* ic0,
                      int32_t* cell, int32_t* nearest, int8_t* keep, int8_t* flag, int32_t* first, int32_t* second)
{
    if (!c) return fail(nullptr, ST_EINVAL, "ctx is NULL");
    if (!c->has_locate) return fail(c, ST_ESTATE, "st_seed_locate: call st_set_locate_grid first");
    if (nP < 0 || !SG || !SC || !ic0 || !cell || !keep) return fail(c, ST_EINVAL, "st_seed_locate: NULL argument");
    if ((first || second) && !flag) return fail(c, ST_EINVAL, "st_seed_locate_ex: first/second come with flag");
    if (nP == 0) return ST_OK;
    CU(c, cudaSetDevice(c->device));
    const size_t n = (size_t)c->Nj * c->Ni;
    Scratch s; double *dSG, *dSC; float* dic; int32_t *dcell, *dnear, *dfirst = nullptr, *dsec = nullptr; int8_t *dkeep, *dflag = nullptr;
    CU(c, s.up(&dSG, SG, (size_t)2 * nP)); CU(c, s.up(&dSC, SC, (size_t)2 * nP)); CU(c, s.up(&dic, ic0, n));
    CU(c, s.alloc(&dcell, (size_t)2 * nP)); CU(c, s.alloc(&dnear, (size_t)2 * nP)); CU(c, s.alloc(&dkeep, (size_t)nP));
    if (flag) { CU(c, s.alloc(&dflag, (size_t)nP)); CU(c, s.alloc(&dfirst, (size_t)nP)); CU(c, s.alloc(&dsec, (size_t)nP)); }
    SeedOut o{(int2*)dcell, (int2*)dnear, dkeep, nullptr, dflag, dfirst, dsec};
    CU(c, launch_seed_locate(c->lg, c->grid, dic, nP, (const pt*)dSG, (const pt*)dSC, o, 1, 1, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    CU(c, cudaMemcpy(cell, dcell, sizeof(int32_t) * 2 * nP, cudaMemcpyDeviceToHost));
    if (nearest) CU(c, cudaMemcpy(nearest, dnear, sizeof(int32_t) * 2 * nP, cudaMemcpyDeviceToHost));
    CU(c, cudaMemcpy(keep, dkeep, (size_t)nP, cudaMemcpyDeviceToHost));
    if (flag) CU(c, cudaMemcpy(flag, dflag, (size_t)nP, cudaMemcpyDeviceToHost));
    if (first) CU(c, cudaMemcpy(first, dfirst, sizeof(int32_t) * nP, cudaMemcpyDeviceToHost));
    if (second) CU(c, cudaMemcpy(second, dsec, sizeof(int32_t) * nP, cudaMemcpyDeviceToHost));
    return ST_OK;
}

int st_seed_locate(st_ctx* c, int64_t nP, const double* SG, const double* SC, const float* ic0,
                   int32_t* cell, int32_t* nearest, int8_t* keep)
{
    return st_seed_locate_ex(c, nP, SG, SC, ic0, cell, nearest, keep, nullptr, nullptr, nullptr);
}

int st_nearest_point(st_ctx* c, int64_t n, const double* latlon, double rd_found_km, int max_itr,
                     int use_brute, int32_t* ji, double* dist_km)
{
    if (!c) return fail(nullptr, ST_EINVAL, "ctx is NULL");
    if (!c->has_locate) return fail(c, ST_ESTATE, "st_nearest_point: call st_set_locate_grid first");
    if (n < 0 || !latlon || !ji) return fail(c, ST_EINVAL, "st_nearest_point: NULL argument");
    if (n == 0) return ST_OK;
    CU(c, cudaSetDevice(c->device));
    double *dll = nullptr, *dd = nullptr; int32_t* dji = nullptr;
    cudaError_t e = upload(&dll, latlon, (size_t)2 * n);
    if (e == cudaSuccess) e = cudaMalloc(&dji, sizeof(int32_t) * 2 * n);
    if (e == cudaSuccess) e = cudaMalloc(&dd, sizeof(double) * n);
    if (e == cudaSuccess) {
        if (use_brute) e = launch_nearest_brute(c->lg, n, (const pt*)dll, (int2*)dji, dd, c->stream);
        else {
            SeedOut o{nullptr, (int2*)dji, nullptr, dd};
            e = launch_seed_locate_opt(c->lg, c->grid, nullptr, n, (const pt*)dll, nullptr, o, rd_found_km, max_itr, 0, 0, c->stream);
        }
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e == cudaSuccess) e = cudaMemcpy(ji, dji, sizeof(int32_t) * 2 * n, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && dist_km) e = cudaMemcpy(dist_km, dd, sizeof(double) * n, cudaMemcpyDeviceToHost);
    cudaFree(dll); cudaFree(dji); cudaFree(dd);
    if (e != cudaSuccess) return cuda_fail(c, e, "st_nearest_point");
    return ST_OK;
}

}  // extern "C" (re-opened below; the kernel of st_find_containing_cell needs C++ linkage)

namespace st {
__global__ void k_find_cell(const AdvectGrid g, long long n, const pt* __restrict__ yx, const int2* __restrict__ near,
                            int2* __restrict__ cell, int8_t* __restrict__ found)
{
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const int dj[5] = {0, 0, 1, 0, -1}, di[5] = {0, 1, 0, -1, 0};
    const pt q = yx[p]; const int2 k = near[p];
    bool in = false; int cj = k.x, ci = k.y;
    for (int kp = 0; kp < 5 && !in; ++kp) {
        cj = k.x + dj[kp]; ci = k.y + di[kp];
        if (cj < 1 || cj >= g.Nj || ci < 1 || ci >= g.Ni) continue;   // (the reference would wrap or raise here)
        const int c = cj * g.Ni + ci;
        in = inside_quad(q.y, q.x, ldg_pt(g.F, c - g.Ni - 1), ldg_pt(g.F, c - g.Ni), ldg_pt(g.F, c), ldg_pt(g.F, c - 1));
    }
    cell[p] = make_int2(cj, ci); found[p] = in;
}
}  // namespace st

namespace st {
// set_buoys: a buoy whose cell lies outside [2,Nj-3] x [2,Ni-3] would fail Survive's first test
// (tracking.py:73-76) the moment it entered that cell; the step kernels gather its stencil unclamped, so such
// a buoy (stale or foreign Initialized_buoys_*.npz, API misuse) starts discontinued instead of faulting.
__global__ void k_init_alive(long long nP, int Nj, int Ni, int2* __restrict__ cell, int8_t* __restrict__ alive,
                             unsigned long long* __restrict__ n_bad)
{
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= nP) return;
    int2 c = cell[p];
    const bool ok = c.x >= 2 && c.x <= Nj - 3 && c.y >= 2 && c.y <= Ni - 3;
    if (!ok) { c.x = (c.x & ~ST_DEAD_BIT) | ST_DEAD_BIT; cell[p] = c; atomicAdd(n_bad, 1ull); }
    alive[p] = ok ? 1 : 0;
}
}  // namespace st

extern "C" {

int st_find_containing_cell(st_ctx* c, int64_t n, const double* yx, const int32_t* ji_near, int32_t* cell, int8_t* found)
{
    if (!c) return fail(nullptr, ST_EINVAL, "ctx is NULL");
    if (n < 0 || !yx || !ji_near || !cell || !found) return fail(c, ST_EINVAL, "st_find_containing_cell: NULL argument");
    if (n == 0) return ST_OK;
    CU(c, cudaSetDevice(c->device));
    double* dyx = nullptr; int32_t *dn = nullptr, *dc = nullptr; int8_t* df = nullptr;
    cudaError_t e = upload(&dyx, yx, (size_t)2 * n);
    if (e == cudaSuccess) e = upload(&dn, ji_near, (size_t)2 * n);
    if (e == cudaSuccess) e = cudaMalloc(&dc, sizeof(int32_t) * 2 * n);
    if (e == cudaSuccess) e = cudaMalloc(&df, (size_t)n);
    if (e == cudaSuccess) {
        k_find_cell<<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>(c->grid, n, (const pt*)dyx, (const int2*)dn, (int2*)dc, df);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e == cudaSuccess) e = cudaMemcpy(cell, dc, sizeof(int32_t) * 2 * n, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(found, df, (size_t)n, cudaMemcpyDeviceToHost);
    cudaFree(dyx); cudaFree(dn); cudaFree(dc); cudaFree(df);
    if (e != cudaSuccess) return cuda_fail(c, e, "st_find_containing_cell");
    return ST_OK;
}

// ---- buoy state ----------------------------------------------------------------------------
// `s`: the stream the caller fills the state on.  The zero fill of fresh capacity must be ordered before that
// fill: a cudaMemset on the legacy default stream is NOT ordered against a non-blocking stream and may land
// after it (seen with two processes sharing a GPU: every buoy dead from the first record).
static int reserve_buoys(st_ctx* c, int64_t nP, bool window, cudaStream_t s)
{
    if (nP > c->capP) {
        cudaFree(c->pos); cudaFree(c->cell); cudaFree(c->alive); cudaFree(c->rec_first); cudaFree(c->rec_last);
        cudaFree(c->wq.P); cudaFree(c->wq.maskW); cudaFree(c->wq.maskX); cudaFree(c->wq.maskA);
        c->wq = WalkScratch{nullptr, nullptr, nullptr, nullptr};
        c->pos = nullptr; c->cell = nullptr; c->alive = nullptr; c->rec_first = c->rec_last = nullptr; c->capP = 0;
        // capacity padded to whole 256-buoy tiles: k_advect_pipe moves state with fixed-size TMA bulk copies
        const long long cap = ((nP + 255) / 256) * 256;
        CU(c, cudaMalloc(&c->pos, sizeof(pt) * cap));
        CU(c, cudaMalloc(&c->cell, sizeof(int2) * cap));
        CU(c, cudaMalloc(&c->alive, (size_t)cap));
        CU(c, cudaMemsetAsync(c->pos, 0, sizeof(pt) * cap, s));
        CU(c, cudaMemsetAsync(c->cell, 0, sizeof(int2) * cap, s));
        CU(c, cudaMemsetAsync(c->alive, 0, (size_t)cap, s));
        c->capP = cap;
    }
    if (window && !c->rec_first) {
        CU(c, cudaMalloc(&c->rec_first, sizeof(int32_t) * c->capP));
        CU(c, cudaMalloc(&c->rec_last, sizeof(int32_t) * c->capP));
    }
    return ST_OK;
}

static int set_buoys_impl(st_ctx* c, int64_t nP, const double* pos, const int32_t* cell, const int32_t* rf,
                          const int32_t* rl, cudaMemcpyKind kind, cudaStream_t s)
{
    if (!c) return fail(nullptr, ST_EINVAL, "ctx is NULL");
    if (nP < 0 || (nP > 0 && (!pos || !cell))) return fail(c, ST_EINVAL, "st_set_buoys: pos and cell are required");
    if ((rf == nullptr) != (rl == nullptr)) return fail(c, ST_EINVAL, "st_set_buoys: rec_first and rec_last go together");
    CU(c, cudaSetDevice(c->device));
    c->nP = 0;
    c->pos_src = nullptr;                                         // a new cloud: nothing to carry over from a chained row
    if (nP > 0) {
        int rc = reserve_buoys(c, nP, rf != nullptr, s);
        if (rc) return rc;
        CU(c, cudaMemcpyAsync(c->pos, pos, sizeof(pt) * nP, kind, s));
        CU(c, cudaMemcpyAsync(c->cell, cell, sizeof(int2) * nP, kind, s));
        if (!c->n_bad_cell) CU(c, cudaMalloc(&c->n_bad_cell, sizeof(unsigned long long)));
        CU(c, cudaMemsetAsync(c->n_bad_cell, 0, sizeof(unsigned long long), s));
        k_init_alive<<<(unsigned)((nP + 255) / 256), 256, 0, s>>>(nP, c->Nj, c->Ni, c->cell, c->alive, c->n_bad_cell);
        CU(c, cudaGetLastError());
        if (rf) {
            CU(c, cudaMemcpyAsync(c->rec_first, rf, sizeof(int32_t) * nP, kind, s));
            CU(c, cudaMemcpyAsync(c->rec_last, rl, sizeof(int32_t) * nP, kind, s));
        }
    }
    c->has_window = rf != nullptr;
    c->nP = nP;
    return ST_OK;
}

int st_set_buoys(st_ctx* c, int64_t nP, const double* pos, const int32_t* cell, const int32_t* rf, const int32_t* rl)
{
    int rc = set_buoys_impl(c, nP, pos, cell, rf, rl, cudaMemcpyHostToDevice, c ? c->stream : nullptr);
    if (rc) return rc;
    CU(c, cudaStreamSynchronize(c->stream));
    return ST_OK;
}

int st_set_buoys_dev(st_ctx* c, int64_t nP, const double* pos, const int32_t* cell, const int32_t* rf,
                     const int32_t* rl, void* stream)
{
    return set_buoys_impl(c, nP, pos, cell, rf, rl, cudaMemcpyDeviceToDevice, (cudaStream_t)stream);
}

int st_get_state(st_ctx* c, double* pos, int32_t* cell, int8_t* alive)
{
    if (!c) return fail(nullptr, ST_EINVAL, "ctx is NULL");
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaDeviceSynchronize());
    if (c->nP == 0) return ST_OK;
    { int rs = sync_pos_blocking(c); if (rs) return rs; }
    if (pos) CU(c, cudaMemcpy(pos, c->pos, sizeof(pt) * c->nP, cudaMemcpyDeviceToHost));
    if (cell) {
        CU(c, cudaMemcpy(cell, c->cell, sizeof(int2) * c->nP, cudaMemcpyDeviceToHost));
        for (long long k = 0; k < c->nP; ++k) cell[2 * k] &= 0x7fffffff;       // bit 31 = discontinued (device encoding)
    }
    if (alive) CU(c, cudaMemcpy(alive, c->alive, (size_t)c->nP, cudaMemcpyDeviceToHost));
    return ST_OK;
}

int st_state_device_ptrs(st_ctx* c, double** pos, int32_t** cell, int8_t** alive)
{
    if (!c) return fail(nullptr, ST_EINVAL, "ctx is NULL");
    { int rs = sync_pos_blocking(c); if (rs) return rs; }          // after chained steps: synchronises the device
    if (pos) *pos = (double*)c->pos;
    if (cell) *cell = (int32_t*)c->cell;
    if (alive) *alive = c->alive;
    return ST_OK;
}

int64_t st_num_buoys(const st_ctx* c) { return c ? c->nP : 0; }

// ---- records -------------------------------------------------------------------------------
int st_record_slots(st_ctx* c, int nslots)
{
    if (!c) return fail(nullptr, ST_EINVAL, "ctx is NULL");
    if (nslots < 1 || nslots > 4096) return fail(c, ST_EINVAL, "st_record_slots: 1..4096 slots");
    CU(c, cudaSetDevice(c->device));
    const size_t bytes = sizeof(float) * 3 * (size_t)c->Nj * c->Ni;
    while ((int)c->d_rec.size() < nslots) {
        float *d = nullptr, *h = nullptr;
        CU(c, cudaMalloc(&d, bytes));
        cudaError_t e = cudaMallocHost(&h, bytes);
        if (e != cudaSuccess) { cudaFree(d); return cuda_fail(c, e, "cudaMallocHost(record staging)"); }
        c->d_rec.push_back(d); c->h_rec.push_back(h);
    }
    return ST_OK;
}

static int check_slot(st_ctx* c, int slot)
{
    if (!c) return fail(nullptr, ST_EINVAL, "ctx is NULL");
    if (slot < 0 || slot >= (int)c->d_rec.size()) return fail(c, ST_EINVAL, "record slot out of range (call st_record_slots)");
    return ST_OK;
}

int st_record_host_buffer(st_ctx* c, int slot, float** staging)
{
    int rc = check_slot(c, slot); if (rc) return rc;
    *staging = c->h_rec[slot];
    return ST_OK;
}
int st_record_device_buffer(st_ctx* c, int slot, float** dev)
{
    int rc = check_slot(c, slot); if (rc) return rc;
    *dev = c->d_rec[slot];
    return ST_OK;
}
int st_submit_record(st_ctx* c, int slot, void* stream)
{
    int rc = check_slot(c, slot); if (rc) return rc;
    CU(c, cudaSetDevice(c->device));
    const size_t bytes = sizeof(float) * 3 * (size_t)c->Nj * c->Ni;
    CU(c, cudaMemcpyAsync(c->d_rec[slot], c->h_rec[slot], bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    return ST_OK;
}

int st_upload_record(st_ctx* c, int slot, const float* host_rec, void* stream)
{
    int rc = check_slot(c, slot); if (rc) return rc;
    if (!host_rec) return fail(c, ST_EINVAL, "st_upload_record: host_rec is NULL");
    CU(c, cudaSetDevice(c->device));
    const size_t bytes = sizeof(float) * 3 * (size_t)c->Nj * c->Ni;
    CU(c, cudaMemcpyAsync(c->d_rec[slot], host_rec, bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    return ST_OK;
}

// ---- the step --------------------------------------------------------------------------------
static BuoyState state_of(st_ctx* c)
{
    BuoyState s;
    s.nP = c->nP; s.pos = c->pos; s.cell = c->cell; s.alive = c->alive;
    s.rec_first = c->has_window ? c->rec_first : nullptr;
    s.rec_last = c->has_window ? c->rec_last : nullptr;
    s.q = c->wq;
    s.pos_in = nullptr; s.chain = 0;
    return s;
}

// st_sync_state: pos <- the chained row for every buoy that is alive; everything that reads pos other than a chained
// step comes through here first
__global__ void k_sync_pos(long long nP, const pt* __restrict__ row, const int2* __restrict__ cell, pt* __restrict__ pos)
{
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < nP && cell[p].x >= 0) pos[p] = row[p];
}
static int sync_pos(st_ctx* c, cudaStream_t s)
{
    if (!c->pos_src) return ST_OK;
    if (c->nP > 0) {
        k_sync_pos<<<(unsigned)((c->nP + 255) / 256), 256, 0, s>>>(c->nP, c->pos_src, c->cell, c->pos);
        CU(c, cudaGetLastError());
    }
    c->pos_src = nullptr;
    return ST_OK;
}
// the same for the synchronous entry points: work the caller queued on any stream finishes first
static int sync_pos_blocking(st_ctx* c)
{
    if (!c->pos_src) return ST_OK;
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaDeviceSynchronize());
    int rc = sync_pos(c, c->stream); if (rc) return rc;
    CU(c, cudaStreamSynchronize(c->stream));
    return ST_OK;
}

int st_set_row_chain(st_ctx* c, int on)
{
    if (!c) return fail(nullptr, ST_EINVAL, "ctx is NULL");
    if (!on) { int rc = sync_pos_blocking(c); if (rc) return rc; }
    c->chain_on = on != 0;
    return ST_OK;
}

int st_sync_state(st_ctx* c, void* stream)
{
    if (!c) return fail(nullptr, ST_EINVAL, "ctx is NULL");
    CU(c, cudaSetDevice(c->device));
    return sync_pos(c, (cudaStream_t)stream);
}

static int step_impl(st_ctx* c, int slot, int jrec, void* out_yx, void* out_latlon, int8_t* out_mask,
                     uint64_t* n_alive, int f4, void* stream)
{
    int rc = check_slot(c, slot); if (rc) return rc;
    CU(c, cudaSetDevice(c->device));
    const size_t npt = (size_t)c->Nj * c->Ni;
    const float* r = c->d_rec[slot];
    StepOut o{(pt*)out_yx, (pt*)out_latlon, out_mask, (unsigned long long*)n_alive};
    o.f4 = f4;
    if (c->variant == 4) { int rs = ensure_walk_scratch(c); if (rs) return rs; }
    BuoyState s = state_of(c);
    // a chained step: f8 rows on this device, every buoy in its window, a kernel of the k_advect_warp family
    const int v = c->variant;
    const bool chain = c->chain_on && !f4 && out_yx && !c->has_window && c->nP > 0 && (v == 0 || v == 2 || v == 3 || v == 5);
    if (chain) { s.pos_in = c->pos_src ? c->pos_src : c->pos; s.chain = 1; }
    else       { int rs = sync_pos(c, (cudaStream_t)stream); if (rs) return rs; }
    CU(c, launch_advect_step(c->grid, r, r + npt, r + 2 * npt, s, jrec, o, c->variant, (cudaStream_t)stream));
    if (chain) c->pos_src = (const pt*)out_yx;
    return ST_OK;
}

int st_step(st_ctx* c, int slot, int jrec, double* out_yx, double* out_latlon, int8_t* out_mask,
            uint64_t* n_alive, void* stream)
{
    return step_impl(c, slot, jrec, out_yx, out_latlon, out_mask, n_alive, 0, stream);
}

int st_step_f4(st_ctx* c, int slot, int jrec, float* out_yx, float* out_latlon, int8_t* out_mask,
               uint64_t* n_alive, void* stream)
{
    return step_impl(c, slot, jrec, out_yx, out_latlon, out_mask, n_alive, 1, stream);
}

int st_step_ext(st_ctx* c, int slot, int jrec, int scheme, int interp, int max_hops, double* out_yx,
                double* out_latlon, int8_t* out_mask, uint64_t* n_alive, void* stream)
{
    int rc = check_slot(c, slot); if (rc) return rc;
    if ((scheme != 1 && scheme != 2 && scheme != 4) || (interp != 0 && interp != 1) || max_hops < 1 || max_hops > 64)
        return fail(c, ST_EINVAL, "st_step_ext: scheme 1|2|4 (Euler, midpoint RK2, RK4), interp 0|1 (face pick, C-grid linear), 1 <= max_hops <= 64");
    if (interp == 1 && (!c->grid.U || !c->grid.V))
        return fail(c, ST_ESTATE, "st_step_ext: C-grid linear interpolation needs the U- and V-point coordinates (st_create with Yu,Xu,Yv,Xv)");
    CU(c, cudaSetDevice(c->device));
    const size_t npt = (size_t)c->Nj * c->Ni;
    const float* r = c->d_rec[slot];
    StepOut o{(pt*)out_yx, (pt*)out_latlon, out_mask, (unsigned long long*)n_alive};
    { int rs = sync_pos(c, (cudaStream_t)stream); if (rs) return rs; }
    CU(c, launch_advect_ext(c->grid, r, r + npt, r + 2 * npt, state_of(c), jrec, o, scheme, interp, max_hops,
                            (cudaStream_t)stream));
    return ST_OK;
}

static int step_multi_impl(st_ctx* c, const float* rec_dev, int64_t rec_stride, int nrec, int jrec0, void* out_yx,
                           void* out_latlon, int8_t* out_mask, int64_t out_stride, uint64_t* n_alive, int f4,
                           void* stream)
{
    if (!c) return fail(nullptr, ST_EINVAL, "ctx is NULL");
    const long long npt = (long long)c->Nj * c->Ni;
    if (!rec_dev || nrec < 0 || rec_stride < 3 * npt) return fail(c, ST_EINVAL, "st_step_multi: bad record stack");
    if (out_stride < c->nP) return fail(c, ST_EINVAL, "st_step_multi: out_stride < nP");
    CU(c, cudaSetDevice(c->device));
    StepOut o{(pt*)out_yx, (pt*)out_latlon, out_mask, (unsigned long long*)n_alive};
    o.f4 = f4;
    { int rs = sync_pos(c, (cudaStream_t)stream); if (rs) return rs; }
    CU(c, launch_advect_multi(c->grid, rec_dev, rec_stride, nrec, state_of(c), jrec0, o, out_stride, (cudaStream_t)stream));
    return ST_OK;
}

int st_step_multi(st_ctx* c, const float* rec_dev, int64_t rec_stride, int nrec, int jrec0, double* out_yx,
                  double* out_latlon, int8_t* out_mask, int64_t out_stride, uint64_t* n_alive, void* stream)
{
    return step_multi_impl(c, rec_dev, rec_stride, nrec, jrec0, out_yx, out_latlon, out_mask, out_stride, n_alive, 0, stream);
}

int st_step_multi_f4(st_ctx* c, const float* rec_dev, int64_t rec_stride, int nrec, int jrec0, float* out_yx,
                     float* out_latlon, int8_t* out_mask, int64_t out_stride, uint64_t* n_alive, void* stream)
{
    return step_multi_impl(c, rec_dev, rec_stride, nrec, jrec0, out_yx, out_latlon, out_mask, out_stride, n_alive, 1, stream);
}

// ---- fused position all-gather over peer memory ---------------------------------------------------
// Block layout, identical on every rank: nbuf gathered arrays of nP_total rows (16 B f8 pairs or 8 B f4
// pairs), then a 256-byte-aligned flag page: ready[world] u64, ack[world] u64 (at +128 B), err u32 (+256 B).
//   ready[s] on rank r : last sequence number whose rows rank s has finished storing into r's buffers
//   ack[s]   on rank r : last sequence number rank s has finished reading from ITS buffers, i.e. r may
//                        overwrite the buffer that sequence used on s
namespace {
constexpr size_t GA_ACK_OFF = 128, GA_ERR_OFF = 256, GA_FLAG_BYTES = 512;
struct FlagTargets { unsigned long long* p[ST_MAX_PEERS + 1]; int n; };

__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p)
{
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long globaltimer_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
// one thread per flag: everything this stream did before (the step kernel's remote row stores included)
// is ordered before the flag by the system-scope release
__global__ void k_gather_signal(FlagTargets t, unsigned long long seq)
{
    const int i = threadIdx.x;
    if (i < t.n) {
        __threadfence_system();
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(t.p[i]), "l"(seq) : "memory");
    }
}
// one thread per flag spins until it reaches `target`; gives up after timeout_ns and raises *err so a
// lost peer turns into an error code on the host instead of a hung GPU
__global__ void k_gather_wait(const unsigned long long* flags, int n, unsigned long long target,
                              unsigned int* err, unsigned long long timeout_ns)
{
    const int i = threadIdx.x;
    if (i < n) {
        const unsigned long long t0 = globaltimer_ns();
        while (ld_acquire_sys(flags + i) < target) {
            if (globaltimer_ns() - t0 > timeout_ns) { atomicExch(err, 1u); break; }
            __nanosleep(200);
        }
    }
}
}  // namespace

int st_gather_create(st_ctx* c, int rank, int world, int64_t nP_total, int64_t offset, int f4, int nbuf,
                     void* handle_out)
{
    if (!c) return fail(nullptr, ST_EINVAL, "ctx is NULL");
    if (world < 1 || world > ST_MAX_PEERS + 1 || rank < 0 || rank >= world || nbuf < 1 || nbuf > 8)
        return fail(c, ST_EINVAL, "st_gather_create: 1 <= world <= 16, 0 <= rank < world, 1 <= nbuf <= 8");
    if (nP_total < 0 || offset < 0 || offset + c->nP > nP_total)
        return fail(c, ST_EINVAL, "st_gather_create: this rank's block [offset, offset+nP) must lie inside nP_total (call st_set_buoys first)");
    CU(c, cudaSetDevice(c->device));
    st_gather_destroy(c);
    st_ctx::Gather& g = c->ga;
    g.rank = rank; g.world = world; g.f4 = f4 ? 1 : 0; g.nbuf = nbuf; g.nP_total = nP_total; g.offset = offset;
    const size_t row = g.f4 ? 8 : 16;
    g.buf_bytes = ((size_t)nP_total * row + 255) / 256 * 256;
    g.flags_off = g.buf_bytes * nbuf;
    g.block_bytes = g.flags_off + GA_FLAG_BYTES;
    CU(c, cudaMalloc(&g.base, g.block_bytes));
    CU(c, cudaMemset(g.base + g.flags_off, 0, GA_FLAG_BYTES));
    CU(c, cudaDeviceSynchronize());                       // default-stream memset: not ordered against the callers' non-blocking streams
    g.peer[rank] = g.base;
    if (handle_out) {
        cudaIpcMemHandle_t h;
        CU(c, cudaIpcGetMemHandle(&h, g.base));
        static_assert(sizeof(h) == ST_IPC_HANDLE_BYTES, "cudaIpcMemHandle_t is 64 bytes");
        memcpy(handle_out, &h, sizeof(h));
    }
    g.connected = (world == 1);
    return ST_OK;
}

int st_gather_connect_ipc(st_ctx* c, const void* handles)
{
    if (!c || !c->ga.base || !handles) return fail(c, ST_ESTATE, "st_gather_connect_ipc: call st_gather_create first");
    CU(c, cudaSetDevice(c->device));
    st_ctx::Gather& g = c->ga;
    for (int r = 0; r < g.world; ++r) {
        if (r == g.rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, (const char*)handles + (size_t)r * ST_IPC_HANDLE_BYTES, sizeof(h));
        void* p = nullptr;
        CU(c, cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
        g.peer[r] = (char*)p; g.ipc_opened[r] = true;
    }
    g.connected = true;
    return ST_OK;
}

int st_gather_connect_ptrs(st_ctx* c, void* const* blocks)
{
    if (!c || !c->ga.base || !blocks) return fail(c, ST_ESTATE, "st_gather_connect_ptrs: call st_gather_create first");
    st_ctx::Gather& g = c->ga;
    for (int r = 0; r < g.world; ++r) {
        if (r == g.rank) continue;
        if (!blocks[r]) return fail(c, ST_EINVAL, "st_gather_connect_ptrs: NULL block");
        g.peer[r] = (char*)blocks[r];
    }
    g.connected = true;
    return ST_OK;
}

int st_gather_block(st_ctx* c, void** block, int64_t* block_bytes)
{
    if (!c || !c->ga.base) return fail(c, ST_ESTATE, "st_gather_block: call st_gather_create first");
    if (block) *block = c->ga.base;
    if (block_bytes) *block_bytes = (int64_t)c->ga.block_bytes;
    return ST_OK;
}

int st_gather_buffer(st_ctx* c, int buf, void** dev)
{
    if (!c || !c->ga.base) return fail(c, ST_ESTATE, "st_gather_buffer: call st_gather_create first");
    if (buf < 0 || buf >= c->ga.nbuf || !dev) return fail(c, ST_EINVAL, "st_gather_buffer: bad buffer index");
    *dev = c->ga.base + (size_t)buf * c->ga.buf_bytes;
    return ST_OK;
}

static int gather_wait_impl(st_ctx* c, size_t off, uint64_t target, void* stream)
{
    st_ctx::Gather& g = c->ga;
    char* fl = g.base + g.flags_off;
    k_gather_wait<<<1, 32, 0, (cudaStream_t)stream>>>((const unsigned long long*)(fl + off), g.world, target,
                                                      (unsigned int*)(fl + GA_ERR_OFF), 10ull * 1000 * 1000 * 1000);
    CU(c, cudaGetLastError());
    return ST_OK;
}
static int gather_signal_impl(st_ctx* c, size_t off, uint64_t seq, void* stream)
{
    st_ctx::Gather& g = c->ga;
    FlagTargets t; t.n = g.world;
    for (int r = 0; r < g.world; ++r)
        t.p[r] = (unsigned long long*)(g.peer[r] + g.flags_off + off) + g.rank;
    k_gather_signal<<<1, 32, 0, (cudaStream_t)stream>>>(t, seq);
    CU(c, cudaGetLastError());
    return ST_OK;
}

int st_step_gather(st_ctx* c, int slot, int jrec, int buf, uint64_t seq, void* out_latlon, int8_t* out_mask,
                   uint64_t* n_alive, void* stream)
{
    int rc = check_slot(c, slot); if (rc) return rc;
    st_ctx::Gather& g = c->ga;
    if (!g.base || !g.connected) return fail(c, ST_ESTATE, "st_step_gather: st_gather_create / st_gather_connect_* first");
    if (buf < 0 || buf >= g.nbuf || seq == 0) return fail(c, ST_EINVAL, "st_step_gather: bad buffer index or seq == 0");
    if (g.offset + c->nP > g.nP_total) return fail(c, ST_ESTATE, "st_step_gather: buoy count changed since st_gather_create");
    CU(c, cudaSetDevice(c->device));
    // the rows written nbuf sequence numbers ago into this buffer must have been consumed everywhere
    if (seq > (uint64_t)g.nbuf) { rc = gather_wait_impl(c, GA_ACK_OFF, seq - g.nbuf, stream); if (rc) return rc; }
    const size_t npt = (size_t)c->Nj * c->Ni;
    const float* r = c->d_rec[slot];
    const size_t row = g.f4 ? 8 : 16;
    const size_t at = (size_t)buf * g.buf_bytes + (size_t)g.offset * row;
    StepOut o{(pt*)(g.base + at), (pt*)out_latlon, out_mask, (unsigned long long*)n_alive};
    o.f4 = g.f4;
    o.npeer = 0;
    o.bulk = 0;
    if (c->variant == 4) { int rs = ensure_walk_scratch(c); if (rs) return rs; }
    { int rs = sync_pos(c, (cudaStream_t)stream); if (rs) return rs; }
    if (g.mode == 1 && g.world > 1) {
        // copy engines: the kernel writes this rank's block only; one peer-to-peer copy per peer follows on its own
        // stream, and the ready flags are released from a side stream once all of them have landed -- the caller's
        // stream goes straight on to the next record
        CU(c, launch_advect_step(c->grid, r, r + npt, r + 2 * npt, state_of(c), jrec, o, c->variant, (cudaStream_t)stream));
        CU(c, cudaEventRecord(g.ev_k, (cudaStream_t)stream));
        CU(c, cudaStreamWaitEvent(g.comm, g.ev_k, 0));
        const size_t bytes = (size_t)c->nP * row;
        for (int k = 1; k < g.world; ++k) {
            const int pr = (g.rank + k) % g.world;
            CU(c, cudaStreamWaitEvent(g.ps[k - 1], g.ev_k, 0));
            CU(c, cudaMemcpyAsync(g.peer[pr] + at, g.base + at, bytes, cudaMemcpyDeviceToDevice, g.ps[k - 1]));
            CU(c, cudaEventRecord(g.ev_c[k - 1], g.ps[k - 1]));
            CU(c, cudaStreamWaitEvent(g.comm, g.ev_c[k - 1], 0));
        }
        return gather_signal_impl(c, 0, seq, g.comm);
    }
    // each rank starts with its right-hand neighbour, so that at any moment the ranks' stores fan out
    // over different destinations instead of all converging on rank 0 first
    for (int k = 1; k < g.world; ++k) o.peer_yx[o.npeer++] = g.peer[(g.rank + k) % g.world] + at;
    // bulk peer stores need 16-byte aligned tiles in every rank's array: this rank's block must start on an even row
    o.bulk = (g.mode == 2 && o.npeer > 0 && (c->variant == 0 || c->variant == 2 || c->variant == 3) &&
              ((size_t)g.offset * row) % 16 == 0) ? 1 : 0;
    CU(c, launch_advect_step(c->grid, r, r + npt, r + 2 * npt, state_of(c), jrec, o, c->variant, (cudaStream_t)stream));
    return gather_signal_impl(c, 0, seq, stream);
}

int st_gather_wait(st_ctx* c, uint64_t seq, void* stream)
{
    if (!c || !c->ga.base || !c->ga.connected) return fail(c, ST_ESTATE, "st_gather_wait: no gather group");
    CU(c, cudaSetDevice(c->device));
    return gather_wait_impl(c, 0, seq, stream);
}

int st_gather_ack(st_ctx* c, uint64_t seq, void* stream)
{
    if (!c || !c->ga.base || !c->ga.connected) return fail(c, ST_ESTATE, "st_gather_ack: no gather group");
    CU(c, cudaSetDevice(c->device));
    return gather_signal_impl(c, GA_ACK_OFF, seq, stream);
}

int st_gather_timed_out(st_ctx* c, int* timed_out)
{
    if (!c || !c->ga.base || !timed_out) return fail(c, ST_ESTATE, "st_gather_timed_out: no gather group");
    CU(c, cudaSetDevice(c->device));
    unsigned int e = 0;
    CU(c, cudaMemcpy(&e, c->ga.base + c->ga.flags_off + GA_ERR_OFF, sizeof(e), cudaMemcpyDeviceToHost));
    *timed_out = (int)e;
    return ST_OK;
}

int st_gather_set_mode(st_ctx* c, int mode)
{
    if (!c || !c->ga.base) return fail(c, ST_ESTATE, "st_gather_set_mode: call st_gather_create first");
    if (mode < 0 || mode > 2) return fail(c, ST_EINVAL, "st_gather_set_mode: 0 per-thread peer stores, 1 copy engines, 2 bulk peer stores");
    st_ctx::Gather& g = c->ga;
    CU(c, cudaSetDevice(c->device));
    if (mode == 1 && !g.comm) {
        CU(c, cudaStreamCreateWithFlags(&g.comm, cudaStreamNonBlocking));
        CU(c, cudaEventCreateWithFlags(&g.ev_k, cudaEventDisableTiming));
        for (int k = 0; k < g.world - 1; ++k) {
            CU(c, cudaStreamCreateWithFlags(&g.ps[k], cudaStreamNonBlocking));
            CU(c, cudaEventCreateWithFlags(&g.ev_c[k], cudaEventDisableTiming));
        }
    }
    g.mode = mode;
    return ST_OK;
}

int st_gather_destroy(st_ctx* c)
{
    if (!c) return ST_OK;
    st_ctx::Gather& g = c->ga;
    if (g.base) {
        cudaSetDevice(c->device);
        cudaDeviceSynchronize();
        if (g.comm) cudaStreamDestroy(g.comm);
        if (g.ev_k) cudaEventDestroy(g.ev_k);
        for (int k = 0; k < ST_MAX_PEERS; ++k) { if (g.ps[k]) cudaStreamDestroy(g.ps[k]); if (g.ev_c[k]) cudaEventDestroy(g.ev_c[k]); }
        for (int r = 0; r < g.world; ++r)
            if (g.ipc_opened[r] && g.peer[r]) cudaIpcCloseMemHandle(g.peer[r]);
        cudaFree(g.base);
    }
    g = st_ctx::Gather{};
    return ST_OK;
}

static int track_record_host_impl(st_ctx* c, int jrec, const float* u, const float* v, const float* ic, void* out_yx,
                                  void* out_latlon, int8_t* out_mask, int64_t* n_alive, int f4)
{
    if (!c) return fail(nullptr, ST_EINVAL, "ctx is NULL");
    if (!u || !v || !ic) return fail(c, ST_EINVAL, "st_track_record_host: u, v, ic are required");
    CU(c, cudaSetDevice(c->device));
    if (c->d_rec.empty()) { int rc = st_record_slots(c, 1); if (rc) return rc; }
    const size_t npt = (size_t)c->Nj * c->Ni;
    cudaStream_t s = c->stream;
    float* d = c->d_rec[0];
    if (v == u + npt && ic == u + 2 * npt) {
        CU(c, cudaMemcpyAsync(d, u, sizeof(float) * 3 * npt, cudaMemcpyHostToDevice, s));
    } else {
        CU(c, cudaMemcpyAsync(d, u, sizeof(float) * npt, cudaMemcpyHostToDevice, s));
        CU(c, cudaMemcpyAsync(d + npt, v, sizeof(float) * npt, cudaMemcpyHostToDevice, s));
        CU(c, cudaMemcpyAsync(d + 2 * npt, ic, sizeof(float) * npt, cudaMemcpyHostToDevice, s));
    }
    if (c->nP > c->capOut) {
        cudaFree(c->o_yx); cudaFree(c->o_ll); cudaFree(c->o_mask);
        c->o_yx = c->o_ll = nullptr; c->o_mask = nullptr; c->capOut = 0;
        CU(c, cudaMalloc(&c->o_yx, sizeof(pt) * c->nP));
        CU(c, cudaMalloc(&c->o_ll, sizeof(pt) * c->nP));
        CU(c, cudaMalloc(&c->o_mask, (size_t)c->nP));
        c->capOut = c->nP;
    }
    if (!c->o_nalive) CU(c, cudaMalloc(&c->o_nalive, sizeof(unsigned long long)));
    if (n_alive) CU(c, cudaMemsetAsync(c->o_nalive, 0, sizeof(unsigned long long), s));
    StepOut o{out_yx ? c->o_yx : nullptr, out_latlon ? c->o_ll : nullptr, out_mask ? c->o_mask : nullptr,
              n_alive ? c->o_nalive : nullptr};
    o.f4 = f4;
    const size_t rowb = f4 ? sizeof(float2) : sizeof(pt);
    if (c->variant == 4) { int rs = ensure_walk_scratch(c); if (rs) return rs; }
    { int rs = sync_pos_blocking(c); if (rs) return rs; }
    CU(c, launch_advect_step(c->grid, d, d + npt, d + 2 * npt, state_of(c), jrec, o, c->variant, s));
    if (c->nP > 0) {
        if (out_yx) CU(c, cudaMemcpyAsync(out_yx, c->o_yx, rowb * c->nP, cudaMemcpyDeviceToHost, s));
        if (out_latlon) CU(c, cudaMemcpyAsync(out_latlon, c->o_ll, rowb * c->nP, cudaMemcpyDeviceToHost, s));
        if (out_mask) CU(c, cudaMemcpyAsync(out_mask, c->o_mask, (size_t)c->nP, cudaMemcpyDeviceToHost, s));
    }
    unsigned long long na = 0;
    if (n_alive) CU(c, cudaMemcpyAsync(&na, c->o_nalive, sizeof(na), cudaMemcpyDeviceToHost, s));
    CU(c, cudaStreamSynchronize(s));
    if (n_alive) *n_alive = (int64_t)na;
    return ST_OK;
}

int st_track_record_host(st_ctx* c, int jrec, const float* u, const float* v, const float* ic, double* out_yx,
                         double* out_latlon, int8_t* out_mask, int64_t* n_alive)
{
    return track_record_host_impl(c, jrec, u, v, ic, out_yx, out_latlon, out_mask, n_alive, 0);
}

int st_track_record_host_f4(st_ctx* c, int jrec, const float* u, const float* v, const float* ic, float* out_yx,
                            float* out_latlon, int8_t* out_mask, int64_t* n_alive)
{
    return track_record_host_impl(c, jrec, u, v, ic, out_yx, out_latlon, out_mask, n_alive, 1);
}

// ---- deformation of buoy triangles (st_deform.cu) ------------------------------------------------
int st_deform_dev(st_ctx* c, int64_t nT, const int32_t* tri, const double* yx0, const int8_t* m0, const double* yx1,
                  const int8_t* m1, double dt_days, float* out, void* stream)
{
    if (nT < 0) return fail(c, ST_EINVAL, "st_deform_dev: nT < 0");
    if (nT == 0) return ST_OK;
    if (!tri || !yx0 || !m0 || !yx1 || !m1 || !out) return fail(c, ST_EINVAL, "st_deform_dev: NULL argument");
    if ((uintptr_t)tri % 16 || (uintptr_t)yx0 % 16 || (uintptr_t)yx1 % 16)
        return fail(c, ST_EINVAL, "st_deform_dev: tri, yx0 and yx1 must be 16-byte aligned");
    if (!(dt_days > 0.0)) return fail(c, ST_EINVAL, "st_deform_dev: dt_days must be positive");
    if (c) CU(c, cudaSetDevice(c->device));
    CU(c, launch_deform(nT, tri, (const pt*)yx0, m0, (const pt*)yx1, m1, dt_days, out, (cudaStream_t)stream));
    return ST_OK;
}

// ---- deformation coarse-grained over a box hierarchy, and its statistics (st_deform_scale.cu) ------
static int scale_plan_checked(st_ctx* c, const char* who, int64_t nT, int levels, const int64_t* level_nbox,
                              const double* min_area, int nedge, ScalePlan* p, long long* bytes)
{
    if (levels < 1 || levels > SC_MAX_LEVELS) return fail(c, ST_EINVAL, std::string(who) + ": levels must be in 1..20");
    if (!level_nbox || !min_area) return fail(c, ST_EINVAL, std::string(who) + ": NULL argument");
    if (nedge < 1 || nedge > SC_MAX_EDGES) return fail(c, ST_EINVAL, std::string(who) + ": nedge must be in 1..4096");
    if (nT < 1 || nT > INT32_MAX) return fail(c, ST_EINVAL, std::string(who) + ": nT must be in 1..2^31-1");
    for (int l = 0; l < levels; ++l) {
        if (level_nbox[l] < 1 || level_nbox[l] > (l ? level_nbox[l - 1] : nT))
            return fail(c, ST_EINVAL, std::string(who) + ": level_nbox must be >= 1 and non-increasing, level 1 <= nT");
        if (!(min_area[l] > 0.0)) return fail(c, ST_EINVAL, std::string(who) + ": min_area must be positive");
    }
    static_assert(sizeof(long long) == sizeof(int64_t), "int64_t is long long");
    *bytes = scale_plan(levels, reinterpret_cast<const long long*>(level_nbox), min_area, nedge, p);
    return ST_OK;
}

int st_deform_scales_scratch_bytes(int64_t nT, int levels, const int64_t* level_nbox, const double* min_area,
                                   int nedge, int64_t* bytes)
{
    ScalePlan p; long long b = 0;
    if (!bytes) return fail(nullptr, ST_EINVAL, "st_deform_scales_scratch_bytes: NULL argument");
    const int rc = scale_plan_checked(nullptr, "st_deform_scales_scratch_bytes", nT, levels, level_nbox, min_area, nedge, &p, &b);
    if (rc != ST_OK) return rc;
    *bytes = b;
    return ST_OK;
}

int st_deform_scales_dev(st_ctx* c, int64_t nT, const int32_t* tri, const double* yx0, const int8_t* m0,
                         const double* yx1, const int8_t* m1, double dt_days, int levels, const int64_t* level_nbox,
                         const double* min_area, const int64_t* tri_off, const int64_t* child_off, int nedge,
                         const double* edges, void* scratch, int64_t scratch_bytes, double* moments, int64_t* hist,
                         float* boxes, void* stream)
{
    ScalePlan p; long long need = 0;
    const int rc = scale_plan_checked(c, "st_deform_scales_dev", nT, levels, level_nbox, min_area, nedge, &p, &need);
    if (rc != ST_OK) return rc;
    if (!tri || !yx0 || !m0 || !yx1 || !m1 || !tri_off || (levels > 1 && !child_off) || !edges || !scratch ||
        !moments || !hist)
        return fail(c, ST_EINVAL, "st_deform_scales_dev: NULL argument");
    if ((uintptr_t)tri % 16 || (uintptr_t)yx0 % 16 || (uintptr_t)yx1 % 16)
        return fail(c, ST_EINVAL, "st_deform_scales_dev: tri, yx0 and yx1 must be 16-byte aligned");
    if ((uintptr_t)tri_off % 8 || (uintptr_t)child_off % 8 || (uintptr_t)edges % 8 || (uintptr_t)scratch % 8 ||
        (uintptr_t)moments % 8 || (uintptr_t)hist % 8 || (uintptr_t)boxes % 4)
        return fail(c, ST_EINVAL, "st_deform_scales_dev: tri_off, child_off, edges, scratch, moments and hist must be 8-byte aligned");
    if (scratch_bytes < need) return fail(c, ST_EINVAL, "st_deform_scales_dev: scratch_bytes is smaller than st_deform_scales_scratch_bytes");
    if (!(dt_days > 0.0)) return fail(c, ST_EINVAL, "st_deform_scales_dev: dt_days must be positive");
    if (c) CU(c, cudaSetDevice(c->device));
    CU(c, launch_deform_scales(p, tri, reinterpret_cast<const long long*>(tri_off),
                               reinterpret_cast<const long long*>(child_off), (const pt*)yx0, m0, (const pt*)yx1, m1,
                               dt_days, edges, scratch, moments, hist, boxes, (cudaStream_t)stream));
    return ST_OK;
}

// ---- deformation coarse-grained over a fixed Eulerian grid, rebuilt every window (st_deform_grid.cu) ----
int st_deform_grid_scratch_bytes(int64_t nT, int levels, int nj, int ni, int nedge, int64_t* bytes)
{
    if (!bytes) return fail(nullptr, ST_EINVAL, "st_deform_grid_scratch_bytes: NULL argument");
    GridPlan g;
    if (const char* why = grid_plan(nT, levels, nj, ni, nullptr, nedge, &g))
        return fail(nullptr, ST_EINVAL, std::string("st_deform_grid_scratch_bytes: ") + why);
    CU(nullptr, grid_plan_cub(&g));
    *bytes = g.bytes;
    return ST_OK;
}

int st_deform_grid_stages_dev(st_ctx* c, int64_t nT, const int32_t* tri, const double* yx0, const int8_t* m0,
                              const double* yx1, const int8_t* m1, double dt_days, int levels, int nj, int ni,
                              double oy, double ox, double L0, const double* min_area, int nedge, const double* edges,
                              void* scratch, int64_t scratch_bytes, double* moments, int64_t* hist, float* fields,
                              int64_t* nbox, int upto, void* stream)
{
    if (upto < GR_STAGE_KEY || upto > GR_STAGE_ALL) return fail(c, ST_EINVAL, "st_deform_grid_stages_dev: upto must be in 1..4");
    GridPlan g;
    if (const char* why = grid_plan(nT, levels, nj, ni, min_area, nedge, &g))
        return fail(c, ST_EINVAL, std::string("st_deform_grid_dev: ") + why);
    if (!tri || !yx0 || !m0 || !yx1 || !m1 || !min_area || !edges || !scratch || !moments || !hist || !fields || !nbox)
        return fail(c, ST_EINVAL, "st_deform_grid_dev: NULL argument");
    if ((uintptr_t)tri % 4 || (uintptr_t)yx0 % 16 || (uintptr_t)yx1 % 16 || (uintptr_t)scratch % 256 ||
        (uintptr_t)edges % 8 || (uintptr_t)moments % 8 || (uintptr_t)hist % 8 || (uintptr_t)nbox % 8 ||
        (uintptr_t)fields % 4)
        return fail(c, ST_EINVAL, "st_deform_grid_dev: yx0 and yx1 must be 16-byte aligned, scratch 256-byte, "
                                  "edges, moments, hist and nbox 8-byte, tri and fields 4-byte");
    for (int l = 0; l < levels; ++l)
        if (!(min_area[l] > 0.0)) return fail(c, ST_EINVAL, "st_deform_grid_dev: min_area must be positive");
    if (!(isfinite(L0) && L0 > 0.0)) return fail(c, ST_EINVAL, "st_deform_grid_dev: L0 must be finite and positive");
    if (!isfinite(oy) || !isfinite(ox)) return fail(c, ST_EINVAL, "st_deform_grid_dev: the origin must be finite");
    if (!(dt_days > 0.0)) return fail(c, ST_EINVAL, "st_deform_grid_dev: dt_days must be positive");
    if (c) CU(c, cudaSetDevice(c->device));
    CU(c, grid_plan_cub(&g));
    if (scratch_bytes < g.bytes)
        return fail(c, ST_EINVAL, "st_deform_grid_dev: scratch_bytes is smaller than st_deform_grid_scratch_bytes");
    CU(c, launch_deform_grid(g, tri, (const pt*)yx0, m0, (const pt*)yx1, m1, dt_days, oy, ox, L0, edges, scratch,
                             moments, hist, fields, reinterpret_cast<long long*>(nbox), upto, (cudaStream_t)stream));
    return ST_OK;
}

int st_deform_grid_dev(st_ctx* c, int64_t nT, const int32_t* tri, const double* yx0, const int8_t* m0,
                       const double* yx1, const int8_t* m1, double dt_days, int levels, int nj, int ni, double oy,
                       double ox, double L0, const double* min_area, int nedge, const double* edges, void* scratch,
                       int64_t scratch_bytes, double* moments, int64_t* hist, float* fields, int64_t* nbox,
                       void* stream)
{
    return st_deform_grid_stages_dev(c, nT, tri, yx0, m0, yx1, m1, dt_days, levels, nj, ni, oy, ox, L0, min_area,
                                     nedge, edges, scratch, scratch_bytes, moments, hist, fields, nbox, GR_STAGE_ALL,
                                     stream);
}

// ---- pair dispersion over time lags, and its statistics (st_disperse.cu) ----------------------------
static const char* disp_check(int64_t nQ, int lags, int nclass_edges, int nedge, int nact)
{
    if (nQ < 1 || nQ > INT32_MAX) return "nQ must be in 1..2^31-1";
    if (lags < 1 || lags > DS_MAX_LAGS) return "lags must be in 1..64";
    if (nclass_edges < 1 || nclass_edges > DS_MAX_CLASS_EDGES) return "nclass_edges must be in 1..63";
    if (nedge < 1 || nedge > SC_MAX_EDGES) return "nedge must be in 1..4096";
    if (nact < 1 || nact > lags) return "the number of active lags must be in 1..lags";
    if (disp_smem(nact, nclass_edges, nedge) > DS_MAX_SMEM)
        return "lags x classes x bins need more than the 227 KB of shared memory a block may have";
    return nullptr;
}

int st_dispersion_scratch_bytes(int64_t nQ, int lags, int nclass_edges, int nedge, int64_t* bytes)
{
    if (!bytes) return fail(nullptr, ST_EINVAL, "st_dispersion_scratch_bytes: NULL argument");
    if (const char* why = disp_check(nQ, lags, nclass_edges, nedge, lags))
        return fail(nullptr, ST_EINVAL, std::string("st_dispersion_scratch_bytes: ") + why);
    *bytes = disp_scratch_bytes(nQ, lags, nclass_edges);
    return ST_OK;
}

int st_dispersion_dev(st_ctx* c, int64_t nQ, const int32_t* pairs, const double* yx1, const int8_t* m1, int nact,
                      const double* const* yx0, const int8_t* const* m0, const int* lag, double dt_days, int lags,
                      int nclass_edges, const double* r_edges, int nedge, const double* bins, void* scratch,
                      int64_t scratch_bytes, int64_t* hist, double* sums, double* per_pair, void* stream)
{
    if (const char* why = disp_check(nQ, lags, nclass_edges, nedge, nact))
        return fail(c, ST_EINVAL, std::string("st_dispersion_dev: ") + why);
    if (!(dt_days > 0.0)) return fail(c, ST_EINVAL, "st_dispersion_dev: dt_days must be positive");
    if (!pairs || !yx1 || !m1 || !yx0 || !m0 || !lag || !r_edges || !bins || !scratch || !hist || !sums)
        return fail(c, ST_EINVAL, "st_dispersion_dev: NULL argument");
    if (per_pair && nact != 1) return fail(c, ST_EINVAL, "st_dispersion_dev: per_pair needs exactly one active lag");
    if ((uintptr_t)pairs % 8 || (uintptr_t)yx1 % 16 || (uintptr_t)r_edges % 8 || (uintptr_t)bins % 8 ||
        (uintptr_t)scratch % 8 || (uintptr_t)hist % 8 || (uintptr_t)sums % 8 || (uintptr_t)per_pair % 8)
        return fail(c, ST_EINVAL, "st_dispersion_dev: rows must be 16-byte aligned, pairs, edges, scratch and outputs "
                                  "8-byte");
    DispOrigins og = {};
    og.nact = nact;
    for (int o = 0; o < nact; ++o) {
        if (!yx0[o] || !m0[o]) return fail(c, ST_EINVAL, "st_dispersion_dev: NULL origin row");
        if ((uintptr_t)yx0[o] % 16) return fail(c, ST_EINVAL, "st_dispersion_dev: rows must be 16-byte aligned");
        if (lag[o] < 1 || lag[o] > lags) return fail(c, ST_EINVAL, "st_dispersion_dev: lag numbers must be in 1..lags");
        for (int p = 0; p < o; ++p)
            if (lag[p] == lag[o]) return fail(c, ST_EINVAL, "st_dispersion_dev: a lag number appears twice");
        og.yx[o] = (const pt*)yx0[o];
        og.m[o] = m0[o];
        og.lag[o] = lag[o];
    }
    if (scratch_bytes < disp_scratch_bytes(nQ, lags, nclass_edges))
        return fail(c, ST_EINVAL, "st_dispersion_dev: scratch_bytes is smaller than st_dispersion_scratch_bytes");
    if (c) CU(c, cudaSetDevice(c->device));
    CU(c, launch_dispersion(og, nQ, pairs, (const pt*)yx1, m1, dt_days, lags, nclass_edges, r_edges, nedge, bins,
                            scratch, hist, sums, per_pair, (cudaStream_t)stream));
    return ST_OK;
}

// ---- finite-size Lyapunov exponents of pairs (st_fsle.cu) ---------------------------------------
static const char* fsle_check(int64_t nQ, int nthr, int ntau_edges)
{
    if (nQ < 1 || nQ > INT32_MAX) return "nQ must be in 1..2^31-1";
    if (nthr < 2 || nthr > FS_MAX_THRESHOLDS) return "nthr must be in 2..64";
    if (ntau_edges < 1 || ntau_edges > FS_MAX_TAU_EDGES) return "ntau_edges must be in 1..512";
    if (fsle_smem(nthr, ntau_edges) > DS_MAX_SMEM)
        return "thresholds x exit-time bins need more than the 227 KB of shared memory a block may have";
    return nullptr;
}

int st_fsle_state_bytes(int64_t nQ, int nthr, int ntau_edges, int64_t* bytes)
{
    if (!bytes) return fail(nullptr, ST_EINVAL, "st_fsle_state_bytes: NULL argument");
    if (const char* why = fsle_check(nQ, nthr, ntau_edges))
        return fail(nullptr, ST_EINVAL, std::string("st_fsle_state_bytes: ") + why);
    *bytes = nQ * 2 * (int64_t)sizeof(int32_t);
    return ST_OK;
}

int st_fsle_dev(st_ctx* c, int64_t nQ, const int32_t* pairs, int32_t* state, const double* yx, const int8_t* m, int t,
                const double* yx0, const int8_t* m0, int nthr, const double* deltas, int ntau_edges,
                const double* tau_edges, int64_t* stats, void* stream)
{
    if (const char* why = fsle_check(nQ, nthr, ntau_edges))
        return fail(c, ST_EINVAL, std::string("st_fsle_dev: ") + why);
    if (t < 1 || t > FS_MAX_SAMPLES) return fail(c, ST_EINVAL, "st_fsle_dev: t must be in 1..65535");
    if (!pairs || !state || !yx || !m || !deltas || !tau_edges || !stats)
        return fail(c, ST_EINVAL, "st_fsle_dev: NULL argument");
    if (!yx0 != !m0) return fail(c, ST_EINVAL, "st_fsle_dev: give both yx_start and m_start, or neither");
    if ((uintptr_t)yx % 16 || (uintptr_t)yx0 % 16 || (uintptr_t)pairs % 8 || (uintptr_t)state % 8 ||
        (uintptr_t)deltas % 8 || (uintptr_t)tau_edges % 8 || (uintptr_t)stats % 8)
        return fail(c, ST_EINVAL, "st_fsle_dev: rows must be 16-byte aligned, pairs, state, edges and stats 8-byte");
    if (c) CU(c, cudaSetDevice(c->device));
    CU(c, launch_fsle(nQ, pairs, state, (const pt*)yx, m, t, (const pt*)yx0, m0, nthr, deltas, ntau_edges, tau_edges,
                      stats, (cudaStream_t)stream));
    return ST_OK;
}

// ---- SI3 T-cell fields sampled along the buoy trajectories (st_sample.cu) ---------------------------------
int st_sample_dev(st_ctx* c, int nF, const float* fields, int64_t plane_stride, const double* yx, const int8_t* mask,
                  int interp, const double* tyx, float* out, void* stream)
{
    if (!c) return fail(nullptr, ST_EINVAL, "st_sample_dev: ctx is NULL");
    if (nF < 1 || nF > SP_MAX_FIELDS) return fail(c, ST_EINVAL, "st_sample_dev: nF must be in 1..16");
    if (interp != 0 && interp != 1) return fail(c, ST_EINVAL, "st_sample_dev: interp must be 0 (cell) or 1 (bilinear)");
    if (!fields || !mask || !out || (interp == 1 && !tyx))
        return fail(c, ST_EINVAL, "st_sample_dev: NULL argument (fields, mask, out; tyx with interp 1)");
    if (plane_stride < (int64_t)c->Nj * c->Ni)
        return fail(c, ST_EINVAL, "st_sample_dev: plane_stride must be at least Nj*Ni");
    if ((uintptr_t)fields % 4 || (uintptr_t)out % 4 || (uintptr_t)yx % 16 || (uintptr_t)tyx % 16)
        return fail(c, ST_EINVAL, "st_sample_dev: fields and out must be 4-byte aligned, yx and tyx 16-byte");
    if (c->nP == 0) return ST_OK;
    CU(c, cudaSetDevice(c->device));
    // NULL: the state's positions, which after chained steps live in the last chained row
    const pt* pos = yx ? (const pt*)yx : (c->pos_src ? c->pos_src : c->pos);
    CU(c, launch_sample(c->nP, c->Nj, c->Ni, c->cell, mask, pos, (const pt*)tyx, c->tmask, fields, plane_stride, nF,
                        interp, out, (cudaStream_t)stream));
    return ST_OK;
}

// ---- projections and batched predicates (host in/out) -------------------------------------------
#define CUS(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return cuda_fail(nullptr, e_, #call); } while (0)

int st_xy2latlon_dev(int64_t n, const double* yx, double* latlon, double lat_ts, double lon0, void* stream)
{
    if (n < 0 || !yx || !latlon) return fail(nullptr, ST_EINVAL, "st_xy2latlon_dev: NULL argument");
    CUS(launch_xy2latlon((const pt*)yx, (pt*)latlon, n, make_proj(lat_ts, lon0), (cudaStream_t)stream));
    return ST_OK;
}

int st_selftest_xy2latlon_fast(int device, int64_t n, const double* yx, double* latlon, double lat_ts, double lon0)
{
    if (n < 0 || !yx || !latlon) return fail(nullptr, ST_EINVAL, "st_selftest_xy2latlon_fast: NULL argument");
    int rc = use_device(nullptr, device); if (rc) return rc;
    if (n == 0) return ST_OK;
    Scratch s; double *a, *b; AngEntry* tab = nullptr;
    CUS(s.up(&a, yx, (size_t)2 * n)); CUS(s.alloc(&b, (size_t)2 * n));
    CUS(make_angle_table(&tab)); s.p.push_back(tab);
    CUS(launch_xy2latlon_fast((const pt*)a, (pt*)b, n, make_proj(lat_ts, lon0), tab, 0));
    CUS(cudaMemcpy(latlon, b, sizeof(double) * 2 * n, cudaMemcpyDeviceToHost));
    return ST_OK;
}

int st_xy2latlon(int device, int64_t n, const double* yx, double* latlon, double lat_ts, double lon0)
{
    if (n < 0 || !yx || !latlon) return fail(nullptr, ST_EINVAL, "st_xy2latlon: NULL argument");
    int rc = use_device(nullptr, device); if (rc) return rc;
    if (n == 0) return ST_OK;
    Scratch s; double *a, *b;
    CUS(s.up(&a, yx, (size_t)2 * n)); CUS(s.alloc(&b, (size_t)2 * n));
    CUS(launch_xy2latlon((const pt*)a, (pt*)b, n, make_proj(lat_ts, lon0), 0));
    CUS(cudaMemcpy(latlon, b, sizeof(double) * 2 * n, cudaMemcpyDeviceToHost));
    return ST_OK;
}

int st_latlon2xy(int device, int64_t n, const double* latlon, double* yx, double lat_ts, double lon0)
{
    if (n < 0 || !yx || !latlon) return fail(nullptr, ST_EINVAL, "st_latlon2xy: NULL argument");
    int rc = use_device(nullptr, device); if (rc) return rc;
    if (n == 0) return ST_OK;
    Scratch s; double *a, *b;
    CUS(s.up(&a, latlon, (size_t)2 * n)); CUS(s.alloc(&b, (size_t)2 * n));
    CUS(launch_latlon2xy((const pt*)a, (pt*)b, n, make_proj_fwd(lat_ts, lon0), 0));
    CUS(cudaMemcpy(yx, b, sizeof(double) * 2 * n, cudaMemcpyDeviceToHost));
    return ST_OK;
}

int st_selftest_proj(int device, int which, int64_t n, const double* in, double* out, double lat_ts, double lon0,
                     double a_m, double f)
{
    if (n < 0 || !in || !out) return fail(nullptr, ST_EINVAL, "st_selftest_proj: NULL argument");
    if (which < 0 || which > 2 || !(a_m > 0.0) || !(f >= 0.0 && f < 0.1)) return fail(nullptr, ST_EINVAL, "st_selftest_proj: which in 0..2, a > 0, 0 <= f < 0.1");
    int rc = use_device(nullptr, device); if (rc) return rc;
    if (n == 0) return ST_OK;
    Scratch s; double *a, *b; AngEntry* tab = nullptr;
    CUS(s.up(&a, in, (size_t)2 * n)); CUS(s.alloc(&b, (size_t)2 * n));
    if (which == 0) CUS(launch_xy2latlon((const pt*)a, (pt*)b, n, make_proj(lat_ts, lon0, a_m, f), 0));
    else if (which == 1) {
        CUS(make_angle_table(&tab)); s.p.push_back(tab);
        CUS(launch_xy2latlon_fast((const pt*)a, (pt*)b, n, make_proj(lat_ts, lon0, a_m, f), tab, 0));
    } else CUS(launch_latlon2xy((const pt*)a, (pt*)b, n, make_proj_fwd(lat_ts, lon0, a_m, f), 0));
    CUS(cudaMemcpy(out, b, sizeof(double) * 2 * n, cudaMemcpyDeviceToHost));
    return ST_OK;
}

int st_selftest_div1000(int device, int64_t n, const double* a, double* q_fast, double* q_div)
{
    if (n < 0 || !a || !q_fast || !q_div) return fail(nullptr, ST_EINVAL, "st_selftest_div1000: NULL argument");
    int rc = use_device(nullptr, device); if (rc) return rc;
    if (n == 0) return ST_OK;
    Scratch s; double *d, *f, *r;
    CUS(s.up(&d, a, (size_t)n)); CUS(s.alloc(&f, (size_t)n)); CUS(s.alloc(&r, (size_t)n));
    CUS(launch_div1000(d, f, r, n, 0));
    CUS(cudaMemcpy(q_fast, f, sizeof(double) * n, cudaMemcpyDeviceToHost));
    CUS(cudaMemcpy(q_div, r, sizeof(double) * n, cudaMemcpyDeviceToHost));
    return ST_OK;
}

int st_selftest_divide(int device, int64_t n, const double* a, const double* b, double* q_fast, double* q_div)
{
    if (n < 0 || !a || !b || !q_fast || !q_div) return fail(nullptr, ST_EINVAL, "st_selftest_divide: NULL argument");
    int rc = use_device(nullptr, device); if (rc) return rc;
    if (n == 0) return ST_OK;
    Scratch s; double *da, *db, *f, *r;
    CUS(s.up(&da, a, (size_t)n)); CUS(s.up(&db, b, (size_t)n)); CUS(s.alloc(&f, (size_t)n)); CUS(s.alloc(&r, (size_t)n));
    CUS(launch_divcore(da, db, f, r, n, 0));
    CUS(cudaMemcpy(q_fast, f, sizeof(double) * n, cudaMemcpyDeviceToHost));
    CUS(cudaMemcpy(q_div, r, sizeof(double) * n, cudaMemcpyDeviceToHost));
    return ST_OK;
}

int st_cert_stats(st_ctx* c, int64_t* admitted, int64_t* examined)
{
    if (!c) return fail(nullptr, ST_EINVAL, "ctx is NULL");
    if (c->grid.filter_ok) { int rc = ensure_frames(c); if (rc) return rc; }
    if (admitted) *admitted = c->grid.frames_ok ? (int64_t)c->frame_stats[0] : 0;
    if (examined) *examined = c->grid.frames_ok ? (int64_t)c->frame_stats[1] : 0;
    return ST_OK;
}

int st_cert_frames(st_ctx* c, float* frames, uint32_t* margins)
{
    if (!c) return fail(nullptr, ST_EINVAL, "ctx is NULL");
    { int rc = ensure_frames(c); if (rc) return rc; }
    CU(c, cudaSetDevice(c->device));
    const size_t n = (size_t)c->Nj * c->Ni;
    std::vector<uint32_t> raw(8 * n);
    CU(c, cudaMemcpy(raw.data(), c->frames, sizeof(float4) * 2 * n, cudaMemcpyDeviceToHost));
    for (size_t k = 0; k < n; ++k) {
        const uint32_t mw = raw[8 * k + 6], ew = raw[8 * k + 7];
        if (margins) margins[k] = mw;
        if (frames) {
            memcpy(frames + 8 * k, &raw[8 * k], 6 * sizeof(float));
            const uint32_t es = ew & 0xffff0000u, et = ew << 16;
            memcpy(frames + 8 * k + 6, &es, 4); memcpy(frames + 8 * k + 7, &et, 4);
        }
    }
    return ST_OK;
}

int st_selftest_cert(st_ctx* c, int64_t n, const double* yx, const int32_t* cell, const float* vel4, uint8_t* flags)
{
    if (!c) return fail(nullptr, ST_EINVAL, "ctx is NULL");
    if (n < 0 || !yx || !cell || !vel4 || !flags) return fail(c, ST_EINVAL, "st_selftest_cert: NULL argument");
    { int rc = ensure_frames(c); if (rc) return rc; }
    if (n == 0) return ST_OK;
    for (int64_t k = 0; k < n; ++k)
        if (cell[2 * k] < 1 || cell[2 * k] >= c->Nj || cell[2 * k + 1] < 1 || cell[2 * k + 1] >= c->Ni)
            return fail(c, ST_EINVAL, "st_selftest_cert: cell outside [1,Nj-1]x[1,Ni-1]");
    CU(c, cudaSetDevice(c->device));
    Scratch s; double* dyx; int32_t* dc; float* dv; uint8_t* df;
    CU(c, s.up(&dyx, yx, (size_t)2 * n)); CU(c, s.up(&dc, cell, (size_t)2 * n)); CU(c, s.up(&dv, vel4, (size_t)4 * n));
    CU(c, s.alloc(&df, (size_t)n));
    CU(c, launch_cert_selftest(c->grid, n, (const pt*)dyx, (const int2*)dc, (const float4*)dv, df, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    CU(c, cudaMemcpy(flags, df, (size_t)n, cudaMemcpyDeviceToHost));
    return ST_OK;
}

int st_intersect2seg(int device, int64_t n, const double* A, const double* B, const double* C, const double* D, int8_t* out)
{
    if (n < 0 || !A || !B || !C || !D || !out) return fail(nullptr, ST_EINVAL, "st_intersect2seg: NULL argument");
    int rc = use_device(nullptr, device); if (rc) return rc;
    if (n == 0) return ST_OK;
    Scratch s; double *a, *b, *c, *d; int8_t* o;
    CUS(s.up(&a, A, (size_t)2 * n)); CUS(s.up(&b, B, (size_t)2 * n)); CUS(s.up(&c, C, (size_t)2 * n)); CUS(s.up(&d, D, (size_t)2 * n));
    CUS(s.alloc(&o, (size_t)n));
    CUS(launch_geom_intersect(n, (pt*)a, (pt*)b, (pt*)c, (pt*)d, o, 0));
    CUS(cudaMemcpy(out, o, (size_t)n, cudaMemcpyDeviceToHost));
    return ST_OK;
}

int st_inside_quad(int device, int64_t n, const double* yx, const double* quads, int8_t* out)
{
    if (n < 0 || !yx || !quads || !out) return fail(nullptr, ST_EINVAL, "st_inside_quad: NULL argument");
    int rc = use_device(nullptr, device); if (rc) return rc;
    if (n == 0) return ST_OK;
    Scratch s; double *a, *q; int8_t* o;
    CUS(s.up(&a, yx, (size_t)2 * n)); CUS(s.up(&q, quads, (size_t)8 * n)); CUS(s.alloc(&o, (size_t)n));
    CUS(launch_geom_inside(n, (pt*)a, (pt*)q, o, 0));
    CUS(cudaMemcpy(out, o, (size_t)n, cudaMemcpyDeviceToHost));
    return ST_OK;
}

int st_cell_walk(int device, int64_t n, const double* p1, const double* p2, const double* ring,
                 const int32_t* kcross_in, int32_t* kcross, int32_t* knhc)
{
    if (n < 0 || !p1 || !p2 || !ring) return fail(nullptr, ST_EINVAL, "st_cell_walk: NULL argument");
    int rc = use_device(nullptr, device); if (rc) return rc;
    if (n == 0) return ST_OK;
    Scratch s; double *a, *b, *r; int32_t *ki = nullptr, *kc, *kn;
    CUS(s.up(&a, p1, (size_t)2 * n)); CUS(s.up(&b, p2, (size_t)2 * n)); CUS(s.up(&r, ring, (size_t)24 * n));
    if (kcross_in) CUS(s.up(&ki, kcross_in, (size_t)n));
    CUS(s.alloc(&kc, (size_t)n)); CUS(s.alloc(&kn, (size_t)n));
    CUS(launch_geom_walk(n, (pt*)a, (pt*)b, (pt*)r, ki, kc, kn, 0));
    if (kcross) CUS(cudaMemcpy(kcross, kc, sizeof(int32_t) * n, cudaMemcpyDeviceToHost));
    if (knhc) CUS(cudaMemcpy(knhc, kn, sizeof(int32_t) * n, cudaMemcpyDeviceToHost));
    return ST_OK;
}

int st_survive(int device, int64_t n, const int32_t* ji, int Nj, int Ni, const int8_t* tm5, const double* ic5,
               double rmin_conc, int32_t* kill)
{
    if (n < 0 || !ji || !tm5 || !kill) return fail(nullptr, ST_EINVAL, "st_survive: NULL argument");
    int rc = use_device(nullptr, device); if (rc) return rc;
    if (n == 0) return ST_OK;
    Scratch s; int32_t *a, *o; int8_t* t; double* c = nullptr;
    CUS(s.up(&a, ji, (size_t)2 * n)); CUS(s.up(&t, tm5, (size_t)5 * n));
    if (ic5) CUS(s.up(&c, ic5, (size_t)5 * n));
    CUS(s.alloc(&o, (size_t)n));
    CUS(launch_geom_survive(n, a, Nj, Ni, t, c, rmin_conc, o, 0));
    CUS(cudaMemcpy(kill, o, sizeof(int32_t) * n, cudaMemcpyDeviceToHost));
    return ST_OK;
}

int st_haversine(int device, int64_t n, double plat, double plon, const double* lat, const double* lon, double* out_km)
{
    if (n < 0 || !lat || !lon || !out_km) return fail(nullptr, ST_EINVAL, "st_haversine: NULL argument");
    int rc = use_device(nullptr, device); if (rc) return rc;
    if (n == 0) return ST_OK;
    Scratch s; double *a, *b, *o;
    CUS(s.up(&a, lat, (size_t)n)); CUS(s.up(&b, lon, (size_t)n)); CUS(s.alloc(&o, (size_t)n));
    CUS(launch_haversine(n, plat, plon, a, b, o, 0));
    CUS(cudaMemcpy(out_km, o, sizeof(double) * n, cudaMemcpyDeviceToHost));
    return ST_OK;
}

}  // extern "C"
