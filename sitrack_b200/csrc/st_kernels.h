// st_kernels.h -- kernel parameter blocks and launchers shared by the .cu files.
#pragma once
#include "st_device.cuh"

namespace st {

constexpr int ST_BLOCK = 256;

// Static grid + run constants, passed by value (lives in the kernel's constant bank).
struct AdvectGrid {
    int Nj, Ni;
    int uv_strategy;            // si3_part_tracker.py:37 iUVstrategy
    double rdt;                 // si3_part_tracker.py:31
    double rmin_conc;           // tracking.py:4
    const pt* F;                // (Nj*Ni) [y,x] km, F-points (cell corners)
    const pt* U;                // U-points (east faces)
    const pt* V;                // V-points (north faces)
    const int8_t* tmask;        // (Nj*Ni)
    const int8_t* cellbits;     // (Nj*Ni) per host cell: bit 0 = ccw(F[c], V[c-Ni], V[c]), bit 1 = ccw(F[c], U[c-1], U[c])
                                //  -- the buoy-independent orientation of the two U/V-pick segment tests (k_cell_bits);
                                //  bit 2 = the cell is a convex anticlockwise quadrangle with edges shorter than 1024 km
    int filter_ok;              // the grid qualifies for the orientation filter of k_advect_warp (st_create checks)
    int cellbits_uniform;       // the bits every cell of [2,Nj-3] x [2,Ni-3] carries, -1 when they differ (st_create)
    // certified fast path (st_cert.cuh, k_cell_frames): per host cell an affine frame and two margins, 32 B
    const float4* frames;       // (2*Nj*Ni) {oy, ox, a, b}, {c, d, bf16(hin) << 16 | bf16(msep), bf16(es) << 16 | bf16(et)};
                                // hin = -1: nothing is certified in this cell
    int frames_ok;              // frames were built (filter_ok and the build succeeded)
    ProjConst proj;
    const AngEntry* atab;       // 47-entry angle table of inv_stere_fast (device)
};

// Scratch between k_advect_cert and k_walk (st_cert.cuh), all of it rewritten by every step.
struct WalkScratch {
    pt* P;                      // (nP) position before the step of the lanes marked in maskW, at the buoy's own index
    unsigned* maskW;            // (ceil(nP/32)) per tile of 32 buoys: lanes whose "still inside" is not certified
    unsigned* maskX;            // (ceil(nP/32)) lanes whose U/V pick is not certified
    unsigned* maskA;            // (ceil(nP/32)) lanes alive when the step began (k_walk sums them into n_alive)
};

// Buoy state, struct of arrays in HBM.
struct BuoyState {
    long long nP;
    pt* pos;                    // [y,x] km
    int2* cell;                 // {jT, iT}: T-point at the centre of the host cell
    int8_t* alive;              // 1 alive, 0 discontinued
    const int32_t* rec_first;   // optional per-buoy record window (no -F); nullptr with -F
    const int32_t* rec_last;
    WalkScratch q;              // q.P == nullptr: not allocated (variant 2 runs instead of the default step)
    // Row chaining (st_set_row_chain, k_advect_warp ROWS 2): the f8 yx row of the previous step IS the position
    // state of the buoys that are alive.  The step reads positions from pos_in (that row, or pos on the first
    // step) and stores the new ones into the new row only -- pos is written at a buoy's death (its last position)
    // and by st_sync_state.  16 B per buoy-step less to write.
    const pt* pos_in;           // nullptr: pos
    int chain;                  // 1: this launch leaves pos alone (set by the API layer only when the launch qualifies)
};

// One trajectory row (all nullable).
constexpr int ST_MAX_PEERS = 15;
struct StepOut {
    pt* yx;                     // (nP) [y,x] km     -> xPosC[jt+1]
    pt* latlon;                 // (nP) [lat,lon]    -> xPosG[jt+1]
    int8_t* mask;               // (nP)              -> xmask[jt+1,:,0]
    unsigned long long* n_alive;
    // Rows in the output file's dtype: yx / latlon (and peer_yx) then point at (nP,2) f4 and every
    // value is rounded once, to nearest even, exactly like the f8 -> f4 cast of ncio.py:156-159.
    int f4;
    // Fused position all-gather: the yx row is also stored, by the same thread in the same kernel, into
    // npeer remote buffers (peer-mapped HBM of the other ranks over NVLink), each already offset to
    // this rank's block of the gathered (nP_total,2) array.
    int npeer;
    void* peer_yx[ST_MAX_PEERS];
    // bulk != 0 (k_advect_warp only): a warp stages the 32 rows of its tile in shared memory and sends them to each
    // peer with ONE cp.async.bulk (256 B as f4, 512 B as f8) instead of 32 per-thread stores per peer
    int bulk;
};

__device__ __forceinline__ void put_row_pt(void* base, long long p, pt v, int f4)
{
    if (f4) __stcs(reinterpret_cast<float2*>(base) + p, make_float2(__double2float_rn(v.y), __double2float_rn(v.x)));
    else    st_stream_pt(reinterpret_cast<pt*>(base) + p, v);
}
// remote rows: plain (write-back) stores, the link packs them; visibility to the peer is given by the
// release of the ready flag that follows the kernel (st_api.cu: k_gather_signal)
__device__ __forceinline__ void put_row_yx(const StepOut& o, long long p, pt v)
{
    put_row_pt(o.yx, p, v, o.f4);
    if (o.npeer) {
        if (o.f4) {
            const float2 w = make_float2(__double2float_rn(v.y), __double2float_rn(v.x));
#pragma unroll 1
            for (int k = 0; k < o.npeer; ++k) reinterpret_cast<float2*>(o.peer_yx[k])[p] = w;
        } else {
            const double2 w = make_double2(v.y, v.x);
#pragma unroll 1
            for (int k = 0; k < o.npeer; ++k) reinterpret_cast<double2*>(o.peer_yx[k])[p] = w;
        }
    }
}

cudaError_t launch_advect_step(const AdvectGrid& g, const float* u, const float* v, const float* ic,
                               const BuoyState& s, int jrec, const StepOut& o, int variant, cudaStream_t st);
cudaError_t launch_advect_ext(const AdvectGrid& g, const float* u, const float* v, const float* ic,
                              const BuoyState& s, int jrec, const StepOut& o, int scheme, int interp, int max_hops,
                              cudaStream_t st);
// span (2 ints, preset {-1, 0}): AND and OR of the bits over the cells a live buoy can occupy
cudaError_t launch_cell_bits(const AdvectGrid& g, int8_t* bits, int* n_bad_coord, int* span, cudaStream_t st);
cudaError_t launch_cell_frames(const AdvectGrid& g, float4* frames, unsigned long long* stats, cudaStream_t st);
cudaError_t launch_cert_selftest(const AdvectGrid& g, long long n, const pt* yx, const int2* cell, const float4* vel,
                                 uint8_t* flags, cudaStream_t st);
cudaError_t launch_divcore(const double* a, const double* b, double* q_fast, double* q_div, long long n, cudaStream_t st);
cudaError_t launch_div1000(const double* a, double* q_fast, double* q_div, long long n, cudaStream_t st);
cudaError_t launch_advect_multi(const AdvectGrid& g, const float* rec0, long long rec_stride, int nrec,
                                const BuoyState& s, int jrec0, const StepOut& o, long long out_stride,
                                cudaStream_t st);
cudaError_t launch_xy2latlon(const pt* yx, pt* latlon, long long n, const ProjConst& pc, cudaStream_t st);
cudaError_t launch_xy2latlon_fast(const pt* yx, pt* latlon, long long n, const ProjConst& pc, const AngEntry* tab, cudaStream_t st);
cudaError_t launch_latlon2xy(const pt* latlon, pt* yx, long long n, const ProjFwdConst& pc, cudaStream_t st);

// ---- locate (st_locate.cu) ---------------------------------------------------------
// Coarse-bin spatial hash of the T-points in a unit-sphere polar stereographic plane.
struct LocateGrid {
    int Nj, Ni;
    const double* latT;         // (Nj*Ni) degrees
    const double* lonT;
    const double* resKM;        // (Nj*Ni) local resolution [km] (ncio.py:56-57)
    // hash
    int nbx, nby;               // bins along x / y
    double x0, y0, inv_bin, bin;   // plane origin, 1/bin size, bin size
    double q2max;               // max |Q|^2 over grid points (plane radius^2)
    double res_max;             // max resKM
    const int* bin_start;       // (nbx*nby+1) exclusive prefix
    const int* bin_pts;         // (Nj*Ni) flat T indices sorted by bin
};

struct SeedOut {
    int2* cell;                 // containing cell {jT,iT}
    int2* nearest;              // nearest T-point or {-1,-1}  (nullable)
    int8_t* keep;               // kmask of SeedInit
    double* dmin;               // haversine distance to the nearest T-point (nullable)
    int8_t* flag;               // (nullable) bit 0: argmin decided by < 1e-11 relative, bit 1: acceptance within 1e-11 of its radius
    int* first;                 // (nullable, with flag) flat index of the nearest T-point before the acceptance test
    int* second;                // (nullable, with flag) flat index of the runner-up when bit 0 is set, else -1
};

cudaError_t locate_build(int Nj, int Ni, const double* d_lat, const double* d_lon, const double* d_res,
                         LocateGrid* out, int** owned_start, int** owned_pts, cudaStream_t st);
cudaError_t seed_compact(long long nP, const pt* pos, const int2* cell, const int8_t* keep, pt* out_pos, int2* out_cell,
                         long long* d_nout, cudaStream_t st);
cudaError_t launch_seed_locate(const LocateGrid& lg, const AdvectGrid& g, const float* ic0,
                               long long nP, const pt* SG, const pt* SC, const SeedOut& o,
                               int do_survive, int do_cell, cudaStream_t st);
cudaError_t launch_nearest_brute(const LocateGrid& lg, long long nP, const pt* SG, int2* nearest,
                                 double* dmin, cudaStream_t st);

// ---- batched geometry predicates on explicit coordinates (st_geom.cu) ----------------
cudaError_t launch_geom_intersect(long long n, const pt* A, const pt* B, const pt* C, const pt* D,
                                  int8_t* out, cudaStream_t st);
cudaError_t launch_geom_inside(long long n, const pt* yx, const pt* quads, int8_t* out, cudaStream_t st);
cudaError_t launch_geom_walk(long long n, const pt* p1, const pt* p2, const pt* ring, const int32_t* kcross_in,
                             int32_t* kcross, int32_t* knhc, cudaStream_t st);
cudaError_t launch_geom_survive(long long n, const int32_t* ji, int Nj, int Ni, const int8_t* tm5,
                                const double* ic5, double rmin_conc, int32_t* out, cudaStream_t st);
cudaError_t launch_haversine(long long n, double plat, double plon, const double* lat, const double* lon,
                             double* out, cudaStream_t st);

// ---- strain rates of buoy triangles between two trajectory rows (st_deform.cu) -------------
// k_deform: tri (nT,3) buoy indices (16-byte aligned), yx0/yx1 (nP) positions and m0/m1 (nP) masks at the two ends
// of the window, dt in days; out = six (nT) f4 planes [divergence | shear | vorticity | area | y_ctr | x_ctr].
cudaError_t launch_deform(long long nT, const int32_t* tri, const pt* yx0, const int8_t* m0, const pt* yx1,
                          const int8_t* m1, double dt, float* out, cudaStream_t st);

// ---- coarse-grained deformation over a hierarchy of material boxes, and its statistics (st_deform_scale.cu) ----
constexpr int SC_MAX_LEVELS = 20;
constexpr int SC_MAX_EDGES = 4096;

// Shapes of one hierarchy, passed by value.  Box records of all levels are concatenated (level 1 first); child
// offsets of levels >= 2 likewise; moment partials: scale s (0 = triangles) owns blocks [blk0[s], blk0[s+1]).
struct ScalePlan {
    int levels, nedge, nbin;                    // nbin = nedge + 1 counts per histogram
    long long nbox_all;
    long long nbox[SC_MAX_LEVELS];
    long long box0[SC_MAX_LEVELS];              // first box of each level
    long long child0[SC_MAX_LEVELS];            // level l >= 1 (0-based): its (nbox[l]+1) offsets start here
    double min_area[SC_MAX_LEVELS];             // a box is valid when its area >= min_area (cover * L^2)
    int blk0[SC_MAX_LEVELS + 2];
};

// Fills *p; returns the scratch bytes launch_deform_scales needs (box sums + moment partials).
long long scale_plan(int levels, const long long* nbox, const double* min_area, int nedge, ScalePlan* p);
// tri (nT,3) buoy indices in hierarchy order; tri_off (nbox[0]+1) level-1 ranges; child_off the concatenated child
// ranges of levels >= 2; edges (nedge) f8 ascending.  Writes mom (levels+1, 4) f8 = sums of L_eff, eps_tot,
// eps_tot^2, eps_tot^3, hist (levels+1, 3, nedge+1) counts of eps_tot, |div|, shear, and, when out is not NULL,
// seven (nbox_all) f4 planes of box outputs.
cudaError_t launch_deform_scales(const ScalePlan& p, const int32_t* tri, const long long* tri_off,
                                 const long long* child_off, const pt* yx0, const int8_t* m0, const pt* yx1,
                                 const int8_t* m1, double dt, const double* edges, void* scratch, double* mom,
                                 int64_t* hist, float* out, cudaStream_t st);
// The same pass with the box counts in device memory (dnbox, levels); p.nbox then holds upper bounds of them, which
// fix the launch grids, the box record layout and the moment partials.
cudaError_t launch_deform_scales_devcount(const ScalePlan& p, const int32_t* tri, const long long* tri_off,
                                          const long long* child_off, const pt* yx0, const int8_t* m0, const pt* yx1,
                                          const int8_t* m1, double dt, const double* edges, void* scratch, double* mom,
                                          int64_t* hist, float* out, const long long* dnbox, cudaStream_t st);

// ---- coarse-grained deformation over a fixed Eulerian grid, rebuilt every window (st_deform_grid.cu) ----
constexpr int GR_MAX_SIDE = 1 << 20;           // level-1 cells a side

// Shapes of one grid pass (host only): per-level bounds, field offsets and the scratch layout, in bytes from the
// front of the scratch.  Layout (every region 256-byte aligned):
//   box    8 * sum(bound) f8 box records, level s at box0[s] (the ScalePlan's; as st_deform_scale.cu), then the
//          moment partials 4 * blk0[levels+1] f8;
//   planes 7 * sum(bound) f4 box outputs (k_scale_stats' planes over the bounds);
//   code   sum(bound) u64 Morton codes of the boxes' keys at their own level, level s at box0[s];
//   off    level-1 ranges of the sorted triangles (bound[0]+1) i8, then the child ranges of levels 2.. (bound+1 each);
//   nbin   1 i8, the number of binned triangles;
//   flag, pos  nT i4 run-head flags and their exclusive scan;
//   kin, kout  nT u64 sort keys;  vin, vout  nT i4 sort values (caller's triangle index);
//   tri    3 * nT i4, the binned triangles' rows in hierarchy order;
//   cub    temporary storage of the sort and the scans.
struct GridPlan {
    ScalePlan sp;                               // nbox = the bounds min(nT, nj_s * ni_s)
    long long nT;
    int levels, nj, ni, end_bit;
    int nj_s[SC_MAX_LEVELS], ni_s[SC_MAX_LEVELS];
    long long field0[SC_MAX_LEVELS + 1];        // f4 offset of each level's seven planes in the field buffer
    long long o_box, o_planes, o_code, o_off, o_nbin, o_flag, o_pos, o_kin, o_kout, o_vin, o_vout, o_tri, o_cub;
    size_t cub_bytes;
    long long bytes;
};

// Fills *g (shapes, layout without CUB's part); 0 on success, else the argument that is out of range.
const char* grid_plan(long long nT, int levels, int nj, int ni, const double* min_area, int nedge, GridPlan* g);
// CUB's temporary storage (a device query); completes g->cub_bytes and g->bytes.
cudaError_t grid_plan_cub(GridPlan* g);
// tri (nT,3) caller's triangle order; fields sum_s 7 nj_s ni_s f4; nbox (levels) i8 out.  upto < GR_STAGE_ALL
// stops after that stage (stage timing only: the outputs are then not written).
enum { GR_STAGE_KEY = 1, GR_STAGE_SORT = 2, GR_STAGE_SEGMENT = 3, GR_STAGE_ALL = 4 };
cudaError_t launch_deform_grid(const GridPlan& g, const int32_t* tri, const pt* yx0, const int8_t* m0, const pt* yx1,
                               const int8_t* m1, double dt, double oy, double ox, double L0, const double* edges,
                               void* scratch, double* mom, int64_t* hist, float* fields, long long* nbox,
                               int upto, cudaStream_t st);

// ---- pair dispersion over time lags, and its statistics (st_disperse.cu) ----
constexpr int DS_MAX_LAGS = 64;
constexpr int DS_MAX_CLASS_EDGES = 63;
constexpr size_t DS_MAX_SMEM = 227 * 1024;     // opt-in dynamic shared memory per block on sm_100

// The active origin rows of one call, passed by value: rows yx[o], m[o] at lag lag[o] (1..lags) before the closing row.
struct DispOrigins {
    int nact;
    const pt* yx[DS_MAX_LAGS];
    const int8_t* m[DS_MAX_LAGS];
    int lag[DS_MAX_LAGS];
};

// Launch grid (a function of nQ only), dynamic shared memory of k_disperse for nact active origins, and the scratch
// (block partials) a call with up to `lags` active origins needs.
int disp_grid(long long nQ);
size_t disp_smem(int nact, int ncedge, int nedge);
long long disp_scratch_bytes(long long nQ, int lags, int ncedge);
// pairs (nQ,2) buoy indices; hist (lags, ncedge+1, nedge+1) int64 and sums (lags, ncedge+1, 4) f8 [r0, dr, dr^2, dD2]
// are zeroed and then written for the active lags; out, if not NULL (one origin only), (4, nQ) f8 r0, r1, dr, dD2.
cudaError_t launch_dispersion(const DispOrigins& og, long long nQ, const int32_t* pairs, const pt* yx1,
                              const int8_t* m1, double dt, int lags, int ncedge, const double* r_edges, int nedge,
                              const double* bins, void* scratch, int64_t* hist, double* sums, double* out,
                              cudaStream_t st);

// ---- finite-size Lyapunov exponents of pairs: exit times between separation thresholds (st_fsle.cu) ----
constexpr int FS_MAX_THRESHOLDS = 64;
constexpr int FS_MAX_TAU_EDGES = 512;
constexpr int FS_MAX_SAMPLES = 65535;

// Dynamic shared memory of k_fsle and the length (int64 words) of its statistics buffer for K thresholds and ntau
// exit-time edges.
size_t fsle_smem(int K, int ntau);
long long fsle_stats_len(int K, int ntau);
// pairs (nQ,2) buoy indices; state (nQ,2) int32 {level, anchor}; sample t of the row yx, m; with yx0 != NULL the
// state is reset and the row yx0, m0 is sample t-1 first.  stats (fsle_stats_len) int64 is zeroed and then written.
cudaError_t launch_fsle(long long nQ, const int32_t* pairs, int32_t* state, const pt* yx, const int8_t* m, int t,
                        const pt* yx0, const int8_t* m0, int K, const double* deltas, int ntau,
                        const double* tau_edges, int64_t* stats, cudaStream_t st);

// ---- SI3 T-cell fields sampled along the buoy trajectories (st_sample.cu) ----
constexpr int SP_MAX_FIELDS = 16;

// cell (nP) the state's cells, mask (nP) the row mask, yx (nP) the f8 positions (bilinear only); T (Nj*Ni) the T-points
// [y,x] km (bilinear only); F nF planes of Nj*Ni f4 at `stride` floats; interp 0 cell, 1 bilinear; out (nF, nP) f4.
cudaError_t launch_sample(long long nP, int Nj, int Ni, const int2* cell, const int8_t* mask, const pt* yx,
                          const pt* T, const int8_t* tmask, const float* F, long long stride, int nF, int interp,
                          float* out, cudaStream_t st);

// ---- buoy transits between regions: connectivity state and statistics (st_connect.cu) ----
constexpr int CN_MAX_REGIONS = 31;
constexpr int CN_MAX_TAU_EDGES = 512;
constexpr int CN_MAX_SAMPLES = 65535;
constexpr size_t CN_MAX_SMEM = 48 * 1024;      // dynamic shared memory a block may have without opting in

// Dynamic shared memory of k_connect for R regions, and the length (int64 words) of its statistics buffer.
size_t connect_smem(int R);
long long connect_stats_len(int R, int ntau);
// labels (Nj*Ni) u8; cell (nP) cell words (bit 31 stripped on read); mask (nP) the row mask of sample t; state (nP,2)
// int32, reset when t = 0; stats (connect_stats_len) int64 is added to, never zeroed.
cudaError_t launch_connect(long long nP, int Nj, int Ni, const uint8_t* labels, int R, const int2* cell,
                           const int8_t* mask, int t, int32_t* state, int ntau, const double* tau_edges,
                           int64_t* stats, cudaStream_t st);

}  // namespace st
