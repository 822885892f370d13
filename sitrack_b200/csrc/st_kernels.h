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
cudaError_t launch_cell_bits(const AdvectGrid& g, int8_t* bits, int* n_bad_coord, cudaStream_t st);
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

}  // namespace st
