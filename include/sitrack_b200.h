/*
 * sitrack_b200.h -- C ABI of libsitrack_b200.so: the B200 (sm_100a) buoy-advection
 * hot path of stephanieleroux/sitrack behind plain pointers and sizes.
 *
 * The reference is pure Python and has no FFI of its own; each entry point below
 * names the reference code it replaces (paths relative to the upstream repo) and
 * is what a ctypes stub in the reference would bind (see INTEGRATION.md).
 *
 * Conventions
 *   - 2-D grids are row-major (Nj, Ni); coordinate pairs are [y, x] in km on
 *     NorthPolarStereo(central_longitude=-45, true_scale_latitude=70), or
 *     [lat, lon] in degrees; cell indices are {jT, iT} int32 pairs.
 *   - "host" pointers are ordinary (or pinned) CPU memory; "dev" pointers are
 *     CUDA device memory on the context's device (e.g. torch tensor data_ptr()).
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *   - every function returns 0 on success or a negative ST_E* code; the message is
 *     available from st_last_error().  Nothing here prints or exits (the reference
 *     prints 'ERROR ...' and calls exit(0); the Python wrappers keep that text).
 *   - entry points marked ASYNC only enqueue work on `stream`.
 *   - there is NO CPU fallback: without a CUDA device every call fails with
 *     ST_ECUDA.
 */
#ifndef SITRACK_B200_H
#define SITRACK_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ST_OK        0
#define ST_EINVAL   -1      /* bad argument                              */
#define ST_ECUDA    -2      /* CUDA runtime error / no device            */
#define ST_ESTATE   -3      /* call order (e.g. step before set_buoys)   */
#define ST_ENOMEM   -4

#define ST_ABI_VERSION 3

typedef struct st_ctx st_ctx;

int         st_abi_version(void);
/* Message of the last failure on this context; ctx may be NULL for st_create errors. */
const char *st_last_error(const st_ctx *ctx);

/* ---- context: static grid resident in HBM -------------------------------------------
 * Replaces the host arrays the tracker builds once per run:
 *   xYf,xXf (GetModelGrid, sitrack/ncio.py:22-63), xYv,xXv,xYu,xXu (GetModelUVGrid,
 *   ncio.py:66-92), imaskt, and the constants iUVstrategy (si3_part_tracker.py:37),
 *   rdt (:31) and rmin_conc (tracking.py:4).
 * All array arguments are host pointers, (Nj,Ni) each.                                  */
int  st_create(st_ctx **out, int device, int Nj, int Ni,
               const double *Yf, const double *Xf, const double *Yu, const double *Xu,
               const double *Yv, const double *Xv, const int8_t *tmask,
               int uv_strategy, double rdt, double rmin_conc);
void st_destroy(st_ctx *ctx);

/* Step-kernel variant, all bit-identical in their results:
 *   0 = 2 (default) k_advect_warp: persistent one-warp CTAs, every warp owns its tiles of 32 buoys and its own
 *     shared-memory queue of cell crossings; orientation filter for the inside test; 3 the same with the
 *     reference's inside test on every lane;
 *   1 k_advect_step_v1, the straightforward kernel (also SITRACK_B200_KERNEL=v1);
 *   4 k_advect_cert + k_walk, the certified two-kernel step: U/V pick and inside test decided from a 32-byte
 *     per-cell frame in f32 when provably equal to the reference's tests, the reference's own tests in a second
 *     dense kernel otherwise (csrc/st_cert.cuh; builds the frames on first use; measured slower than 0 on B200
 *     because the second kernel re-reads what the first had in registers -- kept as an A/B, DESIGN.md section 3b);
 *   5 variant 0 with the U/V pick of the common path taken from the certified cell frames of variant 4 (the four
 *     U/V-point gathers only for the ~3 % of lanes that do not certify); bit-identical, measured 4 % slower than 0;
 *   6-12 round-1 experiments, present only in -DST_EXPERIMENTS builds (ST_EINVAL otherwise).                  */
int  st_set_kernel_variant(st_ctx *ctx, int variant);

/* Polar-stereographic parameters of CartNPSkm2Geo1D (util.py:413: lat0=70, lon0=-45). */
int  st_set_projection(st_ctx *ctx, double lat_ts_deg, double lon0_deg);

/* ---- seeding: SeedInit (tracking.py:98-178) ------------------------------------------
 * st_set_locate_grid uploads platT, plonT, pResolKM (host, (Nj,Ni); resKM may be NULL)
 * and builds the coarse-bin spatial hash on the device.
 * st_seed_locate runs, per buoy, NearestPoint (locate.py:222-276 with
 * rd_found_km=2.5, max_itr=10) -> Survive (tracking.py:62-93, siconc ic0) ->
 * FindContainingCell (locate.py:280-330).  Host in/out:
 *   SG (nP,2) [lat,lon], SC (nP,2) [y,x]; ic0 (Nj,Ni) f4;
 *   cell (nP,2) containing cell, nearest (nP,2) nearest T-point or -1,-1 (nullable),
 *   keep (nP) SeedInit's kmask.  Compaction by `keep` is left to the caller.           */
int  st_set_locate_grid(st_ctx *ctx, const double *latT, const double *lonT, const double *resKM);
int  st_seed_locate(st_ctx *ctx, int64_t nP, const double *SG, const double *SC, const float *ic0,
                    int32_t *cell, int32_t *nearest, int8_t *keep);
/* The same with the near-tie report (SURVEY section 7; locate.py:253-266, util.py:85-103): CUDA's sin/cos/asin
 * and numpy's differ in the last ulp, so a nearest point or an acceptance decided by less than 1e-11 relative is
 * flagged for the caller to re-evaluate with numpy (sitrack_b200/engine.py does): flag (nP) bit 0 = the runner-up
 * is within 1e-11 of the nearest, bit 1 = the distance is within 1e-11 of the acceptance radius; first (nP) = flat
 * index of the nearest T-point before the acceptance test (-1 none in reach), second (nP) = flat index of the
 * runner-up when bit 0 is set, else -1.  flag may be NULL (then so must first and second).                    */
int  st_seed_locate_ex(st_ctx *ctx, int64_t nP, const double *SG, const double *SC, const float *ic0,
                       int32_t *cell, int32_t *nearest, int8_t *keep, int8_t *flag, int32_t *first, int32_t *second);
/* Same as st_seed_locate with device pointers, ASYNC on `stream` (ic0_dev (Nj,Ni) f4 on the device).      */
int  st_seed_locate_dev(st_ctx *ctx, int64_t nP, const double *SG_dev, const double *SC_dev,
                        const float *ic0_dev, int32_t *cell_dev, int32_t *nearest_dev, int8_t *keep_dev,
                        void *stream);
/* SeedInit's shrink to the kept buoys (tracking.py:166-178) on the device: pos (nP,2) f8 and cell (nP,2) i4 compacted
 * by keep (nP) i1 into out_pos / out_cell (capacity nP), order kept; *n_out = buoys kept.  Device pointers; synchronises
 * `stream` (the count comes back to the host).                                                             */
int  st_seed_compact_dev(st_ctx *ctx, int64_t nP, const double *pos_dev, const int32_t *cell_dev, const int8_t *keep_dev,
                         double *out_pos_dev, int32_t *out_cell_dev, int64_t *n_out, void *stream);
/* NearestPoint alone (locate.py:222-276; no ji_prv box).  Host in/out.
 * use_brute != 0 runs the reference's own whole-grid scan on the device instead of
 * the hash search (cross-check).                                                        */
int  st_nearest_point(st_ctx *ctx, int64_t n, const double *latlon, double rd_found_km, int max_itr,
                      int use_brute, int32_t *ji, double *dist_km);
/* FindContainingCell alone (locate.py:280-330) around given T-points.  Host in/out.    */
int  st_find_containing_cell(st_ctx *ctx, int64_t n, const double *yx, const int32_t *ji_near,
                             int32_t *cell, int8_t *found);

/* ---- buoy state (xPosC[jt], vJIt, iAlive; si3_part_tracker.py:324-344) ----------------
 * pos (nP,2) [y,x] km, cell (nP,2).  rec_first/rec_last (nP) are the per-buoy model
 * record windows z1stModelRec/zLstModelRec (:264-312); pass NULL for -F runs.  All
 * buoys start alive, except those whose cell lies outside [2,Nj-3] x [2,Ni-3] (Survive's first
 * test, tracking.py:73-76, would discontinue them on entry; the step gathers their stencil
 * unclamped): they start discontinued.  *_dev variants take device pointers and copy
 * device-to-device.  On the DEVICE a discontinued buoy also carries bit 31 in the jT word of
 * its cell (st_state_device_ptrs shows that encoding; st_get_state strips it).               */
int  st_set_buoys(st_ctx *ctx, int64_t nP, const double *pos, const int32_t *cell,
                  const int32_t *rec_first, const int32_t *rec_last);
int  st_set_buoys_dev(st_ctx *ctx, int64_t nP, const double *pos_dev, const int32_t *cell_dev,
                      const int32_t *rec_first_dev, const int32_t *rec_last_dev, void *stream);
int  st_get_state(st_ctx *ctx, double *pos, int32_t *cell, int8_t *alive);          /* host out, syncs */
int  st_state_device_ptrs(st_ctx *ctx, double **pos_dev, int32_t **cell_dev, int8_t **alive_dev);
int64_t st_num_buoys(const st_ctx *ctx);
/* Row chaining (off by default).  The reference keeps no separate position state: xPosC[jt] IS the
 * input of iteration jt and xPosC[jt+1] its output (si3_part_tracker.py:412,459-460).  With chaining
 * on, st_step does the same on the device: it reads the positions of the buoys that are alive from
 * the f8 out_yx_dev row of the PREVIOUS st_step (from the state on the first one) and stores the new
 * ones into the new row only -- 16 B per buoy-step less to write.  The caller promises that a row
 * handed to st_step stays intact until the next st_step on the same stream has run (the next step
 * may write into the same buffer: every buoy is read before it is written, by the same thread).  A
 * step that cannot chain (f4 rows, out_yx_dev NULL, per-buoy record windows, st_step_multi / _ext /
 * _gather, kernel variants 1 and 4) first brings the state up to date and then runs as without
 * chaining; so do st_get_state, st_state_device_ptrs (which then synchronise the device) and
 * st_set_row_chain(ctx, 0).  st_sync_state does it explicitly (ASYNC on `stream`), e.g. before the
 * last row buffer is released.  Results are bit-identical with and without chaining.             */
int  st_set_row_chain(st_ctx *ctx, int on);
int  st_sync_state(st_ctx *ctx, void *stream);

/* ---- hourly records (xUu, xVv, xIC; si3_part_tracker.py:372-374) ----------------------
 * A slot holds one record as three contiguous (Nj,Ni) f4 planes [u_ice | v_ice |
 * siconc] on the device plus a pinned host staging buffer of the same layout.
 * st_submit_record (ASYNC) copies staging -> device on `stream` with one
 * cudaMemcpyAsync; double-buffer with two slots and a copy stream to overlap the
 * next record's transfer with the current step.                                          */
int  st_record_slots(st_ctx *ctx, int nslots);
int  st_record_host_buffer(st_ctx *ctx, int slot, float **staging);       /* 3*Nj*Ni floats, pinned */
int  st_record_device_buffer(st_ctx *ctx, int slot, float **dev);         /* 3*Nj*Ni floats         */
int  st_submit_record(st_ctx *ctx, int slot, void *stream);
/* ASYNC copy of a whole record [u|v|ic] (3*Nj*Ni f4) from caller-owned host memory
 * (pinned for a truly asynchronous copy) into the slot's device buffer.               */
int  st_upload_record(st_ctx *ctx, int slot, const float *host_rec, void *stream);

/* ---- the step: body of the records x buoys loop (si3_part_tracker.py:378-493) ----------
 * ASYNC.  Advances every alive buoy whose window contains file record `jrec` using
 * the record in `slot`, updates the state in place and writes trajectory row jt+1:
 *   out_yx_dev (nP,2) -> xPosC[jt+1], out_latlon_dev (nP,2) -> xPosG[jt+1],
 *   out_mask_dev (nP) -> xmask[jt+1,:,0]; rows of buoys that did not move get -9999 /
 *   mask 0 (lat/lon of -9999 is converted like the reference does, :493).
 *   n_alive_dev: uint64 counter incremented by the number of buoys alive at the START
 *   of the record (:376); zero it first.  Any output pointer may be NULL.               */
int  st_step(st_ctx *ctx, int slot, int jrec, double *out_yx_dev, double *out_latlon_dev,
             int8_t *out_mask_dev, uint64_t *n_alive_dev, void *stream);
/* nrec consecutive records already on the device at rec_dev (record k at
 * rec_dev + k*rec_stride floats, each [u|v|ic]); outputs (nrec,nP,..) row k at
 * k*out_stride elements; n_alive_dev (nrec).  One launch, ASYNC.                        */
int  st_step_multi(st_ctx *ctx, const float *rec_dev, int64_t rec_stride, int nrec, int jrec0,
                   double *out_yx_dev, double *out_latlon_dev, int8_t *out_mask_dev,
                   int64_t out_stride, uint64_t *n_alive_dev, void *stream);

/* Host-buffer form of one loop iteration -- what a reference-side binding calls per
 * record: copies u,v,ic (host, (Nj,Ni) f4 each) to the device, steps, and returns the
 * trajectory row in host arrays (any of them NULL to skip).  Synchronous.               */
int  st_track_record_host(st_ctx *ctx, int jrec, const float *u, const float *v, const float *ic,
                          double *out_yx, double *out_latlon, int8_t *out_mask, int64_t *n_alive);

/* ---- optional physics beyond the reference (default off) ----------------------------------
 * The reference takes ONE Euler step per record from a face velocity picked by two segment
 * tests and follows a buoy over at most ONE cell boundary (si3_part_tracker.py:423-484).
 * st_step_ext is st_step with the choice left to the caller:
 *   scheme   1 Euler, 2 midpoint Runge-Kutta, 4 classical Runge-Kutta (the record is frozen
 *            during the step: stages differ in space only);
 *   interp   0 the reference's pick (iUVstrategy of st_create), 1 C-grid linear (u between the
 *            west/east U-points of the host cell, v between its south/north V-points);
 *   max_hops cell boundaries a step or a stage may cross (>= 1); every cell entered must pass
 *            Survive (tracking.py:62-93).
 * State, records, kill rules, outputs and call protocol are those of st_step.  Results are NOT
 * comparable with the reference bit for bit, not even for (1, 0, 1): the Euler update is h*u
 * with h = rdt/1000 and the cell search is an orientation walk.  Validated against closed
 * forms in tests/test_ext_physics.py.                                                      */
int  st_step_ext(st_ctx *ctx, int slot, int jrec, int scheme, int interp, int max_hops,
                 double *out_yx_dev, double *out_latlon_dev, int8_t *out_mask_dev,
                 uint64_t *n_alive_dev, void *stream);

/* ---- rows in the output file's dtype ----------------------------------------------------
 * The reference keeps xPosC/xPosG as f8 in memory and casts to f4 when it writes the file
 * (sitrack/ncio.py:153-159: every trajectory variable is created 'f4').  These variants
 * write the trajectory row as (nP,2) f4 directly -- each value rounded once, to nearest even,
 * exactly like that cast -- so a caller that only feeds the writer moves 17 B per buoy off
 * the device instead of 33 B.  The buoy STATE stays f8 on the device; results of later
 * records are unaffected.  Same arguments and behaviour as the f8 forms otherwise.          */
int  st_step_f4(st_ctx *ctx, int slot, int jrec, float *out_yx_dev, float *out_latlon_dev,
                int8_t *out_mask_dev, uint64_t *n_alive_dev, void *stream);
int  st_step_multi_f4(st_ctx *ctx, const float *rec_dev, int64_t rec_stride, int nrec, int jrec0,
                      float *out_yx_dev, float *out_latlon_dev, int8_t *out_mask_dev,
                      int64_t out_stride, uint64_t *n_alive_dev, void *stream);
int  st_track_record_host_f4(st_ctx *ctx, int jrec, const float *u, const float *v, const float *ic,
                             float *out_yx, float *out_latlon, int8_t *out_mask, int64_t *n_alive);

/* ---- fused per-record all-gather of positions over peer memory (multi-GPU) ----------------
 * Buoys are sharded over ranks (one process per GPU; they never interact,
 * si3_part_tracker.py:378-488).  When every rank needs the whole xPosC[jt+1] row, the step
 * kernel itself stores each buoy's new position into the gathered (nP_total,2) array of EVERY
 * rank -- its own HBM plus the peer-mapped HBM of the others over NVLink -- so the transfer
 * overlaps the arithmetic thread by thread and no separate collective runs.
 *
 *   st_gather_create   allocates this rank's block (nbuf gathered arrays + a flag page) and
 *                      returns its 64-byte CUDA IPC handle; call after st_set_buoys.  `offset`
 *                      is the index of this rank's first buoy in the global order; f4 != 0
 *                      gathers (nP_total,2) f4 instead of f8.
 *   st_gather_connect_ipc   maps the other ranks' blocks; `handles` = world x 64 bytes in rank
 *                      order (exchange them with any host-side all-gather).
 *   st_gather_connect_ptrs  same for ranks living in ONE process (contexts on one device, or
 *                      on devices with peer access enabled): `blocks` = world device pointers
 *                      from st_gather_block.
 *   st_step_gather     ASYNC: st_step whose yx row goes to buffer `buf` of every rank.  `seq`
 *                      (1, 2, 3, ... per record) orders producers and consumers: before storing,
 *                      the stream waits until every rank has acknowledged sequence seq - nbuf;
 *                      after the kernel it releases ready[rank] = seq on every rank.
 *   st_gather_wait     ASYNC: `stream` waits until the rows of sequence `seq` from ALL ranks
 *                      have landed in this rank's buffer (st_gather_buffer).
 *   st_gather_ack      ASYNC: tells every rank this one is done reading sequence `seq`.
 *   st_gather_timed_out  1 if a device-side wait gave up after 10 s (a peer died); syncs.   */
#define ST_IPC_HANDLE_BYTES 64
int  st_gather_create(st_ctx *ctx, int rank, int world, int64_t nP_total, int64_t offset, int f4, int nbuf,
                      void *handle_out);
int  st_gather_connect_ipc(st_ctx *ctx, const void *handles);
int  st_gather_connect_ptrs(st_ctx *ctx, void *const *blocks);
int  st_gather_block(st_ctx *ctx, void **block_dev, int64_t *block_bytes);
int  st_gather_buffer(st_ctx *ctx, int buf, void **gathered_dev);
int  st_step_gather(st_ctx *ctx, int slot, int jrec, int buf, uint64_t seq, void *out_latlon_dev,
                    int8_t *out_mask_dev, uint64_t *n_alive_dev, void *stream);
int  st_gather_wait(st_ctx *ctx, uint64_t seq, void *stream);
int  st_gather_ack(st_ctx *ctx, uint64_t seq, void *stream);
int  st_gather_timed_out(st_ctx *ctx, int *timed_out);
/* How st_step_gather moves this rank's rows to the peers (default 0; all three deliver the same bytes):
 *   0  the step kernel stores every row into every peer's array itself (one 8- or 16-byte store per thread per peer);
 *   1  the step kernel writes this rank's block only, then one peer-to-peer cudaMemcpyAsync per peer runs on the
 *      copy engines (own streams) and the ready flags are released when they have landed;
 *   2  the step kernel stages each tile of 32 rows in shared memory and sends it to each peer with one
 *      cp.async.bulk (256 B as f4, 512 B as f8), peer order rotating with the tile.  Needs this rank's block to
 *      start on an even row (falls back to 0 otherwise).                                                  */
int  st_gather_set_mode(st_ctx *ctx, int mode);
int  st_gather_destroy(st_ctx *ctx);

/* ---- sea-ice deformation: strain rates of buoy triangles (RGPS-style) ---------------------
 * ASYNC.  For nT triangles tri_dev (nT,3) int32 (buoy indices, 16-byte aligned; each triangle anticlockwise
 * in the (x,y) plane) between two trajectory rows dt_days days apart -- positions yx0_dev, yx1_dev (nP,2) f8
 * [y,x] km and masks m0_dev, m1_dev (nP) i1 -- writes out_dev (6,nT) f4, one plane per output:
 *   divergence ux+vy, shear sqrt((ux-vy)^2+(uy+vx)^2), vorticity vx-uy [1/day], area [km^2, on the projection
 *   plane, at mid-time], y_ctr, x_ctr [km, mid-time centroid];
 * the velocity gradient is the line integral over the triangle's edges of the velocities (x1-x0)/dt at the
 * mid-time positions (x0+x1)/2 (Lindsay & Stern 2003).  A triangle with a vertex of mask 0 at either end, or a
 * signed area that is not positive at either end or at mid-time, gets -9999 in every output.  Computed in f8,
 * rounded once to f4; bit-identical to oracle/deform_ref.py (DESIGN.md section 10).  Indices are not
 * range-checked on the device.  ctx may be NULL: the current device, errors through st_last_error(NULL).     */
int  st_deform_dev(st_ctx *ctx, int64_t nT, const int32_t *tri_dev, const double *yx0_dev, const int8_t *m0_dev,
                   const double *yx1_dev, const int8_t *m1_dev, double dt_days, float *out_dev, void *stream);

/* ---- deformation coarse-grained over material boxes, and per-scale statistics ------------------
 * A hierarchy of `levels` (1..20) box levels over the nT triangles (DESIGN.md section 11, sit.BoxHierarchy):
 * tri_dev (nT,3) int32 is the mesh in hierarchy order (sorted by the Morton code of each triangle's level-1 box),
 * tri_off_dev (level_nbox[0]+1) int64 the level-1 boxes' ranges of it, child_off_dev the ranges of children of the
 * boxes of levels 2..levels, concatenated ((level_nbox[l]+1) each; may be NULL when levels = 1).  level_nbox and
 * min_area (HOST, levels): boxes per level and the area [km^2] from which a box counts (cover * L^2).
 * st_deform_scales_scratch_bytes gives the size of the scratch buffer st_deform_scales_dev needs (box sums and
 * moment partials); allocate it once per hierarchy.
 * ASYNC st_deform_scales_dev: between two rows dt_days apart (positions and masks as st_deform_dev), per box the sums
 * over its valid triangles of 2A and of the edge line integrals (f8, in a fixed order without atomics; an invalid
 * triangle adds +0.0); per box divergence, shear, vorticity, eps_tot = sqrt(div^2 + shear^2), L_eff = sqrt(area),
 * centroid.  Per scale s (0 = the triangles themselves, s = the boxes of level s):
 *   moments_dev (levels+1, 4) f8   sums of L_eff, eps_tot, eps_tot^2, eps_tot^3 over the valid cells;
 *   hist_dev (levels+1, 3, nedge+1) int64   counts of eps_tot, |div|, shear [1/day] binned on edges_dev (nedge f8,
 *                                           ascending) by searchsorted(edges, v, side="right").
 * boxes_dev, if not NULL, (7, sum level_nbox) f4 planes divergence, shear, vorticity, eps_tot, L_eff, y_ctr, x_ctr
 * of every box, -9999 where invalid.  Bit-identical to oracle/deform_scale_ref.py and run to run.  No host
 * synchronisation, no allocation; indices and ranges are not checked on the device.                          */
int  st_deform_scales_scratch_bytes(int64_t nT, int levels, const int64_t *level_nbox, const double *min_area,
                                    int nedge, int64_t *bytes);
int  st_deform_scales_dev(st_ctx *ctx, int64_t nT, const int32_t *tri_dev, const double *yx0_dev,
                          const int8_t *m0_dev, const double *yx1_dev, const int8_t *m1_dev, double dt_days,
                          int levels, const int64_t *level_nbox, const double *min_area, const int64_t *tri_off_dev,
                          const int64_t *child_off_dev, int nedge, const double *edges_dev, void *scratch_dev,
                          int64_t scratch_bytes, double *moments_dev, int64_t *hist_dev, float *boxes_dev,
                          void *stream);

/* ---- deformation coarse-grained over a fixed Eulerian grid, rebuilt every window ----------------
 * A grid of nj x ni (1..2^20 each) level-1 cells of side L0 km from the origin (oy, ox) km (DESIGN.md section 12,
 * sit.EulerianGrid): cell (bj, bi) covers [oy + bj L0, oy + (bj+1) L0) x [ox + bi L0, ox + (bi+1) L0); level s
 * (1..levels, levels 1..20) has side L0 2^(s-1), key (bj, bi) >> (s-1), nj_s = ((nj-1) >> (s-1)) + 1 rows and ni_s
 * likewise.  tri_dev (nT,3) int32 is the mesh in the caller's triangle order (buoy indices as stored on the device).
 * st_deform_grid_scratch_bytes gives the scratch st_deform_grid_dev needs (box records, moment partials, sort
 * buffers, CUB's temporary storage, segmentation arrays); it checks its arguments before any CUDA call and then
 * needs a device (CUB's size query).
 * ASYNC st_deform_grid_dev: between two rows dt_days apart (positions and masks as st_deform_dev) a triangle is binned
 * when it is valid by st_deform_dev's rule and its mid-time centroid lies in the grid (floor((Yc - oy)/L0) in
 * [0, nj) compared in f8; NaN and inf never are).  Binned triangles are sorted stably by the Morton code of their
 * level-1 key (ties in the caller's order) on the device; each level's boxes are the runs of that order, and the
 * sums, box outputs, cover rule (area >= min_area[s], HOST (levels)), moments_dev and hist_dev are those of
 * st_deform_scales_dev over these boxes (scale 0 = the binned triangles).  fields_dev (sum_s 7 nj_s ni_s) f4: per
 * level, seven (nj_s, ni_s) planes divergence, shear, vorticity, eps_tot, L_eff, y_ctr, x_ctr, -9999 where a cell
 * has no binned triangle or does not count; nbox_dev (levels) int64 the boxes per level.  The front of the scratch
 * holds the f8 box records (8 doubles per box: a2, Nux, Nuy, Nvx, Nvy, NY, NX, pad), level s from the prefix sum of
 * the bounds min(nT, nj_s ni_s).  Launch shapes depend on (nT, nj, ni, levels) only: bit-identical run to run.  No
 * host synchronisation, no allocation; indices are not checked on the device.  Refuses nT < 1, dt_days <= 0 or
 * NaN, a non-finite origin, L0 <= 0 and writes nothing then.                                               */
int  st_deform_grid_scratch_bytes(int64_t nT, int levels, int nj, int ni, int nedge, int64_t *bytes);
int  st_deform_grid_dev(st_ctx *ctx, int64_t nT, const int32_t *tri_dev, const double *yx0_dev, const int8_t *m0_dev,
                        const double *yx1_dev, const int8_t *m1_dev, double dt_days, int levels, int nj, int ni,
                        double oy, double ox, double L0, const double *min_area, int nedge, const double *edges_dev,
                        void *scratch_dev, int64_t scratch_bytes, double *moments_dev, int64_t *hist_dev,
                        float *fields_dev, int64_t *nbox_dev, void *stream);
/* The same pass stopped after stage `upto` (1 cell keys, 2 sort, 3 segmentation, 4 everything = st_deform_grid_dev),
 * for timing the stages with events; below 4 the outputs are not written.                                   */
int  st_deform_grid_stages_dev(st_ctx *ctx, int64_t nT, const int32_t *tri_dev, const double *yx0_dev,
                               const int8_t *m0_dev, const double *yx1_dev, const int8_t *m1_dev, double dt_days,
                               int levels, int nj, int ni, double oy, double ox, double L0, const double *min_area,
                               int nedge, const double *edges_dev, void *scratch_dev, int64_t scratch_bytes,
                               double *moments_dev, int64_t *hist_dev, float *fields_dev, int64_t *nbox_dev, int upto,
                               void *stream);

/* ---- two-particle (pair) dispersion over time lags, and per-(lag, class) statistics ----------
 * nQ (1..2^31-1) pairs pairs_dev (nQ,2) int32 of buoy indices (8-byte aligned; not range-checked on the device) between
 * the closing row yx1_dev, m1_dev and nact origin rows yx0[o], m0[o] (HOST arrays of device pointers) that lie lag[o]
 * (HOST, distinct, 1..lags) steps of dt_days days before it (DESIGN.md section 13, oracle/dispersion_ref.py).  Per pair
 * and origin, valid when both buoys have mask != 0 in both rows, in f8: r0 = |p_a - p_b| at the origin, r1 at the
 * closing row, dr = r1 - r0, dD2 = |(p_a - p_b)_1 - (p_a - p_b)_0|^2, stretch rate s = |dr| / (r0 lag dt_days) [day-1];
 * separation class searchsorted(r_edges, r0, side="right") over nclass_edges (1..63) ascending f8 edges, stretch bin
 * the same over nedge (1..4096) bins.  Outputs, zeroed and then written for the active lags only:
 *   hist_dev (lags, nclass_edges+1, nedge+1) int64   counts of s (exact);
 *   sums_dev (lags, nclass_edges+1, 4) f8            sums of r0, dr, dr^2, dD2 over the valid pairs;
 *   per_pair_dev, if not NULL (nact = 1 only), (4, nQ) f8 r0, r1, dr, dD2, -9999 for invalid pairs.
 * The sums use no floating-point atomics and a launch grid that depends on nQ only: bit-identical run to run and
 * between one call over several origins and one call per origin.  The shared-memory counters limit the shapes:
 * nact (nclass_edges+1)(nedge+1) ints plus (nclass_edges + nedge + 4 (nclass_edges+1)(nact + 16)) doubles must fit in
 * 227 KB.  st_dispersion_scratch_bytes checks (nQ, lags, classes, bins) for nact = lags on the host, before any CUDA
 * call, and gives the scratch (block partials) to allocate once.  ASYNC st_dispersion_dev: no host synchronisation,
 * no allocation; refuses nQ < 1, dt_days <= 0 or NaN, nact outside 1..lags and shapes past the limit, and writes
 * nothing then.                                                                                               */
int  st_dispersion_scratch_bytes(int64_t nQ, int lags, int nclass_edges, int nedge, int64_t *bytes);
int  st_dispersion_dev(st_ctx *ctx, int64_t nQ, const int32_t *pairs_dev, const double *yx1_dev, const int8_t *m1_dev,
                       int nact, const double *const *yx0, const int8_t *const *m0, const int *lag, double dt_days,
                       int lags, int nclass_edges, const double *r_edges_dev, int nedge, const double *bins_dev,
                       void *scratch_dev, int64_t scratch_bytes, int64_t *hist_dev, double *sums_dev,
                       double *per_pair_dev, void *stream);

/* ---- finite-size Lyapunov exponents of pairs: exit times between separation thresholds ----
 * nQ (1..2^31-1) pairs pairs_dev (nQ,2) int32 of buoy indices (8-byte aligned; not range-checked on the device), one
 * sample t (1..65535) per call: the row yx_dev, m_dev (DESIGN.md section 14, oracle/fsle_ref.py).  Per pair and sample,
 * in f8 and in this order: dy = y_a - y_b, dx = x_a - x_b, r = sqrt(dy*dy + dx*dx); the sample is valid when both
 * masks are != 0 and r is finite; b = searchsorted(deltas, r, side="right") over nthr (2..64) positive, strictly
 * increasing f8 thresholds deltas_dev, so a tie reaches the threshold.
 * state_dev (nQ,2) int32 {level, anchor} in the caller's pair order (8-byte aligned): level -1 not started, -2 ended,
 * 0..nthr thresholds reached; anchor the sample at which that level was first reached, -1 when unknown.  Update:
 *   not started, valid:    level = b, anchor = -1, n_start[b] += 1 (a pair starting above delta_j is not timed there);
 *   not started, invalid:  nothing;
 *   started, invalid:      level = -2; n_censored[level-1] += 1 when anchor >= 0 and level < nthr;
 *   started, valid, b > level: record tau = t - anchor for transition level-1 when level >= 1 and anchor >= 0, record
 *                          tau = 0 for transitions level .. b-2, then anchor = t, level = b (levels never go down).
 * Recording tau for transition j (0..nthr-2) adds 1 to hist_tau[j][searchsorted(tau_edges, tau, side="right")], tau to
 * sum_tau[j] and tau^2 to sum_tau2[j]; tau_edges_dev holds ntau_edges (1..512) ascending f8 edges in samples.
 * With yx_start_dev, m_start_dev (both or neither) the call first resets every pair to not started and evaluates the
 * start row as sample t-1, then the row as sample t: the first call of a run, with row 0 as the start row.
 * stats_dev, one int64 buffer (8-byte aligned), zeroed and then written with the events of this call, in this order:
 *   n_start (nthr+1) | hist_tau (nthr-1, ntau_edges+1) | sum_tau (nthr-1) | sum_tau2 (nthr-1) | n_censored (nthr-1),
 * nthr+1 + (nthr-1)(ntau_edges+4) words.  Integer atomics only: exact, independent of the launch grid, the device and
 * the buoy storage order.  Sample indices up to 65535 keep sum_tau2 below 2^63.  The shared-memory counters need
 * 8 (nthr + ntau_edges + 2 (nthr-1)) + 4 (nthr+1 + (nthr-1)(ntau_edges+2)) B of the 227 KB a block may have.
 * st_fsle_state_bytes checks (nQ, nthr, ntau_edges) on the host before any CUDA call and gives the size of state_dev.
 * ASYNC st_fsle_dev: no host synchronisation, no allocation; refuses nQ < 1, t outside 1..65535, shapes past the
 * limits, a NULL pointer, rows not 16-byte aligned and pairs, state, edges or stats not 8-byte aligned, and writes
 * nothing then.                                                                                                       */
int  st_fsle_state_bytes(int64_t nQ, int nthr, int ntau_edges, int64_t *bytes);
int  st_fsle_dev(st_ctx *ctx, int64_t nQ, const int32_t *pairs_dev, int32_t *state_dev, const double *yx_dev,
                 const int8_t *m_dev, int t, const double *yx_start_dev, const int8_t *m_start_dev, int nthr,
                 const double *deltas_dev, int ntau_edges, const double *tau_edges_dev, int64_t *stats_dev,
                 void *stream);

/* ---- SI3 T-cell fields sampled along the buoy trajectories (DESIGN.md section 15, oracle/sample_ref.py) ----
 * One row of the trajectory: for every buoy p of the context, its host cell (jT, iT) from the cell state (bit 31
 * stripped), its f8 position from yx_dev (nP,2) [y,x] km, or from the state when yx_dev is NULL (the chained row after
 * a chained step), and its row mask mask_dev (nP,) int8.  fields_dev holds nF (1..16) planes of Nj*Ni f4 (the T-cell
 * values of one record, e.g. siconc as plane 2 of a record slot), plane f at fields_dev + f * plane_stride floats
 * (plane_stride >= Nj*Ni).  out_dev (nF, nP) f4 gets, per field and buoy, in the caller's buoy order of the state:
 *   FillValue (-9999) when the mask is 0 or the cell lies outside 1..Nj-2 x 1..Ni-2;
 *   interp 0 (cell):      F[jT,iT], an exact copy;
 *   interp 1 (bilinear):  the T-quad on P's side of the grid lines T[jT-1,iT]->T[jT+1,iT] and T[jT,iT-1]->T[jT,iT+1]
 *     (f8 orientation tests, a point on a line goes to the higher index), the closed-form inverse bilinear (xi, eta)
 *     of P in it (k2 == 0: the parallelogram's linear root), clamped to [0,1]; corners SW, SE, NE, NW weighted
 *     (1-xi)(1-eta), xi(1-eta), xi eta, (1-xi) eta, those with tmask 0 or a non-finite value dropped and the rest
 *     renormalised in that order; no weight kept: the cell value.  f8 without FMA, rounded once to f4.
 *     tyx_dev (Nj*Ni,2) f8 [y,x] km are the T-points of a right-handed grid (i eastward, j northward: the quad pick
 *     reads "west" and "south" from the signs of the two orientation tests); the stencil reaches T[jT+-1, iT+-1].
 *   a non-finite result: FillValue.
 * ASYNC st_sample_dev: no host synchronisation, no allocation; refuses (before any CUDA call, writing nothing) a NULL
 * context, fields, mask or out, tyx NULL with interp 1, nF outside 1..16, plane_stride < Nj*Ni, interp other than 0
 * or 1, fields or out not 4-byte aligned and yx or tyx not 16-byte aligned.                                        */
int  st_sample_dev(st_ctx *ctx, int nF, const float *fields_dev, int64_t plane_stride, const double *yx_dev,
                   const int8_t *mask_dev, int interp, const double *tyx_dev, float *out_dev, void *stream);

/* ---- projections (util.py:394-472 via cartopy NorthPolarStereo) ------------------------ */
int  st_xy2latlon(int device, int64_t n, const double *yx, double *latlon, double lat_ts, double lon0);
int  st_latlon2xy(int device, int64_t n, const double *latlon, double *yx, double lat_ts, double lon0);
int  st_xy2latlon_dev(int64_t n, const double *yx_dev, double *latlon_dev, double lat_ts, double lon0,
                      void *stream);

/* ---- batched scalar predicates on explicit coordinates (host in/out) -------------------
 * st_intersect2seg : tracking.py:51-58, A,B,C,D (n,2)            -> out (n) 0/1
 * st_inside_quad   : locate.py:49-78,  yx (n,2), quads (n,4,2)   -> out (n) 0/1
 * st_cell_walk     : tracking.py:182-249; ring (n,12,2) = 4 cell vertices (BL,BR,UR,UL)
 *                    then F[jbl-1,ibl] F[jbr-1,ibr] F[jbr,ibr+1] F[jur,iur+1] F[jul+1,iul]
 *                    F[jur+1,iur] F[jul,iul-1] F[jbl,ibl-1]; kcross_in NULL => CrossedEdge
 *                    first, else NewHostCell for the given edge -> kcross (n), knhc (n)
 * st_survive       : tracking.py:62-93 on gathered stencils tm5 (n,5) i1, ic5 (n,5) f8 or
 *                    NULL (order [j,i] [j,i+1] [j+1,i] [j,i-1] [j-1,i-1])   -> kill (n)
 * st_haversine     : util.py:85-103, one point against n grid points       -> km (n)      */
int  st_intersect2seg(int device, int64_t n, const double *A, const double *B, const double *C,
                      const double *D, int8_t *out);
int  st_inside_quad(int device, int64_t n, const double *yx, const double *quads, int8_t *out);
int  st_cell_walk(int device, int64_t n, const double *p1, const double *p2, const double *ring,
                  const int32_t *kcross_in, int32_t *kcross, int32_t *knhc);
int  st_survive(int device, int64_t n, const int32_t *ji, int Nj, int Ni, const int8_t *tm5,
                const double *ic5, double rmin_conc, int32_t *kill);
int  st_haversine(int device, int64_t n, double plat, double plon, const double *lat, const double *lon,
                  double *out_km);

/* Diagnostics: the step kernel's own inverse projection (polynomial latitude above ~37N, table-
 * driven angles), host in/out like st_xy2latlon; tests compare it with the accurate kernel.   */
int  st_selftest_xy2latlon_fast(int device, int64_t n, const double *yx, double *latlon, double lat_ts, double lon0);

/* Diagnostics: the step kernel divides displacements by 1000 (si3_part_tracker.py:457-458)
 * with a reciprocal + exact-residual sequence; q_fast is that result, q_div the IEEE
 * division, for n host values a.                                                          */
/* The three projection kernels on an arbitrary ellipsoid (semi-major axis a_m [m], flattening f), so that they can be
 * pinned to published values that are not on WGS84 (tests/golden/proj_kat.json: Snyder 1987's worked example on
 * Clarke 1866, NSIDC's grid-corner table on Hughes 1980).  which = 0: inv_stere (st_xy2latlon), 1: inv_stere_fast
 * (the step kernel's), 2: fwd_stere (st_latlon2xy).  in/out are (n,2): [y,x] km <-> [lat,lon] degrees.            */
int  st_selftest_proj(int device, int which, int64_t n, const double *in, double *out, double lat_ts, double lon0,
                      double a_m, double f);

int  st_selftest_div1000(int device, int64_t n, const double *a, double *q_fast, double *q_div);
/* Same for the branch-free general division of the inside test (locate.py:72): q_fast = the
 * kernel's nine-operation sequence, q_div = IEEE division, for n host pairs a/b.            */
int  st_selftest_divide(int device, int64_t n, const double *a, const double *b, double *q_fast, double *q_div);

/* Diagnostics of the certified fast path of step variant 4 (csrc/st_cert.cuh).  The kernel decides the
 * U/V pick (si3_part_tracker.py:430-441) and "still inside its cell" (locate.py:49-78) from a per-cell affine
 * frame in f32 whenever the buoy is farther than proven margins from every line involved, and runs the
 * reference's own tests otherwise.
 *   st_cert_stats     cells admitted to the fast path / cells examined (0/0 when the grid has no frames).
 *   st_cert_frames    host copies of the frames ((Nj,Ni,8) f32: oy ox a b c d es et, es/et expanded from their bf16
 *                     storage) and of the packed margins ((Nj,Ni) u32: bf16(hin) << 16 | bf16(msep)); either may be NULL.
 *   st_selftest_cert  for n host triples (position yx (n,2), host cell (n,2), face velocities vel4 (n,4) f4 =
 *                     uL uR vB vT) returns flags (n) u8: bit0 pick certified, bit1 stay certified, bit2/bit3 the
 *                     certified llum1/llvm1, bit4/bit5 the reference's llum1/llvm1, bit6 the reference's
 *                     IsInsideQuadrangle of the reference's new position.                                        */
int  st_cert_stats(st_ctx *ctx, int64_t *admitted, int64_t *examined);
int  st_cert_frames(st_ctx *ctx, float *frames, uint32_t *margins);
int  st_selftest_cert(st_ctx *ctx, int64_t n, const double *yx, const int32_t *cell, const float *vel4,
                      uint8_t *flags);

#ifdef __cplusplus
}
#endif
#endif /* SITRACK_B200_H */
