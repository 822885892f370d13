// st_warp.cuh -- k_advect_warp: the tuned step with every warp on its own.
//
// k_advect_persist keeps one walk queue per CTA: each tile costs a __syncthreads, a shared count per warp
// and a prefix over them (~45 warp instructions of bookkeeping per tile, 4 % of stall samples on the
// barrier).  Here the bookkeeping goes:
//   * a WARP owns its tiles of 32 buoys and its own shared-memory queue of crossings; appending is a
//     ballot + popc, draining (32 entries, every lane busy) needs a __syncwarp only -- no CTA barrier, no
//     counters; the alive count is one warp reduction and one atomic per warp at the end;
//   * FILT 1: the inside test of the common path is an orientation filter (inside_margin, st_advect.cu) that
//     certifies "inside" for lanes clear of every edge; the others are queued and the dense pass applies the
//     reference's own test before walking -- the exact test runs on ~15 % of the buoys instead of all;
//   * CB >= 0: every cell a live buoy can occupy carries the cell bits CB (st_create: cellbits_uniform), so the pick
//     and the filter take them from the instruction stream instead of gathering g.cellbits[c] per lane;
//   * the row-store mode is a template parameter (ROWS 0: f8 rows into local HBM; 1: f4 rows and/or
//     remote rows of the fused all-gather; 2: f8 rows that are also the position state, see BuoyState::pos_in),
//     so the default path carries no per-row mode branches.
// Arithmetic, store addresses and results are those of k_advect_persist / k_advect_step_v1, bit for bit.
#pragma once
#include "st_kernels.h"

namespace st {

// FILT 2 (variant 5): as FILT 1, and the U/V pick of the common path comes from the cell's certified frame
// (st_cert.cuh: k_cell_frames proves per cell that msep < |s|,|t| < hin  =>  llum1 = (s < 0), llvm1 = (t < 0)); the
// four U/V-point gathers and the two segment tests then run only for the ~1 % of lanes that are not certified.
__device__ __forceinline__ float4 ldg_frame(const float4* a)
{
    float4 r;
    asm("ld.global.nc.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;"
        : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(a), "l"(l2_keep_policy()));
    return r;
}

template <int UV, bool WIN, int ROWS, int FILT, int CB, int BLK, int MINB>
__global__ void __launch_bounds__(BLK, MINB)
k_advect_warp(const AdvectGrid g, const float* __restrict__ u, const float* __restrict__ v,
              const float* __restrict__ ic, BuoyState s, int jrec, StepOut o, int ntiles)
{
    constexpr int NW = BLK / 32, QCAP = 64;
    constexpr bool PEER = ROWS == 1, CHAIN = ROWS == 2;
    static_assert(!(CHAIN && WIN), "a buoy outside its record window has a fill row but a live position");
    const pt* __restrict__ pos_in = CHAIN ? s.pos_in : s.pos;
    __shared__ pt qP[NW][QCAP], qPn[NW][QCAP];
    __shared__ int2 qC[NW][QCAP];
    __shared__ unsigned qI[NW][QCAP];
    __shared__ __align__(128) double2 sRow[PEER ? NW : 1][PEER ? 32 : 1];    // tile staging of the bulk peer stores

    bool bulk_pending = false;                                              // lane 0: a bulk group may still read sRow

    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const unsigned lt = (1u << lane) - 1u;
    const int nwarps = (int)gridDim.x * NW;

    // buoy indices as 32-bit unsigned (the walk queue stores them so too; launch_advect_step refuses nP >= 2^32): one
    // IMAD.WIDE.U32 per address instead of 64-bit index arithmetic, ~25 instructions per tile less (215.2 -> 212.7 us)
    typedef unsigned idx_t;
    const idx_t nP_ = (idx_t)s.nP;
    auto load_state = [&](int tile, int8_t& al, pt& P, int2& c2) {
        const idx_t p = (idx_t)tile * 32 + lane;
        P.y = 0.0; P.x = 0.0;                                     // never used for a buoy that is not alive
        c2 = make_int2(ST_DEAD_BIT | 2, 2);
        if (tile < ntiles && p < nP_) {
            P = ld_stream_pt(pos_in + p);
            // evict-normal: the sector is still in L2 when a walk pass rewrites 8 bytes of it (a partial store into a
            // sector that has left L2 costs a DRAM read-modify-write, profiles/README.md round 2)
            c2 = __ldcg(s.cell + p);
        }
#ifdef ST_ALIVE_BYTE
        al = 0;
        if (tile < ntiles && p < nP_) al = __ldcs(s.alive + p);
#else
        al = (int8_t)(c2.x >= 0);                                 // bit 31 of jT = discontinued: `alive` is not read (24 B of state in)
#endif
    };
    auto walk_pass = [&](int lo, int n) {
        __syncwarp();                                             // queue entries of this warp visible
        if (lane < n) {
            const int e = lo + lane;
            int2 cc = qC[wid][e];
            const int j0 = cc.x, i0 = cc.y;
            int8_t a2 = 1;
            pt A, B;
            { const double2 q = *reinterpret_cast<const double2*>(&qP[wid][e]); A.y = q.x; A.x = q.y; }
            { const double2 q = *reinterpret_cast<const double2*>(&qPn[wid][e]); B.y = q.x; B.x = q.y; }
            const int Ni = g.Ni, c = cc.x * Ni + cc.y;
            ST_CHECK_CELL(c, 2 * Ni + 2, g.Nj, Ni);
            const pt bl = ldg_pt(g.F, c - Ni - 1), br = ldg_pt(g.F, c - Ni);
            const pt ul = ldg_pt(g.F, c - 1),      ur = ldg_pt(g.F, c);
            // queued as "not certainly inside" (FILT): the reference's test decides; the walk reuses its corners
            const bool out = !FILT || !inside_quad_flat(B.y, B.x, bl, br, ur, ul);
            if (out) {
                walk_cell_at(g, ic, A, B, c, bl, br, ur, ul, cc.x, cc.y, a2);
                const unsigned p = qI[wid][e];
                if (!a2) cc.x |= ST_DEAD_BIT;
                if (cc.x != j0 || cc.y != i0) __stcg(s.cell + p, cc);
                if (!a2) s.alive[p] = 0;
                if (CHAIN && !a2) st_stream_pt(s.pos + p, B);     // the rows from here on hold the fill value
            }
        }
        __syncwarp();                                             // slots may be overwritten again
    };

    int8_t al; pt P; int2 c2;
    const int tile0 = (int)blockIdx.x * NW + wid;
    load_state(tile0, al, P, c2);
    int qn = 0, my_alive = 0;
    for (int tile = tile0; tile < ntiles; tile += nwarps) {
        const idx_t p = (idx_t)tile * 32 + lane;
        const bool valid = p < nP_;
        // next tile's state: in flight while this tile is computed
        int8_t nal; pt nPt; int2 nc2;
        load_state(tile + nwarps, nal, nPt, nc2);

        my_alive += (al == 1);
        bool active = valid && al == 1;
        bool prestart = false;
        if (WIN && active) {
            const int f = s.rec_first[p], l = s.rec_last[p];
            prestart = (jrec + 1 == f);
            active = (jrec >= f) && (jrec <= l);
        }
        const int2 cw = active ? c2 : make_int2(2, 2);
        const int Ni = g.Ni;
        const int c = cw.x * Ni + cw.y;
        ST_CHECK_CELL(c, Ni + 1, g.Nj, Ni);
        const pt bl = ldg_pt(g.F, c - Ni - 1), br = ldg_pt(g.F, c - Ni);
        const pt ul = ldg_pt(g.F, c - 1),      ur = ldg_pt(g.F, c);
        double zU, zV;
        bool convex = true;                                       // FILT 2: bit 2 of the cell's orientation bits
        if (UV == 1 && FILT == 2) {
            const float4 f0 = ldg_frame(g.frames + 2 * (size_t)c), f1 = ldg_frame(g.frames + 2 * (size_t)c + 1);
            const float uL = __ldg(u + c - 1), uR = __ldg(u + c);
            const float vB = __ldg(v + c - Ni), vT = __ldg(v + c);
            // frame coordinates of P (st_cert.cuh: cert_eval): f0 = {oy, ox, a, b}, f1 = {c, d, hin|msep, es|et}
            const unsigned mw = __float_as_uint(f1.z), ew = __float_as_uint(f1.w);
            const float hin = __uint_as_float(mw & 0xffff0000u), msep = __uint_as_float(mw << 16);
            const float fy = __double2float_rn(__dsub_rn(P.y, (double)f0.x));
            const float fx = __double2float_rn(__dsub_rn(P.x, (double)f0.y));
            const float fs = __fmaf_rn(f0.z, fx, __fmaf_rn(f0.w, fy, __uint_as_float(ew & 0xffff0000u)));
            const float ft = __fmaf_rn(f1.x, fx, __fmaf_rn(f1.y, fy, __uint_as_float(ew << 16)));
            const float as = fabsf(fs), at = fabsf(ft);
            const bool pick_ok = (as < hin) & (at < hin) & (as > msep) & (at > msep);   // an admitted cell is convex (bit 2)
            bool llum1 = fs < 0.0f, llvm1 = ft < 0.0f;            // si3_part_tracker.py:430-431 when certified
            const bool need = active && !pick_ok;
            if (__any_sync(0xffffffffu, need)) {                  // the reference's own segment tests for the others
                if (need) {
                    const pt v0 = ldg_pt(g.V, c - Ni), v1 = ldg_pt(g.V, c);
                    const pt u0 = ldg_pt(g.U, c - 1),  u1 = ldg_pt(g.U, c);
                    const int cb = __ldg(g.cellbits + c);
                    llum1 = intersect2seg_pre(P, ur, v0, v1, cb & 1);
                    llvm1 = intersect2seg_pre(P, ur, u0, u1, cb & 2);
                    convex = (cb & 4) != 0;
                }
            }
            zU = (double)(llum1 ? uL : uR);
            zV = (double)(llvm1 ? vB : vT);
        } else if (UV == 1) {
            const pt v0 = ldg_pt(g.V, c - Ni), v1 = ldg_pt(g.V, c);
            const pt u0 = ldg_pt(g.U, c - 1),  u1 = ldg_pt(g.U, c);
            const float uL = __ldg(u + c - 1), uR = __ldg(u + c);
            const float vB = __ldg(v + c - Ni), vT = __ldg(v + c);
            const int cb = CB >= 0 ? CB : __ldg(g.cellbits + c);  // orientation of (ur,v0,v1) and (ur,u0,u1)
            const bool llum1 = intersect2seg_pre(P, ur, v0, v1, cb & 1);      // si3_part_tracker.py:430
            const bool llvm1 = intersect2seg_pre(P, ur, u0, u1, cb & 2);      // :431
            zU = (double)(llum1 ? uL : uR);
            zV = (double)(llvm1 ? vB : vT);
        } else {
            zU = __dmul_rn(0.5, __dadd_rn((double)__ldg(u + c), (double)__ldg(u + c - 1)));
            zV = __dmul_rn(0.5, __dadd_rn((double)__ldg(v + c), (double)__ldg(v + c - Ni)));
        }
        pt Pn;
        Pn.x = __dadd_rn(P.x, div1000(__dmul_rn(zU, g.rdt)));      // :452-458
        Pn.y = __dadd_rn(P.y, div1000(__dmul_rn(zV, g.rdt)));
        bool in;
        if (FILT == 2 && UV == 1) in = inside_margin(Pn.y, Pn.x, bl, br, ur, ul) && convex;
        else if (FILT) in = inside_margin(Pn.y, Pn.x, bl, br, ur, ul) && ((CB >= 0 ? CB : __ldg(g.cellbits + c)) & 4);   // same byte as the pick's
        else      in = inside_quad2(Pn.y, Pn.x, bl, br, ur, ul, active);
        const bool cross = active && !in;
        pt outp = {ST_FILL, ST_FILL};
        int8_t m = 0;
        if (active) {
            outp = Pn; m = 1;
            if (!CHAIN) st_stream_pt(s.pos + p, outp);
        } else if (WIN && prestart) {
            outp = P; m = 1;
        }
        if (valid) {
            if (!PEER) {
                if (o.yx) st_stream_pt(o.yx + p, outp);
            } else if (o.bulk && (long long)tile * 32 + 32 <= s.nP) {      // warp-uniform: a full tile
                // own block: plain row store; peers: the tile goes through shared memory and one bulk copy per peer
                put_row_pt(o.yx, p, outp, o.f4);
                if (lane == 0 && bulk_pending) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                __syncwarp();
                if (o.f4) reinterpret_cast<float2*>(sRow[wid])[lane] = make_float2(__double2float_rn(outp.y), __double2float_rn(outp.x));
                else      sRow[wid][lane] = make_double2(outp.y, outp.x);
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if (lane == 0) {
                    const unsigned bytes = o.f4 ? 256u : 512u;
                    const size_t at = (size_t)tile * bytes;
                    const uint32_t src = smem_u32(sRow[wid]);
                    // the peer order rotates with the tile, so that at any moment the warps of a GPU write to different peers
                    int k = tile % o.npeer;
#pragma unroll 1
                    for (int q = 0; q < o.npeer; ++q) {
                        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                                     ::"l"(reinterpret_cast<char*>(o.peer_yx[k]) + at), "r"(src), "r"(bytes) : "memory");
                        k = (k + 1 == o.npeer) ? 0 : k + 1;
                    }
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    bulk_pending = true;
                }
            } else {
                if (o.yx) put_row_yx(o, p, outp);
            }
            if (o.mask) __stcs(o.mask + p, m);
            if (o.latlon) {
                pt ll; ll.y = g.proj.fill_lat; ll.x = g.proj.fill_lon;            // :493 on a fill row
                if (m) ll = inv_stere_fast(outp, g.proj, g.atab);
                if (!PEER) st_stream_pt(o.latlon + p, ll);
                else           put_row_pt(o.latlon, p, ll, o.f4);
            }
        }
        // append this tile's crossings to the warp's queue (lane order)
        const unsigned bal = __ballot_sync(0xffffffffu, cross);
        if (cross) {
            const int e = qn + __popc(bal & lt);
            *reinterpret_cast<double2*>(&qP[wid][e]) = make_double2(P.y, P.x);
            *reinterpret_cast<double2*>(&qPn[wid][e]) = make_double2(outp.y, outp.x);
            qC[wid][e] = c2; qI[wid][e] = (unsigned)p;
        }
        qn += __popc(bal);
        if (qn >= 32) {                                            // warp-uniform
            qn -= 32;
            walk_pass(qn, 32);
        }
        al = nal; P = nPt; c2 = nc2;
    }
    if (PEER && lane == 0 && bulk_pending) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // the peers' rows have left
    walk_pass(0, qn);                                             // flush (qn < 32)
    if (o.n_alive) {
        const int wsum = __reduce_add_sync(0xffffffffu, my_alive);
        if (lane == 0 && wsum) atomicAdd(o.n_alive, (unsigned long long)wsum);
    }
}

}  // namespace st
