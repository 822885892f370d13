#!/usr/bin/env python3
"""Generate tests/golden/*.npz by running the UNMODIFIED upstream sitrack
functions (imported from /root/reference, see ref_loader.py) on small synthetic
inputs.  Run in the build container:  python oracle/make_golden.py

TEST INFRASTRUCTURE ONLY.  The fixtures pin the C oracle (oracle/st_oracle.c),
the pure-Python port (oracle/pyport.py) and, through them, the CUDA kernels.

The record x buoy loop of the reference lives in the `__main__` block of
si3_part_tracker.py (:361-496) and cannot be imported; `ref_loop` below drives
it the same way -- same state arrays (xPosC, vJIt, VRTCS, vMesh, lStillIn,
iAlive), same call order -- and calls the reference's own intersect2Seg /
IsInsideQuadrangle / CrossedEdge / NewHostCell / UpdtInd4NewCell / Survive.
"""
import contextlib
import io
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import ref_loader            # noqa: E402
import synth                             # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
FILL = -9999.0


def ref_loop(sit, g, U, V, IC, pos0, vJIt0, VRTCS0, kstrt=0, first=None, last=None,
             iUVstrategy=1, rdt=3600.0):
    """si3_part_tracker.py:324-496 with the reference's functions; -F semantics when
    first/last are None.  Returns xPosC, xmask[:,:,0], jiT history, alive history."""
    xYf, xXf, xYu, xXu, xYv, xXv = (g[k] for k in ("Yf", "Xf", "Yu", "Xu", "Yv", "Xv"))
    imaskt = g["tmask"]
    Nt = U.shape[0]
    nP = pos0.shape[0]
    kstop = kstrt + Nt - 1
    z1st = np.zeros(nP, dtype=int) + kstrt if first is None else np.array(first, dtype=int)
    zLst = np.zeros(nP, dtype=int) + kstop if last is None else np.array(last, dtype=int)
    IDs = np.arange(nP) + 1
    vJIt = np.array(vJIt0, dtype=int).copy()
    VRTCS = np.array(VRTCS0, dtype=int).copy()
    iAlive = np.zeros(nP, dtype='i1') + 1
    xmask = np.zeros((Nt + 1, nP, 2), dtype='i1')
    xPosC = np.zeros((Nt + 1, nP, 2)) + FILL
    vMesh = np.zeros((nP, 4, 2))
    lStillIn = np.zeros(nP, dtype=bool)
    for jb in range(nP):
        k0 = z1st[jb] - kstrt
        xPosC[k0, jb, :] = pos0[jb, :]
        xmask[k0, jb, :] = 1
    jh = np.zeros((Nt + 1, nP, 2), np.int32); jh[0] = vJIt
    ah = np.zeros((Nt + 1, nP), np.int8); ah[0] = iAlive
    nal = np.zeros(Nt, np.int64)
    (Nj, Ni) = imaskt.shape
    xUu, xVv, xIC = np.zeros((Nj, Ni)), np.zeros((Nj, Ni)), np.zeros((Nj, Ni))
    for jt in range(Nt):
        jrec = jt + kstrt
        xIC[:, :] = IC[jt]; xUu[:, :] = U[jt]; xVv[:, :] = V[jt]        # f4 -> f8, as :372-374
        nal[jt] = iAlive.sum()
        for jP in range(nP):
            if iAlive[jP] == 1 and jrec >= z1st[jP] and jrec <= zLst[jP]:
                [ry, rx] = xPosC[jt, jP, :]
                if not lStillIn[jP]:
                    [[jbl, jbr, jur, jul], [ibl, ibr, iur, iul]] = VRTCS[jP, :, :]
                    vMesh[jP, :, :] = [[xYf[jbl, ibl], xXf[jbl, ibl]], [xYf[jbr, ibr], xXf[jbr, ibr]],
                                       [xYf[jur, iur], xXf[jur, iur]], [xYf[jul, iul], xXf[jul, iul]]]
                [jT, iT] = vJIt[jP, :]
                if iUVstrategy == 0:
                    zU = 0.5 * (xUu[jT, iT] + xUu[jT, iT - 1])
                    zV = 0.5 * (xVv[jT, iT] + xVv[jT - 1, iT])
                else:
                    Fpnt = [xYf[jT, iT], xXf[jT, iT]]
                    llum1 = sit.intersect2Seg([ry, rx], Fpnt, [xYv[jT - 1, iT], xXv[jT - 1, iT]], [xYv[jT, iT], xXv[jT, iT]])
                    llvm1 = sit.intersect2Seg([ry, rx], Fpnt, [xYu[jT, iT - 1], xXu[jT, iT - 1]], [xYu[jT, iT], xXu[jT, iT]])
                    zU = xUu[jT, iT - 1] if llum1 else xUu[jT, iT]
                    zV = xVv[jT - 1, iT] if llvm1 else xVv[jT, iT]
                dx = zU * rdt
                dy = zV * rdt
                rx_nxt = rx + dx / 1000.
                ry_nxt = ry + dy / 1000.
                xPosC[jt + 1, jP, :] = [ry_nxt, rx_nxt]
                xmask[jt + 1, jP, :] = [1, 1]
                lSI = sit.IsInsideQuadrangle(ry_nxt, rx_nxt, vMesh[jP, :, :])
                lStillIn[jP] = lSI
                if not lSI:
                    icross = sit.CrossedEdge([ry, rx], [ry_nxt, rx_nxt], VRTCS[jP, :, :], xYf, xXf)
                    inhc = sit.NewHostCell(icross, [ry, rx], [ry_nxt, rx_nxt], VRTCS[jP, :, :], xYf, xXf)
                    VRTCS[jP, :, :], vJIt[jP, :] = sit.UpdtInd4NewCell(inhc, VRTCS[jP, :, :], vJIt[jP, :])
                    icncl = sit.Survive(IDs[jP], vJIt[jP, :], imaskt, pIceC=xIC)
                    if icncl > 0:
                        iAlive[jP] = 0
        jh[jt + 1] = vJIt
        ah[jt + 1] = iAlive
    return xPosC, xmask[:, :, 0].copy(), jh, ah, nal


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def gold_predicates(sit):
    rng = np.random.default_rng(11)
    out = {}
    # the only known-answer vector upstream: tools/tests/test_pnt_inside_quad.py:16-24
    quad1 = np.array([[0., 0.], [3., 0.], [4., 4.], [1., 3.5]])
    pts1 = np.array([[2., 2.], [6., 6.], [-1., 2.], [3.1, 3.6]])
    out["kat_quad"] = quad1
    out["kat_pts"] = pts1
    out["kat_inside"] = np.array([sit.IsInsideQuadrangle(p[0], p[1], quad1) for p in pts1])
    # unit-square edge semantics + random quads
    sq = np.array([[0., 0.], [0., 1.], [1., 1.], [1., 0.]])        # [y,x]: BL, BR, UR, UL
    epts = np.array([[0., .5], [.5, 0.], [1., .5], [.5, 1.], [0., 0.], [1., 1.], [0., 1.], [1., 0.], [.5, .5]])
    out["sq_quad"], out["sq_pts"] = sq, epts
    out["sq_inside"] = np.array([sit.IsInsideQuadrangle(p[0], p[1], sq) for p in epts])
    n = 400
    quads = np.zeros((n, 4, 2))
    base = np.array([[0., 0.], [0., 1.], [1., 1.], [1., 0.]])
    for k in range(n):
        quads[k] = (base + 0.35 * rng.uniform(-1, 1, (4, 2))) * rng.uniform(1, 20) + rng.uniform(-50, 50, 2)
    pts = quads.mean(axis=1) + rng.uniform(-1.2, 1.2, (n, 2)) * (quads.max(axis=1) - quads.min(axis=1))
    # some points exactly on vertices / sharing a vertex ordinate (the half-open rules)
    pts[:40] = quads[:40, rng.integers(0, 4, 40)[0]]
    pts[40:80, 0] = quads[40:80, 1, 0]
    out["rq_quads"], out["rq_pts"] = quads, pts
    out["rq_inside"] = np.array([sit.IsInsideQuadrangle(pts[k, 0], pts[k, 1], quads[k]) for k in range(n)])
    # intersect2Seg: random, plus touching / collinear / shared end points on an integer lattice
    segs = rng.uniform(-5, 5, (600, 4, 2))
    segs[300:] = rng.integers(-2, 3, (300, 4, 2)).astype(float)
    out["seg_pts"] = segs
    out["seg_hit"] = np.array([sit.intersect2Seg(*[list(s[k]) for k in range(4)]) for s in segs])
    # Haversine samples (util.py:85-103) -- transcendental, compare with tolerance
    ll = np.stack([rng.uniform(50, 90, 64), rng.uniform(0, 360, 64)], 1)
    glat, glon = rng.uniform(50, 90, (8, 8)), rng.uniform(0, 360, (8, 8))
    out["hav_pts"], out["hav_glat"], out["hav_glon"] = ll, glat, glon
    out["hav_d"] = np.array([sit.Haversine(p[0], p[1], glat, glon) for p in ll])
    return out


def gold_walk(sit, g):
    """CrossedEdge / NewHostCell / Survive on grid cells with random displacement segments."""
    rng = np.random.default_rng(12)
    Nj, Ni = g["tmask"].shape
    n = 500
    jT = rng.integers(3, Nj - 3, n); iT = rng.integers(3, Ni - 3, n)
    p1 = np.zeros((n, 2)); p2 = np.zeros((n, 2))
    ce = np.zeros(n, np.int32); nh = np.zeros(n, np.int32)
    dxk = g["dx_km"]
    for k in range(n):
        y, x = g["warp"](jT[k] + rng.uniform(-.49, .49), iT[k] + rng.uniform(-.49, .49))
        p1[k] = [y, x]
        p2[k] = p1[k] + rng.uniform(-1.6, 1.6, 2) * dxk
        if k % 25 == 0:                      # straight through the UR corner -> diagonal (SURVEY §8c)
            p2[k] = 2.0 * np.array([g["Yf"][jT[k], iT[k]], g["Xf"][jT[k], iT[k]]]) - p1[k]
        V = np.array([[jT[k] - 1, jT[k] - 1, jT[k], jT[k]], [iT[k] - 1, iT[k], iT[k], iT[k] - 1]])
        ce[k] = sit.CrossedEdge(list(p1[k]), list(p2[k]), V, g["Yf"], g["Xf"])
        nh[k] = sit.NewHostCell(ce[k], list(p1[k]), list(p2[k]), V, g["Yf"], g["Xf"])
    return dict(walk_jT=jT, walk_iT=iT, walk_p1=p1, walk_p2=p2, walk_cross=ce, walk_newcell=nh)


def gold_survive(sit, g, ic):
    rng = np.random.default_rng(13)
    Nj, Ni = g["tmask"].shape
    n = 600
    jT = rng.integers(0, Nj, n); iT = rng.integers(0, Ni, n)
    jT[:8] = [0, 1, Nj - 2, Nj - 1, 5, 5, 5, 5]; iT[:8] = [5, 5, 5, 5, 0, 1, Ni - 2, Ni - 1]
    xic = np.zeros((Nj, Ni)); xic[:, :] = ic
    res = np.array([quiet(sit.Survive, 1, [jT[k], iT[k]], g["tmask"], pIceC=xic) for k in range(n)], np.int32)
    return dict(sv_jT=jT, sv_iT=iT, sv_kill=res)


def gold_host(sit):
    """host_ref.npz: inputs and answers of the host-side surface (tests/test_host_logic.py): time span, index
    update, seeding helpers, time strings.  The inputs are drawn as the tests drew them next to the imported
    reference; `sit` is the module whose answers are stored (main() passes the reference)."""
    rng = np.random.default_rng(0)
    out = {}
    t = 850608000 + 1800 + 3600 * np.arange(240)
    span = []
    for _ in range(50):
        seed = int(850608000 + rng.integers(0, 200) * 3600 + rng.integers(0, 3600))
        stop = int(seed + rng.integers(1, 30) * 3600) if rng.random() < 0.7 else 0           # 0: no iStop
        span.append([seed, stop] + [int(v) for v in quiet(sit.GetTimeSpan, 3600., t, seed, t[0], t[-1],
                                                            iStop=stop or None)])
    out["span"] = np.array(span, np.int64)                  # seed, stop -> Nt, kt0, ktN, itM0, itMN
    updt = [(rng.integers(5, 50, (2, 4)), rng.integers(5, 50, 2)) for _ in range(8)]
    out["updt_V"], out["updt_ji"] = np.array([u[0] for u in updt]), np.array([u[1] for u in updt])
    res = [sit.UpdtInd4NewCell(k + 1, V.copy(), ji.copy()) for k, (V, ji) in enumerate(updt)]
    out["updt_V_out"], out["updt_ji_out"] = np.array([r[0] for r in res]), np.array([r[1] for r in res])
    out["debug_seeding"] = sit.debugSeeding()
    x = rng.uniform(0, 360, 20)
    out["degE"], out["degWE"], out["degWE_270"] = x, sit.degE_to_degWE(x), sit.degE_to_degWE(270.)
    it = np.array([0, 850608000, 861494399]); prec = np.array(list("smhD"))
    out["clock_epoch"], out["clock_precision"] = it, prec
    out["clock"] = np.array([[sit.epoch2clock(int(a), precision=str(p)) for p in prec] for a in it])
    msk = (rng.random((40, 30)) > 0.2).astype('i1'); lat = rng.uniform(50, 90, (40, 30))
    lon = rng.uniform(0, 360, (40, 30)); ic = rng.random((40, 30))
    out.update(nemo_msk=msk, nemo_lat=lat, nemo_lon=lon, nemo_ic=ic)
    out["nemo_khss1"] = sit.nemoSeed(msk, lat, lon, ic, khss=1)
    out["nemo_khss3"] = sit.nemoSeed(msk, lat, lon, ic, khss=3)
    out["nemo_F"] = quiet(sit.nemoSeed, msk, lat, lon, ic, khss=1, platF=lat + 0.1, plonF=lon + 0.1)
    return out


def grid_arrays(g):
    keys = ["Yt", "Xt", "Yf", "Xf", "Yu", "Xu", "Yv", "Xv", "latT", "lonT", "tmask", "ResKM"]
    return {"g_" + k: g[k] for k in keys}


def main():
    sit = ref_loader.load()
    os.makedirs(GOLD, exist_ok=True)

    # ---- predicates ------------------------------------------------------------------
    tiny = synth.make_grid(**synth.GRID_PRESETS["tiny"], seed=0)
    U, V, IC = synth.make_records(tiny, 48, seed=1)
    pred = gold_predicates(sit)
    pred.update(gold_walk(sit, tiny))
    pred.update(gold_survive(sit, tiny, IC[7]))
    # NearestPoint threshold ladder (locate.py:259-266): resolkm=40 -> 20,24,28.8,...
    lad = [20.0]
    for _ in range(8):
        lad.append(1.2 * lad[-1])
    pred["np_ladder"] = np.array(lad)
    np.savez_compressed(os.path.join(GOLD, "predicates.npz"), **grid_arrays(tiny), **pred)

    # ---- seeding on the 'small' grid ---------------------------------------------------
    small = synth.make_grid(**synth.GRID_PRESETS["small"], seed=0)
    Us, Vs, ICs = synth.make_records(small, 2, seed=1)
    ids_h, SG_h, SC_h = synth.hss_seeds(small, ICs[0], khss=4)
    ids_s, SG_s, SC_s = synth.scattered_seeds(small, 160, seed=2)
    ids = np.concatenate([ids_h, ids_s + ids_h.size])
    SG = np.concatenate([SG_h, SG_s]); SC = np.concatenate([SC_h, SC_s])
    xic = np.zeros(small["tmask"].shape); xic[:, :] = ICs[0]
    nP, pSG, pSC, pIDs, zjiT, zJIvrt, iKeep = quiet(
        sit.SeedInit, ids.copy(), SG, SC, small["latT"], small["lonT"], small["Yf"], small["Xf"],
        small["ResKM"], small["tmask"], xIceConc=xic)
    near = np.array([quiet(sit.NearestPoint, (SG[k, 0], SG[k, 1]), small["latT"], small["lonT"],
                           rd_found_km=2.5, resolkm=small["ResKM"], max_itr=10) for k in range(SG.shape[0])])
    # FCC (locate.py:139-218), the geographic variant: T-centred cells whose vertices are F-points
    latF, lonF = synth.grid.km_to_latlon(small["Yf"], small["Xf"])
    lonF = np.mod(lonF, 360.)
    kk = [k for k in range(SG.shape[0]) if near[k][0] >= 3 and near[k][1] >= 3
          and near[k][0] < small["Nj"] - 3 and near[k][1] < small["Ni"] - 3][:60]
    fcc_ji, fcc_vrt = [], []
    for k in kk:
        ji, vr = quiet(sit.FCC, (SG[k, 0], SG[k, 1]), small["latT"], small["lonT"], latF, lonF, cellType='T',
                       rd_found_km=2.5, resolkm=small["ResKM"], max_itr=10)
        fcc_ji.append(ji); fcc_vrt.append(np.array(vr))
    np.savez_compressed(os.path.join(GOLD, "seedinit_small.npz"), **grid_arrays(small), ic0=ICs[0],
                        fcc_idx=np.array(kk), fcc_ji=np.array(fcc_ji), fcc_vrt=np.array(fcc_vrt), g_latF=latF, g_lonF=lonF,
                        ids=ids, SG=SG, SC=SC, out_nP=nP, out_SG=pSG, out_SC=pSC, out_IDs=pIDs,
                        out_jiT=zjiT, out_VRTCS=zJIvrt, out_iKeep=iKeep, out_nearest=near)
    print("seedinit_small: %d seeds -> %d kept" % (SG.shape[0], nP))

    # NearestPoint with the `ji_prv` local box (locate.py:241-244,255-256; FCC forwards it at :180): the box around a
    # previous guess is searched first, the whole domain only when that fails; note that the first radius is
    # 0.5*resolkm[jy,jx] with (jy,jx) the BOX-LOCAL indices of the box's argmin (upstream quirk, kept)
    rng = np.random.default_rng(21)
    nb_pt, nb_prv, nb_r, nb_out = [], [], [], []
    for k in range(SG.shape[0]):
        for rep in range(2):
            far = rng.random() < 0.3
            j0 = int(near[k][0]) if near[k][0] >= 0 else int(rng.integers(0, small["Nj"]))
            i0 = int(near[k][1]) if near[k][1] >= 0 else int(rng.integers(0, small["Ni"]))
            off = rng.integers(-25, 26, 2) if far else rng.integers(-4, 5, 2)
            jp = int(np.clip(j0 + off[0], 0, small["Nj"] - 1)); ip = int(np.clip(i0 + off[1], 0, small["Ni"] - 1))
            rbox = int(rng.choice([3, 10]))
            out = quiet(sit.NearestPoint, (SG[k, 0], SG[k, 1]), small["latT"], small["lonT"], rd_found_km=2.5,
                        resolkm=small["ResKM"], ji_prv=(jp, ip), np_box_r=rbox, max_itr=10)
            nb_pt.append(SG[k]); nb_prv.append((jp, ip)); nb_r.append(rbox); nb_out.append(out)
    np.savez_compressed(os.path.join(GOLD, "nearest_box.npz"), pt=np.array(nb_pt), ji_prv=np.array(nb_prv),
                        np_box_r=np.array(nb_r), out=np.array(nb_out))
    print("nearest_box: %d cases, %d not found" % (len(nb_out), int((np.array(nb_out)[:, 0] < 0).sum())))
    np.savez_compressed(os.path.join(GOLD, "host_ref.npz"), **gold_host(sit))

    # ---- tracking on the 'tiny' grid, 48 records ---------------------------------------
    ids_t, SG_t, SC_t = synth.hss_seeds(tiny, IC[0], khss=2)
    xic = np.zeros(tiny["tmask"].shape); xic[:, :] = IC[0]
    nPt, tSG, tSC, tIDs, tji, tV, tK = quiet(
        sit.SeedInit, ids_t.copy(), SG_t, SC_t, tiny["latT"], tiny["lonT"], tiny["Yf"], tiny["Xf"],
        tiny["ResKM"], tiny["tmask"], xIceConc=xic)
    print("track_tiny: %d buoys" % nPt)
    cases = {}
    # (a) as shipped: nearest U/V, -F
    cases["uv1"] = quiet(ref_loop, sit, tiny, U, V, IC, tSC, tji, tV)
    # (b) mean U/V (iUVstrategy=0)
    cases["uv0"] = quiet(ref_loop, sit, tiny, U, V, IC, tSC, tji, tV, iUVstrategy=0)
    # (c) 4x faster ice: multi-cell jumps, diagonal exits, many kills
    cases["fast"] = quiet(ref_loop, sit, tiny, 4 * U, 4 * V, IC, tSC, tji, tV)
    # (d) per-buoy record windows (no -F), file record offset kstrt=3
    rng = np.random.default_rng(5)
    first = 3 + rng.integers(0, 6, nPt); last = 3 + 47 - rng.integers(0, 10, nPt)
    cases["win"] = quiet(ref_loop, sit, tiny, U, V, IC, tSC, tji, tV, kstrt=3, first=first, last=last)
    save = dict(U=U, V=V, IC=IC, pos0=tSC, posG0=tSG, jiT0=tji, win_first=first, win_last=last)
    for name, (pc, mk, jh, ah, nal) in cases.items():
        save.update({name + "_posC": pc, name + "_mask": mk, name + "_jiT": jh, name + "_alive": ah,
                     name + "_nalive": nal})
        ncross = int((np.diff(jh, axis=0) != 0).any(axis=2).sum())
        print("  case %-5s alive at end %4d / %d, cell changes %d" % (name, ah[-1].sum(), nPt, ncross))
    np.savez_compressed(os.path.join(GOLD, "track_tiny.npz"), **grid_arrays(tiny), **save)
    for f in sorted(os.listdir(GOLD)):
        print("  %-24s %8.1f KB" % (f, os.path.getsize(os.path.join(GOLD, f)) / 1024))


if __name__ == "__main__":
    main()
