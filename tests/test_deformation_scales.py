"""Buoy-triangle deformation coarse-grained over material boxes, and its per-scale statistics
(sitrack_b200.deform_scales, csrc/st_deform_scale.cu).

CPU: the oracle (oracle/deform_scale_ref.py) against closed forms and boundary line integrals, the BoxHierarchy
invariants, the oracle's histograms against a direct count, the writer and the CLI's argument checks.  GPU:
CoarseGrainedRates bit for bit against the oracle, TrackEngine.track(deform=dict(scales=...)) against the oracle on
the series the same call returns and across buoy storage orders, and the CLI end to end."""
import contextlib
import io
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import TRACK_CASES, engine_for

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

RDT = 3600.0
FILL = np.float32(-9999.0)


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def _lattice(n, d=3.0, jitter=0.6, hole=None, seed=1):
    """Jittered n x n lattice [y,x] km, two anticlockwise triangles per square; triangles whose centroid lies in the
    disk `hole` = (yc, xc, r) are dropped."""
    rng = np.random.default_rng(seed)
    jj, ii = np.divmod(np.arange(n * n, dtype=np.int64), n)
    yx = np.stack([jj * d, ii * d], 1) + rng.uniform(-jitter, jitter, (n * n, 2))
    a = (np.arange(n - 1)[:, None] * n + np.arange(n - 1)[None, :]).ravel()
    tri = np.empty((2 * a.size, 3), np.int64)
    tri[0::2] = np.stack([a, a + 1, a + n + 1], 1)
    tri[1::2] = np.stack([a, a + n + 1, a + n], 1)
    if hole is not None:
        c = yx[tri].mean(1)
        tri = tri[np.hypot(c[:, 0] - hole[0], c[:, 1] - hole[1]) > hole[2]]
    return yx, tri.astype(np.int32)


def _apply(M, yx):
    x, y = yx[:, 1], yx[:, 0]
    return np.stack([M[1, 0] * x + M[1, 1] * y, M[0, 0] * x + M[0, 1] * y], 1)


# ---- CPU: the oracle and the hierarchy ----------------------------------------------------------

@pytest.mark.parametrize("kind", ["rotation", "dilation", "shear", "general"])
def test_oracle_affine_drift_every_scale(kind):
    """p1 = M p0: the mid-time velocity is linear in position, so the line integral around any union of triangles is
    exact and every valid cell of every scale gives the gradient 2 (M - I)(M + I)^-1 / dt."""
    from oracle import deform_scale_ref as O
    yx0, tri = _lattice(50, hole=(75.0, 75.0, 20.0))
    dt = 6 * RDT / 86400.0
    th, s, g = 0.07, 1.03, 0.04
    M = dict(rotation=np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]]),
             dilation=np.array([[s, 0.0], [0.0, s]]),
             shear=np.array([[1.0 + g, 0.0], [0.0, 1.0 / (1.0 + g)]]) @ np.array([[1.0, g], [0.0, 1.0]]),
             general=np.array([[1.02, 0.03], [-0.05, 0.97]]))[kind]
    yx1 = _apply(M, yx0)
    one = np.ones(yx0.shape[0], np.int8)
    G = 2.0 * (M - np.eye(2)) @ np.linalg.inv(M + np.eye(2)) / dt
    H = O.hierarchy(yx0, tri, 9.0, 5)
    boxes, st = O.coarse_grain(yx0, yx1, one, one, tri, dt, H, L0=9.0)
    for b in boxes:
        S = b["S"][b["valid"]]
        assert S.shape[0] > 0
        got = S[:, 1:5] / S[:, :1]
        assert np.abs(got - G.ravel()).max() <= 1e-12 * np.abs(G).max()
    assert (st["n"] > 0).all() and st["n"][0] == tri.shape[0]


def test_oracle_box_sums_equal_boundary_line_integrals():
    """Non-affine drift: for every box of two levels, the summed line integral and twice the area equal those over
    the boundary edges of the union of its triangles (directed edges whose reverse is absent)."""
    from oracle import deform_scale_ref as O
    from oracle import deform_ref as R
    yx0, tri = _lattice(40, hole=(60.0, 60.0, 12.0))
    yx1 = yx0 + np.stack([np.sin(yx0[:, 1] / 20.0), np.cos(yx0[:, 0] / 15.0)], 1) * 0.8
    dt = 0.25
    one = np.ones(yx0.shape[0], np.int8)
    H = O.hierarchy(yx0, tri, 10.0, 2)
    boxes, _ = O.coarse_grain(yx0, yx1, one, one, tri, dt, H, L0=10.0)
    X, Y = 0.5 * (yx0[:, 1] + yx1[:, 1]), 0.5 * (yx0[:, 0] + yx1[:, 0])
    U = (yx1[:, 1] - yx0[:, 1]) / dt
    ts = tri[H["order"]]
    nbox = 0
    for lv, b in zip(H["levels"], boxes):
        for k in range(lv["off"].size - 1):
            sel = ts[lv["off"][k]:lv["off"][k + 1]]
            E = {(int(t[j]), int(t[(j + 1) % 3])) for t in sel for j in range(3)}
            bd = np.array([(i, j) for (i, j) in E if (j, i) not in E])
            i, j = bd[:, 0], bd[:, 1]
            c = (U[j] + U[i]) * (Y[j] - Y[i])
            a = X[i] * Y[j] - X[j] * Y[i]
            assert abs(b["S"][k, 1] - c.sum()) <= 1e-12 * np.abs(c).sum()
            assert abs(b["S"][k, 0] - a.sum()) <= 1e-12 * np.abs(a).sum()
            nbox += 1
    assert nbox > 30


def test_box_hierarchy_invariants():
    import sitrack_b200 as sit
    from oracle import deform_scale_ref as O
    yx, tri = _lattice(40, hole=(60.0, 60.0, 12.0))
    rng = np.random.default_rng(2)
    tri = tri[rng.permutation(tri.shape[0])]
    L0, levels = 7.0, 5
    H = sit.BoxHierarchy(yx, tri, L0, levels)
    nT = tri.shape[0]
    assert np.array_equal(np.sort(H.order), np.arange(nT))            # each triangle in exactly one level-1 box
    assert H.tri_off[0] == 0 and H.tri_off[-1] == nT and (np.diff(H.tri_off) > 0).all()
    c = np.stack([((yx[tri[:, 0], k] + yx[tri[:, 1], k]) + yx[tri[:, 2], k]) / 3.0 for k in (0, 1)], 1)
    origin = np.floor(c.min(0) / L0) * L0
    assert np.array_equal(H.origin, origin)
    key = np.floor((c - origin) / L0).astype(np.int64)
    box_of = np.repeat(np.arange(H.nbox[0]), np.diff(H.tri_off))
    assert np.array_equal(key[H.order], H.keys[0][box_of])           # keys are the floor of the centroid
    for s in range(levels):
        off = H.box_tri_off[s]
        assert off[0] == 0 and off[-1] == nT and (np.diff(off) > 0).all()
        assert np.unique(H.keys[s], axis=0).shape[0] == H.nbox[s]
        # contiguous ranges: within each range all triangles have the same level-s key
        bo = np.repeat(np.arange(H.nbox[s]), np.diff(off))
        assert np.array_equal(key[H.order] >> s, H.keys[s][bo])
        if s == 0:                                     # the caller's order within a level-1 box (a stable sort)
            same = bo[1:] == bo[:-1]
            assert (H.order[1:][same] > H.order[:-1][same]).all()
        if s:
            ch = H.child_off[s]
            assert ch[0] == 0 and ch[-1] == H.nbox[s - 1] and (np.diff(ch) >= 1).all() and (np.diff(ch) <= 4).all()
            par = np.repeat(np.arange(H.nbox[s]), np.diff(ch))
            assert np.array_equal(H.keys[s - 1] >> 1, H.keys[s][par])
            assert np.array_equal(off, np.r_[H.box_tri_off[s - 1][ch[:-1]], nT])
    assert np.array_equal(H.L_km, L0 * 2.0 ** np.arange(levels)) and np.array_equal(H.min_area, 0.5 * H.L_km ** 2)
    assert H.scale_km[0] == FILL and H.scale_km.shape == (levels + 1,)
    assert H.bin_edges.size == 61 and H.bin_edges[0] == 1e-5 and H.bin_edges[-1] == 10.0
    G = O.hierarchy(yx, tri, L0, levels)                               # the oracle builds the same hierarchy
    assert np.array_equal(G["order"], H.order)
    for s in range(levels):
        assert np.array_equal(G["levels"][s]["key"], H.keys[s]) and np.array_equal(G["levels"][s]["off"], H.box_tri_off[s])
    one = sit.BoxHierarchy(yx, tri, 1000.0, 2)
    assert one.nbox.tolist() == [1, 1] and np.array_equal(one.order, np.arange(nT))
    assert H.matches(tri, yx.shape[0]) and not H.matches(tri[::-1], yx.shape[0]) and not H.matches(tri, yx.shape[0] + 1)


@pytest.mark.parametrize("kw", [dict(L0_km=0.0), dict(L0_km=-3.0), dict(L0_km=np.nan), dict(levels=0),
                                dict(levels=21), dict(levels=2.5), dict(cover=0.0), dict(bins=[1.0, 1.0]),
                                dict(tri=[[0, 1, 10 ** 6]]), dict(tri=np.zeros((0, 3), np.int32))])
def test_box_hierarchy_rejects(kw):
    import sitrack_b200 as sit
    yx, tri = _lattice(8)
    a = dict(pYX=yx, tri=tri, L0_km=5.0, levels=3)
    a.update(kw)
    with pytest.raises(ValueError):
        sit.BoxHierarchy(**a)


def test_oracle_histograms_against_direct_count():
    from oracle import deform_scale_ref as O
    rng = np.random.default_rng(4)
    edges = O.DEFAULT_EDGES
    v = np.concatenate([10 ** rng.uniform(-7, 3, 3000), edges, [0.0, edges[0] * (1 - 1e-16), np.inf]])
    o = dict(total=v, divergence=-v[::-1], shear=v * 0.5, L_eff=np.ones_like(v))
    ok = rng.random(v.size) < 0.9
    st = O.cell_stats(o, ok, edges)
    for h, vals in zip(st["hist"], (v[ok], np.abs(-v[::-1])[ok], (v * 0.5)[ok])):
        direct = np.zeros(edges.size + 1, np.int64)
        for x in vals:
            direct[sum(1 for e in edges if e <= x)] += 1
        assert np.array_equal(h, direct)
    assert st["n"] == ok.sum() and st["hist"].sum(1).tolist() == [ok.sum()] * 3


def test_scaling_writer_npz(tmp_path):
    import sitrack_b200 as sit
    scale_km = np.array([-9999.0, 10.0, 20.0])
    edges = np.array([0.01, 0.1, 1.0])
    f = str(tmp_path / "s.npz")
    st = lambda jw: dict(n=np.array([4, 2, 0]), sum_L_eff=np.array([8.0, 2.0, 0.0]), sum_eps_tot=np.array([1.0, 0.5, 0.0]),
                         sum_eps_tot2=np.array([2.0, 1.0, 0.0]), sum_eps_tot3=np.array([4.0, 3.0, 0.0]),
                         hist_total=np.full((3, 4), jw), hist_divergence=np.ones((3, 4)), hist_shear=np.zeros((3, 4)))
    with quiet(sit.DeformationScalingWriter, f, 2, scale_km, edges) as w:
        for jw in range(2):
            w.write(jw, 100 + jw, 200 + jw, st(jw))
    z = np.load(f)
    assert z["time_start"].tolist() == [100, 101] and z["time_end"].dtype == np.int32
    assert np.array_equal(z["scale_km"], scale_km) and np.array_equal(z["bin_edges"], edges)
    assert z["n"].dtype == np.int64 and z["n"].tolist() == [[4, 2, 0]] * 2
    assert z["L_eff"][0].tolist() == [2.0, 1.0, -9999.0] and z["eps_tot3"][1].tolist() == [1.0, 1.5, -9999.0]
    assert z["eps_tot"].dtype == np.float64 and z["hist_total"].shape == (2, 3, 4) and z["hist_total"].dtype == np.int64
    assert z["hist_total"][1].tolist() == [[1] * 4] * 3
    for n in ("time_start", "scale_km", "bin_edges", "n", "L_eff", "eps_tot", "eps_tot2", "eps_tot3", "hist_total",
              "hist_divergence", "hist_shear"):
        assert str(z[n + "_units"])
    assert str(z["eps_tot2_units"]) == "day-2" and float(z["FillValue"]) == -9999.0


def _synth_argv(r, *extra):
    return ["si3_part_tracker.py", "-i", r["si3"], "-m", r["mesh"], "-s", r["seed"], "-F", "-N", "SYNTH4"] + list(extra)


@pytest.mark.parametrize("extra", [["--deform-scales", "75", "3"], ["--deform", "6", "--deform-scales", "0", "3"],
                                   ["--deform", "6", "--deform-scales", "75", "0"],
                                   ["--deform", "6", "--deform-scales", "75", "21"],
                                   ["--deform", "6", "--deform-scales", "75", "2.5"]])
def test_cli_deform_scales_argument_errors(tmp_path, monkeypatch, extra):
    """--deform-scales needs --deform, a positive L0 and 1..20 levels; each error is an ERROR line printed before
    anything is read or written."""
    import si3_part_tracker as cli
    monkeypatch.chdir(tmp_path)
    monkeypatch.setattr(sys, "argv", ["si3_part_tracker.py", "-i", "x.npz", "-m", "y.npz", "-s",
                                      "sitrack_seeding_nemoTsi3_19961215_00_HSS2.npz", "-F"] + extra)
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf), pytest.raises(SystemExit):
        cli.main()
    assert any(l.startswith("ERROR") and "--deform-scales" in l for l in buf.getvalue().splitlines())
    assert not os.listdir(tmp_path)


# ---- GPU ---------------------------------------------------------------------------------------

def _check_stats(got, ref, H):
    assert np.array_equal(got["n"], ref["n"]) and got["n"].dtype == np.int64
    for j, k in enumerate(("hist_total", "hist_divergence", "hist_shear")):
        assert np.array_equal(got[k], ref["hist"][:, j]), k
        assert np.array_equal(got[k].sum(1), got["n"])
    for j, k in enumerate(("sum_L_eff", "sum_eps_tot", "sum_eps_tot2", "sum_eps_tot3")):
        assert (np.abs(got[k] - ref["sums"][:, j]) <= 1e-11 * np.abs(ref["sums"][:, j])).all(), k
    assert np.array_equal(got["scale_km"], H.scale_km) and np.array_equal(got["bin_edges"], H.bin_edges)


def _check_vs_oracle(sit, yx0, yx1, m0, m1, tri, dt, L0, levels):
    from oracle import deform_scale_ref as O
    H = sit.BoxHierarchy(yx0, tri, L0, levels)
    boxes, st = sit.CoarseGrainedRates(yx0, yx1, m0, m1, H, dt)
    G = O.hierarchy(yx0, tri, L0, levels)
    rb, rs = O.coarse_grain(yx0, yx1, m0, m1, tri, dt, G, L0=L0, edges=H.bin_edges)
    assert len(boxes) == levels
    for s, (a, b) in enumerate(zip(boxes, rb)):
        assert np.array_equal(a["key"], b["key"])
        for k in O.BOX_NAMES:
            assert a[k].dtype == np.float32 and np.array_equal(a[k], b[k]), (s, k)
    _check_stats(st, rs, H)
    boxes2, st2 = sit.CoarseGrainedRates(yx0, yx1, m0, m1, H, dt)    # run to run: the same bits
    for k in st:
        assert np.array_equal(st[k], st2[k]), k
    for a, b in zip(boxes, boxes2):
        for k in O.BOX_NAMES:
            assert np.array_equal(a[k], b[k])
    return H, boxes, st


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TRACK_CASES))
def test_coarse_grained_vs_oracle_golden(sit, gold_track, name):
    T, _ = gold_track
    posC, mask = T[name + "_posC"], T[name + "_mask"]
    tri = sit.TriangulateCloud(T["pos0"])
    n = 0
    for k0, k1 in [(0, 6), (5, 29), (12, 48)]:
        _, _, st = _check_vs_oracle(sit, posC[k0], posC[k1], mask[k0], mask[k1], tri, (k1 - k0) * RDT / 86400.0,
                                    20.0, 5)
        n += st["n"]
    assert n[0] > 50 and n[1] > 5


@pytest.mark.gpu
def test_coarse_grained_vs_oracle_lattice(sit):
    """~200 k buoys: 2 % masked, some vertices moved across their neighbours (flipped triangles), a hole."""
    rng = np.random.default_rng(11)
    yx0, tri = _lattice(450, hole=(600.0, 700.0, 90.0), seed=3)
    nP = yx0.shape[0]
    yx1 = yx0 + 1.2 + np.stack([np.sin(yx0[:, 1] / 40.0), np.cos(yx0[:, 0] / 55.0)], 1) * 0.7
    jump = rng.choice(nP, 300, replace=False)
    yx1[jump] += rng.choice([-1.0, 1.0], (300, 2)) * 7.0
    m0 = (rng.random(nP) >= 0.02).astype(np.int8)
    m1 = (rng.random(nP) >= 0.02).astype(np.int8)
    H, boxes, st = _check_vs_oracle(sit, yx0, yx1, m0, m1, tri, 0.25, 12.0, 6)
    assert st["n"][0] < tri.shape[0] * 0.95 and (st["n"] > 0).all()
    assert (boxes[0]["total"] == FILL).any() and (boxes[0]["total"] != FILL).sum() > 1000


@pytest.mark.gpu
def test_coarse_grained_vs_oracle_box_sizes(sit):
    """Level-1 boxes of 1, 31, 32, 33, 64, 65 and several hundred triangles (lane counts around the warp width), and a
    top level of one box."""
    rng = np.random.default_rng(12)
    sizes = [1, 31, 32, 33, 64, 65, 417]
    yx, tri = [], []
    for b, n in enumerate(sizes):
        c = np.array([5.0, 10.0 * b + 5.0]) + rng.uniform(-3, 3, (n, 2))
        r = rng.uniform(0.2, 0.8, (n, 1))
        ang = rng.uniform(0, 2 * np.pi, (n, 1)) + np.array([0.0, 2.1, 4.2])
        p = np.stack([c[:, [0]] + r * np.sin(ang), c[:, [1]] + r * np.cos(ang)], -1).reshape(-1, 2)
        tri.append(np.arange(3 * n).reshape(n, 3) + sum(len(q) for q in yx))
        yx.append(p)
    yx0, tri = np.concatenate(yx), np.concatenate(tri).astype(np.int32)
    perm = rng.permutation(tri.shape[0])
    tri = tri[perm]
    yx1 = yx0 + rng.normal(0, 0.01, yx0.shape)
    one = np.ones(yx0.shape[0], np.int8)
    H = sit.BoxHierarchy(yx0, tri, 10.0, 4)
    assert sorted(np.diff(H.tri_off).tolist()) == sorted(sizes) and H.nbox[-1] == 1
    # small boxes: cover 0.5 of 10 km squares is not reached by these clusters, so compare the sums too
    _check_vs_oracle(sit, yx0, yx1, one, one, tri, 0.25, 10.0, 4)
    Hs = sit.BoxHierarchy(yx0, tri, 10.0, 4, cover=1e-4)
    from oracle import deform_scale_ref as O
    boxes, st = sit.CoarseGrainedRates(yx0, yx1, one, one, Hs, 0.25)
    rb, rs = O.coarse_grain(yx0, yx1, one, one, tri, 0.25, O.hierarchy(yx0, tri, 10.0, 4), cover=1e-4, L0=10.0)
    for a, b in zip(boxes, rb):
        assert (a["total"] != FILL).all()
        for k in O.BOX_NAMES:
            assert np.array_equal(a[k], b[k]), k
    _check_stats(st, rs, Hs)


def _engine_run(T, g, name, sort, rows, every, deform):
    c = TRACK_CASES[name]
    s = np.float32(c["scale"])
    nP = T["pos0"].shape[0]
    sh = np.random.default_rng(7).permutation(nP)
    pos0, cell0 = T["pos0"][sh], T["jiT0"][sh].astype(np.int32)
    first = T["win_first"][sh] if c["win"] else None
    last = T["win_last"][sh] if c["win"] else None
    eng = engine_for(g, uv_strategy=c["uv_strategy"], device=0)
    if sort == "dev":
        import torch
        tt = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a, np.int32)).cuda()
        eng.set_buoys_dev(torch.from_numpy(pos0).cuda(), torch.from_numpy(cell0).cuda(), tt(first), tt(last), sort=True)
        torch.cuda.synchronize()
    else:
        eng.set_buoys(pos0, cell0, first, last, sort=sort == "host")
    res = eng.track((s * T["U"], s * T["V"], T["IC"]), T["U"].shape[0], kstrt=c["kstrt"], pos0=pos0, rec_first=first,
                    row_dtype=rows, deform=deform)
    eng.close()
    return res, sh


@pytest.mark.gpu
@pytest.mark.parametrize("every", [6, 7])
@pytest.mark.parametrize("rows", ["f8", "f4"])
@pytest.mark.parametrize("name", ["uv1", "win"])
def test_track_deform_scales(torch, sit, gold_track, name, rows, every):
    """track(deform=dict(..., scales=H)): per-window statistics equal the oracle's on the series the call works on,
    with the same bits whether the buoys are stored in the caller's order or sorted on the host or the device; the
    per-triangle outputs are those of the same call without `scales`."""
    from oracle import deform_scale_ref as O
    T, g = gold_track
    sh = np.random.default_rng(7).permutation(T["pos0"].shape[0])
    pos0 = T["pos0"][sh]
    tri = sit.TriangulateCloud(pos0)
    H = sit.BoxHierarchy(pos0, tri, 20.0, 5)
    posC, mask = T[name + "_posC"][:, sh], T[name + "_mask"][:, sh]
    ref = O.coarse_grain_series(posC, mask, tri, every, RDT, O.hierarchy(pos0, tri, 20.0, 5), L0=20.0,
                                edges=H.bin_edges)
    first = None
    for sort in ("none", "host", "dev"):
        res, _ = _engine_run(T, g, name, sort, rows, every, dict(tri=tri, every=every, scales=H))
        plain, _ = _engine_run(T, g, name, sort, rows, every, dict(tri=tri, every=every))
        got = res["deform_scales"]
        assert len(got) == len(ref) == 48 // every
        for a, b in zip(got, ref):
            _check_stats(a, b, H)
        if first is None:
            first = got
        for a, b in zip(got, first):
            for k in a:
                assert np.array_equal(a[k], b[k]), (sort, k)
        assert "deform_scales" not in plain
        for a, b in zip(res["deform"], plain["deform"]):
            for k in sit.DEFORM_NAMES:
                assert np.array_equal(a[k], b[k]), (sort, k)
    assert sum(int(s["n"][1]) for s in first) > 10


@pytest.mark.gpu
def test_track_deform_scales_sink_and_wrong_mesh(torch, sit, gold_track):
    T, g = gold_track
    tri = sit.TriangulateCloud(T["pos0"])
    H = sit.BoxHierarchy(T["pos0"], tri, 20.0, 3)
    seen = []
    eng = engine_for(g, device=0)
    eng.set_buoys(T["pos0"], T["jiT0"].astype(np.int32))
    r = eng.track((T["U"], T["V"], T["IC"]), 48, sink=lambda *a: None,
                  deform=dict(tri=tri, every=12, scales=H, scale_sink=lambda w, st: seen.append((w, st))))
    assert [w for w, _ in seen] == [0, 1, 2, 3] and "deform_scales" not in r
    assert all(st["hist_total"].shape == (4, 62) for _, st in seen)
    eng.set_buoys(T["pos0"], T["jiT0"].astype(np.int32))
    with pytest.raises(ValueError):
        eng.track((T["U"], T["V"], T["IC"]), 48, sink=lambda *a: None,
                  deform=dict(tri=tri[::-1], every=12, scales=H))
    eng.close()


@pytest.mark.gpu
def test_cli_deform_scales_end_to_end(tmp_path, monkeypatch):
    """si3_part_tracker.py -F --deform 6 --deform-scales 75 3 on the 'small' synthetic case: the scaling file's
    variables, shapes and units; per-scale histogram totals equal n; values agree with the oracle applied to the
    tracking file's f4 rows; the tracking and per-triangle files are those of a run without --deform-scales."""
    import si3_part_tracker as cli
    from make_synth_case import write_case
    from oracle import deform_scale_ref as O
    r = write_case(str(tmp_path / "in"), grid="small", nrec=24, hss=3)
    runs = {}
    for tag, extra in (("plain", ["--deform", "6"]), ("scales", ["--deform", "6", "--deform-scales", "75", "3"])):
        d = tmp_path / tag
        d.mkdir()
        monkeypatch.chdir(d)
        monkeypatch.setattr(sys, "argv", _synth_argv(r, *extra))
        quiet(cli.main)
        runs[tag] = d / "nc"
    files = sorted(os.listdir(runs["plain"]))
    sfiles = [f for f in os.listdir(runs["scales"]) if "_deformation-scaling_" in f]
    assert sfiles == ["NEMO-SI3_SYNTH4_SYN00_deformation-scaling_nemoTsi3_idlSeed_19961215h00_19961216h00.npz"], sfiles
    assert sorted(set(os.listdir(runs["scales"])) - set(sfiles)) == files
    for f in files:                                     # tracking and per-triangle files do not change
        a, b = np.load(runs["plain"] / f), np.load(runs["scales"] / f)
        assert sorted(a.files) == sorted(b.files)
        for k in a.files:
            assert a[k].dtype == b[k].dtype and a[k].tobytes() == b[k].tobytes(), (f, k)
    trk = np.load(runs["plain"] / [f for f in files if "_tracking_" in f][0])
    dfm = np.load(runs["plain"] / [f for f in files if "_deformation_" in f][0])
    z = np.load(runs["scales"] / sfiles[0])
    S = 4
    assert z["scale_km"].tolist() == [-9999.0, 75.0, 150.0, 300.0] and z["bin_edges"].shape == (61,)
    assert z["time_start"].tolist() == dfm["time_start"].tolist() and z["time_end"].tolist() == dfm["time_end"].tolist()
    assert z["n"].shape == (4, S) and z["n"].dtype == np.int64
    for k in ("hist_total", "hist_divergence", "hist_shear"):
        assert z[k].shape == (4, S, 62) and z[k].dtype == np.int64 and np.array_equal(z[k].sum(2), z["n"])
    units = dict(time_start="seconds since 1970-01-01 00:00:00", scale_km="km", bin_edges="day-1", n="1",
                 L_eff="km", eps_tot="day-1", eps_tot2="day-2", eps_tot3="day-3", hist_total="1")
    for k, u in units.items():
        assert str(z[k + "_units"]) == u, k
    # the oracle on the tracking file's f4 rows: the device works on the f8 positions those rows round, so counts may
    # move by the few cells whose value sits within the rounding of a bin edge or of the cover threshold, and means
    # by the relative rounding of the rates (~1e-5 here); the bounds below are far wider than that and far narrower
    # than any change of definition
    yx = np.stack([trk["y_pos"], trk["x_pos"]], -1).astype(np.float64)
    tri = dfm["vertices"]
    G = O.hierarchy(yx[0], tri, 75.0, 3)
    assert (z["n"][:, 0] > 100).all() and (z["n"][:, 1] > 3).all()
    for w in range(4):
        _, ref = O.coarse_grain(yx[6 * w], yx[6 * w + 6], trk["mask"][6 * w], trk["mask"][6 * w + 6], tri,
                                0.25, G, L0=75.0)
        assert (np.abs(z["n"][w] - ref["n"]) <= 1 + ref["n"] // 100).all(), w
        for j, k in enumerate(("L_eff", "eps_tot", "eps_tot2", "eps_tot3")):
            m = ref["sums"][:, j] / np.maximum(ref["n"], 1)
            ok = ref["n"] > 0
            assert (np.abs(z[k][w][ok] - m[ok]) <= 1e-3 * np.abs(m[ok])).all(), (w, k)
        for j, k in enumerate(("hist_total", "hist_divergence", "hist_shear")):
            assert (np.abs(z[k][w] - ref["hist"][:, j]).sum(1) <= 2 + ref["n"] // 50).all(), (w, k)


@pytest.mark.gpu
def test_bench_deform_small():
    """tools/bench_deform.py end to end on a small lattice: exit 0, sample exactness and run-to-run identity."""
    import json
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_deform.py"), "--ny", "300", "--nx", "300",
                        "--seconds", "0.05"], stdout=subprocess.PIPE, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    sc = res["scales"]
    assert res["bit_identical_to_oracle_on_sample"] and sc["sample_boxes_bit_identical"] and sc["run_to_run_identical"]
