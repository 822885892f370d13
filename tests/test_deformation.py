"""Sea-ice deformation of buoy triangles (sitrack_b200.deform, csrc/st_deform.cu).

CPU: the oracle (oracle/deform_ref.py) against closed forms, its validity rules, TriangulateCloud, the writer and the
CLI's argument checks.  GPU: k_deform bit for bit against the oracle on every vertex triple of the golden buoys,
TrackEngine.track(deform=...) against the oracle on the series the same call returns, and the CLI end to end."""
import contextlib
import io
import itertools
import os
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


def _random_triangles(rng, n, span=100.0, size=(5.0, 20.0)):
    """n anticlockwise triangles (3n buoys, yx (3n,2) [y,x] km) with a minimum angle of ~15 degrees."""
    c = rng.uniform(-span, span, (n, 2))
    r = rng.uniform(*size, (n, 1))
    ang = np.sort(rng.uniform(0, 2 * np.pi, (n, 3)), axis=1)
    ang = ang[:, [0]] + np.array([0.0, 2 * np.pi / 3, 4 * np.pi / 3]) + rng.uniform(-0.5, 0.5, (n, 3))
    x = c[:, [1]] + r * np.cos(ang)
    y = c[:, [0]] + r * np.sin(ang)                  # increasing angle = anticlockwise in (x, y)
    yx = np.stack([y.ravel(), x.ravel()], 1)
    return yx, np.arange(3 * n).reshape(n, 3)


def _apply(M, yx):
    x, y = yx[:, 1], yx[:, 0]
    return np.stack([M[1, 0] * x + M[1, 1] * y, M[0, 0] * x + M[0, 1] * y], 1)


# ---- CPU: the oracle ---------------------------------------------------------------------------

@pytest.mark.parametrize("kind", ["rotation", "dilation", "shear", "general"])
def test_oracle_affine_drift_closed_form(kind):
    """p1 = M p0 in (x, y): the mid-time velocity field is linear, the line integral exact, and every triangle gives
    the gradient 2 (M - I)(M + I)^-1 / dt."""
    from oracle import deform_ref as R
    rng = np.random.default_rng(3)
    yx0, tri = _random_triangles(rng, 2000)
    dt = 6 * RDT / 86400.0
    th, s, g = 0.07, 1.03, 0.04
    M = dict(rotation=np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]]),
             dilation=np.array([[s, 0.0], [0.0, s]]),
             shear=np.array([[1.0 + g, 0.0], [0.0, 1.0 / (1.0 + g)]]) @ np.array([[1.0, g], [0.0, 1.0]]),
             general=np.array([[1.02, 0.03], [-0.05, 0.97]]))[kind]
    yx1 = _apply(M, yx0)
    one = np.ones(yx0.shape[0], np.int8)
    r, valid = R.rates_f8(yx0, yx1, one, one, tri, dt)
    assert valid.all()
    G = 2.0 * (M - np.eye(2)) @ np.linalg.inv(M + np.eye(2)) / dt        # [[ux, uy], [vx, vy]]
    got = np.stack([r["ux"], r["uy"], r["vx"], r["vy"]], 1)
    assert np.abs(got - G.ravel()).max() <= 1e-12 * np.abs(G).max()
    out = R.deform(yx0, yx1, one, one, tri, dt)
    if kind == "rotation":
        assert np.abs(r["divergence"]).max() <= 1e-12 * np.abs(G).max()
        assert np.abs(r["shear"]).max() <= 1e-12 * np.abs(G).max()
        assert np.allclose(r["vorticity"], 4 * np.tan(th / 2) / dt, rtol=1e-12, atol=0)
    if kind == "dilation":
        assert np.allclose(r["divergence"], 4 * (s - 1) / ((s + 1) * dt), rtol=1e-12, atol=0)
        assert np.abs(r["shear"]).max() <= 1e-12 * np.abs(G).max()
        assert np.abs(r["vorticity"]).max() <= 1e-12 * np.abs(G).max()
    if kind == "shear":                              # area-preserving: no divergence to first order, shear > 0
        ux, uy, vx, vy = G.ravel()
        assert np.allclose(r["shear"], np.hypot(ux - vy, uy + vx), rtol=1e-12, atol=0) and np.hypot(ux - vy, uy + vx) > 0
    # the f4 outputs are the f8 values rounded once
    for k in R.NAMES:
        assert np.array_equal(out[k], r[k].astype(np.float32))
    # area and centroid of the mid-time triangle
    mid = 0.5 * (yx0 + yx1)
    y, x = mid[tri, 0], mid[tri, 1]
    A = 0.5 * ((x[:, 1] - x[:, 0]) * (y[:, 2] - y[:, 0]) - (x[:, 2] - x[:, 0]) * (y[:, 1] - y[:, 0]))
    assert np.allclose(r["area"], A, rtol=1e-10) and np.allclose(r["y_ctr"], y.mean(1), rtol=0, atol=1e-12)


def test_oracle_invalid_triangles_are_filled():
    from oracle import deform_ref as R
    yx0 = np.array([[0, 0], [0, 10], [10, 0],             # 0-2 a good triangle (y, x): (x,y) = (0,0) (10,0) (0,10)
                    [0, 0], [0, 10], [0, 20],              # 3-5 collinear
                    [50, 50], [50, 60], [60, 50]], float)  # 6-8 good at k0, flipped at k1
    yx1 = yx0 + 0.1
    yx1[8] = [40, 50]                                      # vertex 8 crosses the opposite edge
    tri = np.array([[0, 1, 2], [0, 2, 1], [3, 4, 5], [6, 7, 8], [0, 1, 2], [0, 1, 2]])
    m0 = np.ones(9, np.int8); m1 = np.ones(9, np.int8)
    out = R.deform(yx0, yx1, m0, m1, tri, 0.25)
    ok = np.array([True, False, False, False, True, True])
    for k in R.NAMES:
        assert (out[k][~ok] == FILL).all() and (out[k][ok] != FILL).all(), k
    m0[1] = 0
    out = R.deform(yx0, yx1, m0, m1, tri[:1], 0.25)
    assert all(out[k][0] == FILL for k in R.NAMES)
    m0[1] = 1; m1[2] = 0
    out = R.deform(yx0, yx1, m0, m1, tri[:1], 0.25)
    assert all(out[k][0] == FILL for k in R.NAMES)


def test_triangulate_cloud_on_a_lattice_with_a_hole():
    pytest.importorskip("scipy")
    import sitrack_b200 as sit
    rng = np.random.default_rng(5)
    d, R_hole = 10.0, 60.0
    jj, ii = np.mgrid[0:40, 0:40]
    yx = np.stack([jj.ravel() * d, ii.ravel() * d], 1) + rng.uniform(-0.2 * d, 0.2 * d, (1600, 2))
    c = np.array([200.0, 200.0])
    yx = yx[np.hypot(*(yx - c).T) > R_hole]
    tri = sit.TriangulateCloud(yx)
    assert tri.dtype == np.int32 and tri.ndim == 2 and tri.shape[1] == 3 and tri.shape[0] > 2000
    y, x = yx[tri, 0], yx[tri, 1]
    assert (((x[:, 1] - x[:, 0]) * (y[:, 2] - y[:, 0]) - (x[:, 2] - x[:, 0]) * (y[:, 1] - y[:, 0])) > 0).all()
    e = np.stack([yx[tri[:, (k + 1) % 3]] - yx[tri[:, k]] for k in range(3)], 1)
    L = np.sqrt((e * e).sum(-1))
    # the default cut is twice the median edge of the unfiltered mesh: well below the hole's width
    assert L.max() < 2 * R_hole / 3
    tri2 = sit.TriangulateCloud(yx, max_edge_km=12.0)
    e2 = np.stack([yx[tri2[:, (k + 1) % 3]] - yx[tri2[:, k]] for k in range(3)], 1)
    assert np.sqrt((e2 * e2).sum(-1)).max() <= 12.0 and 0 < tri2.shape[0] < tri.shape[0]
    # no triangle covers a point of the hole
    th = np.linspace(0, 2 * np.pi, 64, endpoint=False)
    probes = np.concatenate([[c], c + (R_hole - d) * np.stack([np.sin(th), np.cos(th)], 1)])
    for p in probes:
        ux, uy = x - p[1], y - p[0]
        cr = np.stack([ux[:, k] * uy[:, (k + 1) % 3] - uy[:, k] * ux[:, (k + 1) % 3] for k in range(3)], 1)
        assert not (cr >= 0).all(1).any()
    # no interior angle below MIN_ANGLE_DEG
    for k in range(3):
        a, b = -e[:, (k + 2) % 3], e[:, k]
        ang = np.degrees(np.arccos((a * b).sum(1) / (np.linalg.norm(a, axis=1) * np.linalg.norm(b, axis=1))))
        assert ang.min() >= sit.MIN_ANGLE_DEG - 1e-9


def test_deformation_writer_npz(tmp_path):
    import sitrack_b200 as sit
    tri = np.array([[0, 1, 2], [2, 1, 3]], np.int32)
    ids = np.array([10, 11, 12, 13], np.int64)
    f = str(tmp_path / "d.npz")
    with quiet(sit.DeformationWriter, f, 2, tri, ids) as w:
        for jw in range(2):
            w.write(jw, 100 + jw, 200 + jw, {n: np.full(2, jw + 0.5, np.float32) for n in sit.DEFORM_NAMES})
    z = np.load(f)
    assert np.array_equal(z["vertices"], tri) and z["vertices"].dtype == np.int32
    assert np.array_equal(z["id_vertices"], ids[tri]) and z["id_vertices"].dtype == np.int64
    assert z["time_start"].tolist() == [100, 101] and z["time_end"].dtype == np.int32
    for n in sit.DEFORM_NAMES:
        assert z[n].shape == (2, 2) and z[n].dtype == np.float32 and z[n][1, 0] == 1.5
        assert str(z[n + "_units"]) == sit.DEFORM_UNITS[n]
    assert z["FillValue"] == FILL


def _synth_argv(r, *extra):
    return ["si3_part_tracker.py", "-i", r["si3"], "-m", r["mesh"], "-s", r["seed"], "-F", "-N", "SYNTH4"] + list(extra)


@pytest.mark.parametrize("extra,env", [(["--deform", "1.5"], {}), (["--deform", "-1"], {}),
                                       (["--deform", "6"], {"WORLD_SIZE": "2", "RANK": "0"})])
def test_cli_deform_argument_errors(tmp_path, monkeypatch, extra, env):
    """--deform HOURS must be a positive multiple of the time step, and is refused with several processes; both end
    with an ERROR line before anything is read or written."""
    import si3_part_tracker as cli
    monkeypatch.chdir(tmp_path)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    monkeypatch.setattr(sys, "argv", ["si3_part_tracker.py", "-i", "x.npz", "-m", "y.npz", "-s",
                                      "sitrack_seeding_nemoTsi3_19961215_00_HSS2.npz", "-F"] + extra)
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf), pytest.raises(SystemExit):
        cli.main()
    assert any(l.startswith("ERROR") and "--deform" in l for l in buf.getvalue().splitlines())
    assert not os.listdir(tmp_path)


# ---- GPU ---------------------------------------------------------------------------------------

def _all_triples(n):
    t = np.array(list(itertools.combinations(range(n), 3)), np.int32)
    return np.concatenate([t, t[:, ::-1]])             # both orientations: C(n,3) anticlockwise or clockwise each


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TRACK_CASES))
def test_kernel_vs_oracle_all_triples(torch, sit, gold_track, name):
    """k_deform on every vertex triple of the 94 golden buoys (both orientations: degenerate, huge, flipping and
    masked triangles included) between several pairs of golden rows: bit-identical to the oracle."""
    from oracle import deform_ref as R
    T, _ = gold_track
    posC, mask = T[name + "_posC"], T[name + "_mask"]
    tri = _all_triples(posC.shape[1])
    assert tri.shape[0] == 2 * 134044
    n_valid = 0
    for k0, k1 in [(0, 1), (0, 6), (5, 29), (12, 48), (47, 48)]:
        dt = (k1 - k0) * RDT / 86400.0
        got = sit.DeformationRates(posC[k0], posC[k1], mask[k0], mask[k1], tri, dt)
        ref = R.deform(posC[k0], posC[k1], mask[k0], mask[k1], tri, dt)
        n_valid += int((ref["divergence"] != FILL).sum())
        for k in R.NAMES:
            assert got[k].dtype == np.float32 and np.array_equal(got[k], ref[k]), (name, k0, k1, k)
    assert n_valid > 10000


def _gold_engine(T, g, name, sort, rows, every, tri):
    c = TRACK_CASES[name]
    s = np.float32(c["scale"])
    nP = T["pos0"].shape[0]
    sh = np.random.default_rng(7).permutation(nP) if sort != "none" else np.arange(nP)
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
                    row_dtype=rows, deform=dict(tri=tri, every=every))
    eng.close()
    return res, sh


@pytest.mark.gpu
@pytest.mark.parametrize("every", [6, 7])
@pytest.mark.parametrize("sort", ["none", "host", "dev"])
@pytest.mark.parametrize("rows", ["f8", "f4"])
@pytest.mark.parametrize("name", ["uv1", "fast", "win"])
def test_track_deform_vs_oracle(torch, gold_track, name, rows, sort, every):
    """track(..., deform=) against the oracle on the series the same call returns: the chained f8 rows, or the f8
    series that f4 rows are the rounding of (the golden one, which the f8 rows equal bit for bit).  Windows
    [w*every, (w+1)*every], the trailing partial window dropped; buoys stored in the caller's order, cell-major by
    set_buoys, or cell-major by set_buoys_dev (whose full series comes back in engine order, so the golden series
    in the caller's order stands for it)."""
    from oracle import deform_ref as R
    T, g = gold_track
    tri = _all_triples(T["pos0"].shape[0])[::7]
    res, sh = _gold_engine(T, g, name, sort, rows, every, tri)
    posC, mask = T[name + "_posC"][:, sh], T[name + "_mask"][:, sh]
    if sort != "dev":
        assert np.array_equal(res["posC"], posC.astype(np.float32) if rows == "f4" else posC)
        assert np.array_equal(res["mask"], mask)
    ref = R.deform_series(posC, mask, tri, every, RDT)
    got = res["deform"]
    assert len(got) == len(ref) == 48 // every
    for w, (a, b) in enumerate(zip(got, ref)):
        for k in R.NAMES:
            assert np.array_equal(a[k], b[k]), (w, k)
    assert sum(int((b["divergence"] != FILL).sum()) for b in ref) > 100


@pytest.mark.gpu
def test_track_deform_sink_and_chunked_refusal(torch, gold_track):
    T, g = gold_track
    tri = _all_triples(T["pos0"].shape[0])[::11]
    seen = []
    eng = engine_for(g, device=0)
    eng.set_buoys(T["pos0"], T["jiT0"].astype(np.int32))
    r = eng.track((T["U"], T["V"], T["IC"]), 48, sink=lambda *a: None,
                  deform=dict(tri=tri, every=12, sink=lambda w, out: seen.append((w, {k: v.copy() for k, v in out.items()}))))
    assert [w for w, _ in seen] == [0, 1, 2, 3] and "deform" not in r
    eng.set_buoys(T["pos0"], T["jiT0"].astype(np.int32))
    with pytest.raises(ValueError):
        eng.track((T["U"], T["V"], T["IC"]), 48, chunk=8, deform=dict(tri=tri, every=12))
    with pytest.raises(ValueError):
        eng.track((T["U"], T["V"], T["IC"]), 48, sink=lambda *a: None, deform=dict(tri=tri + 1000, every=12))
    eng.close()


@pytest.mark.gpu
def test_cli_deform_end_to_end(tmp_path, monkeypatch):
    """si3_part_tracker.py -F --deform 6 on the 'small' synthetic case: the deformation file's variables, shapes,
    units and fill; its vertices index the tracking file's buoys; its values agree with the oracle applied to the
    tracking file's f4 rows within what f4 position rounding allows; the tracking files are those of a run without
    --deform, variable by variable and byte for byte."""
    import si3_part_tracker as cli
    from make_synth_case import write_case
    from oracle import deform_ref as R
    import sitrack_b200 as sit
    r = write_case(str(tmp_path / "in"), grid="small", nrec=24, hss=3)
    runs = {}
    for tag, extra in (("plain", []), ("deform", ["--deform", "6"])):
        d = tmp_path / tag
        d.mkdir()
        monkeypatch.chdir(d)
        monkeypatch.setattr(sys, "argv", _synth_argv(r, *extra))
        quiet(cli.main)
        runs[tag] = d / "nc"
    files = sorted(os.listdir(runs["plain"]))
    dfiles = [f for f in os.listdir(runs["deform"]) if "_deformation_" in f]
    assert dfiles == ["NEMO-SI3_SYNTH4_SYN00_deformation_nemoTsi3_idlSeed_19961215h00_19961216h00.npz"], dfiles
    assert sorted(set(os.listdir(runs["deform"])) - set(dfiles)) == files
    for f in files:                                     # the tracking files do not change
        a, b = np.load(runs["plain"] / f), np.load(runs["deform"] / f)
        assert sorted(a.files) == sorted(b.files)
        for k in a.files:
            assert a[k].dtype == b[k].dtype and a[k].tobytes() == b[k].tobytes(), (f, k)
    trk = np.load(runs["plain"] / [f for f in files if "_tracking_" in f][0])
    z = np.load(runs["deform"] / dfiles[0])
    nP, nT = trk["id_buoy"].shape[0], z["vertices"].shape[0]
    assert nT > 100 and z["vertices"].shape == (nT, 3) and z["vertices"].dtype == np.int32
    assert z["vertices"].min() >= 0 and z["vertices"].max() < nP
    assert np.array_equal(z["id_vertices"], trk["id_buoy"][z["vertices"]])
    assert z["time_start"].tolist() == trk["time"][[0, 6, 12, 18]].tolist()
    assert z["time_end"].tolist() == trk["time"][[6, 12, 18, 24]].tolist()
    assert float(z["FillValue"]) == -9999.0
    for n in R.NAMES:
        assert z[n].shape == (4, nT) and z[n].dtype == np.float32 and str(z[n + "_units"]) == sit.DEFORM_UNITS[n]
    # oracle on the f4 rows of the tracking file; tolerance from f4 position rounding (half an ulp at the largest
    # coordinate, eps): to first order, every velocity moves by <= 2 eps/dt, every mid-time coordinate by <= eps and
    # 2A by <= 4 eps P (P = sum over the edges of |dX| + |dY|)
    yx = np.stack([trk["y_pos"], trk["x_pos"]], -1).astype(np.float64)
    eps = float(np.spacing(np.float32(np.abs(yx[trk["mask"] == 1]).max()))) / 2
    tri = z["vertices"]
    n_valid = 0
    for w in range(4):
        k0, k1 = 6 * w, 6 * w + 6
        dt = 6 * RDT / 86400.0
        rf, valid = R.rates_f8(yx[k0], yx[k1], trk["mask"][k0], trk["mask"][k1], tri, dt)
        mid = 0.5 * (yx[k0] + yx[k1])
        Y, X = mid[tri, 0], mid[tri, 1]
        P = sum(np.abs(X[:, (k + 1) % 3] - X[:, k]) + np.abs(Y[:, (k + 1) % 3] - Y[:, k]) for k in range(3))
        vel = np.abs(yx[k1] - yx[k0])[tri].max((1, 2)) / dt
        a2 = 2 * rf["area"]
        G = np.max([np.abs(rf[k]) for k in ("ux", "uy", "vx", "vy")], 0)
        tol_g = (4 * (2 * eps / dt) * P + 6 * vel * 2 * eps + G * 4 * eps * P) / np.abs(a2)
        safe = valid & (np.abs(a2) > 64 * eps * P)       # validity cannot flip under the rounding
        got_valid = z["divergence"][w] != FILL
        assert np.array_equal(got_valid[safe], valid[safe])
        for k, tol in (("divergence", 2 * tol_g), ("vorticity", 2 * tol_g), ("shear", 2 * np.sqrt(2) * tol_g),
                       ("area", 2 * eps * P), ("y_ctr", eps), ("x_ctr", eps)):
            ref = rf[k][safe]
            bound = 4 * tol[safe] if np.ndim(tol) else 4 * tol
            bound = bound + 2 * np.spacing(np.abs(ref).astype(np.float32)).astype(np.float64)
            assert (np.abs(z[k][w][safe] - ref) <= bound).all(), (w, k)
            assert (z[k][w][~got_valid] == FILL).all()
        n_valid += int(safe.sum())
    assert n_valid > 100
