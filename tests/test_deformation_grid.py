"""Buoy-triangle deformation coarse-grained over the fixed cells of an Eulerian grid, rebuilt every window
(sitrack_b200.deform_grid, csrc/st_deform_grid.cu).

CPU: the oracle's Eulerian hierarchy against the material one where both must agree, against closed forms for affine
drift, at cell edges and for non-finite centroids; level shapes; EulerianGrid's and st_deform_grid_scratch_bytes'
argument checks; the writer (npz and netCDF4 branches) and the CLI's argument errors.  GPU: the pass bit for bit
against the oracle (f8 box sums from the front of the scratch, f4 fields, counts, histograms, box counts), the device
segmentation against the host-built material hierarchy, determinism across runs and buoy storage orders, the engine's
windows, the entry point's refusals and the CLI end to end."""
import contextlib
import ctypes as C
import io
import os
import sys

import numpy as np
import pytest

from conftest import TRACK_CASES
from test_deformation_edges import _device_pass, _drift, _same_bits
from test_deformation_scales import FILL, RDT, _apply, _check_stats, _engine_run, _lattice, _synth_argv, quiet

NAMES = ("divergence", "shear", "vorticity", "total", "L_eff", "y_ctr", "x_ctr")


def _covering(yx, tri, L0, margin=0):
    """origin and shape of a grid of side L0 holding every build-time centroid (as BoxHierarchy's origin)."""
    c = np.stack([((yx[tri[:, 0], k] + yx[tri[:, 1], k]) + yx[tri[:, 2], k]) / 3.0 for k in (0, 1)], 1)
    origin = np.floor(c.min(0) / L0) * L0 - margin * L0
    shape = tuple(int(n) for n in np.floor((c.max(0) - origin) / L0) + 1 + margin)
    return origin, shape


def _oracle(yx0, yx1, m0, m1, tri, dt, G):
    """-> (eulerian hierarchy, boxes, stats, per-level fields) of deform_grid_ref on the grid G."""
    from oracle import deform_grid_ref as O
    E = O.eulerian_hierarchy(yx0, yx1, m0, m1, tri, G.origin, G.L0_km, G.shape, G.levels)
    boxes, st = O.coarse_grain(yx0, yx1, m0, m1, tri, dt, E, cover=G.cover, edges=G.bin_edges, L0=G.L0_km)
    return E, boxes, st, O.grid_fields(boxes, G.shape)


# ---- CPU: the oracle ---------------------------------------------------------------------------

def test_oracle_eulerian_equals_material_on_build_positions():
    """yx0 = yx1 = P (the mid-time centroid is then the build centroid bit for bit), masks 1, BoxHierarchy's origin
    and a shape holding every key: the Eulerian hierarchy is the material one in order, ranges, children and keys."""
    from oracle import deform_grid_ref as O
    from oracle import deform_scale_ref as S
    yx, tri = _lattice(60, hole=(90.0, 80.0, 25.0))
    tri = tri[np.random.default_rng(3).permutation(tri.shape[0])]
    one = np.ones(yx.shape[0], np.int8)
    for L0, levels in ((7.0, 5), (3.0, 8), (1000.0, 2)):
        H = S.hierarchy(yx, tri, L0, levels)
        origin, shape = _covering(yx, tri, L0)
        assert np.array_equal(origin, H["origin"])
        E = O.eulerian_hierarchy(yx, yx, one, one, tri, origin, L0, shape, levels)
        assert E["binned"].all() and np.array_equal(E["order"], H["order"])
        for a, b in zip(E["levels"], H["levels"]):
            assert np.array_equal(a["key"], b["key"]) and np.array_equal(a["off"], b["off"])
            assert (a["child"] is None) == (b["child"] is None)
            if a["child"] is not None:
                assert np.array_equal(a["child"], b["child"])


@pytest.mark.parametrize("kind", ["rotation", "dilation", "general"])
def test_oracle_affine_drift_every_level(kind):
    """p1 = M p0: every counting cell of every level gives the gradient 2 (M - I)(M + I)^-1 / dt within 1e-12."""
    yx0, tri = _lattice(50, hole=(75.0, 75.0, 20.0))
    dt = 6 * RDT / 86400.0
    th, s = 0.07, 1.03
    M = dict(rotation=np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]]),
             dilation=np.array([[s, 0.0], [0.0, s]]), general=np.array([[1.02, 0.03], [-0.05, 0.97]]))[kind]
    yx1 = _apply(M, yx0)
    one = np.ones(yx0.shape[0], np.int8)
    Gr = 2.0 * (M - np.eye(2)) @ np.linalg.inv(M + np.eye(2)) / dt
    import sitrack_b200 as sit
    G = sit.EulerianGrid((-10.0, -20.0), 9.0, (14, 21), 5)
    E, boxes, st, _ = _oracle(yx0, yx1, one, one, tri, dt, G)
    assert not E["binned"].all() and E["binned"].sum() > tri.shape[0] // 2      # the grid cuts the mesh
    for b in boxes:
        S = b["S"][b["valid"]]
        assert S.shape[0] > 0
        assert np.abs(S[:, 1:5] / S[:, :1] - Gr.ravel()).max() <= 1e-12 * np.abs(Gr).max()
    assert st["n"][0] == E["binned"].sum() and (st["n"] > 0).all()


def _dyadic_tri(cy, cx):
    """Three vertices whose f8 centroid ((y0+y1)+y2)/3 is exactly (cy, cx) (dyadic offsets summing to zero)."""
    return np.array([[cy - 0.25, cx - 0.25], [cy - 0.25, cx + 0.5], [cy + 0.5, cx - 0.25]])


EDGE_GRID = dict(origin_yx=(-8.0, 4.0), L0_km=2.0, shape=(5, 3))


def _edge_case():
    """Triangles (yx0 = yx1) with centroids exactly on an interior edge (upper cell), on the origin (cell 0), on
    oy + nj L0 and on ox + ni L0 (outside), just inside the far corner (last cell), just below the origin (outside);
    valid triangles whose centroid is +inf in y or in x (their coordinate sums overflow); a triangle with a NaN vertex.
    -> (yx, tri, expected key or None per triangle, the exact centroids of the first seven)."""
    oy, ox, L0 = -8.0, 4.0, 2.0
    cases = [((oy + 2 * L0, ox + L0), (2, 1)), ((oy, ox), (0, 0)), ((oy + 5 * L0, ox), None), ((oy, ox + 3 * L0), None),
             ((oy + 5 * L0 - 0.5, ox + 3 * L0 - 0.5), (4, 2)), ((oy - 0.5, ox), None), ((oy, ox - 0.5), None)]
    P = [_dyadic_tri(*c) for c, _ in cases]
    want = [w for _, w in cases]
    P.append(np.array([[0.85e308, 0.0], [0.85e308, 1.0], [0.89e308, 0.0]]))  # Yc = +inf
    P.append(np.array([[0.0, 0.85e308], [0.0, 0.89e308], [1.0, 0.85e308]]))  # Xc = +inf
    P.append(np.array([[0.0, np.nan], [0.0, 1.0], [1.0, 0.0]]))              # NaN
    want += [None, None, None]
    yx = np.concatenate(P)
    return yx, np.arange(yx.shape[0], dtype=np.int32).reshape(-1, 3), want, [c for c, _ in cases]


def test_oracle_cell_edges_and_nonfinite():
    from oracle import deform_grid_ref as O
    from oracle import deform_ref as R
    yx, tri, want, cent = _edge_case()
    one = np.ones(yx.shape[0], np.int8)
    with np.errstate(all="ignore"):
        c = np.stack([((yx[tri[:, 0], k] + yx[tri[:, 1], k]) + yx[tri[:, 2], k]) / 3.0 for k in (0, 1)], 1)
        _, valid = R.rates_f8(yx, yx, one, one, tri, 1.0)
    for k in range(7):                                         # the premises: exact centroids, all valid
        assert valid[k] and tuple(c[k]) == cent[k], k
    assert valid[7] and valid[8] and c[7, 0] == np.inf and c[8, 1] == np.inf and np.isnan(c[9]).any()
    binned, key = O.eulerian_binning(yx, yx, one, one, tri, EDGE_GRID["origin_yx"], EDGE_GRID["L0_km"],
                                     EDGE_GRID["shape"])
    for k, w in enumerate(want):
        assert bool(binned[k]) == (w is not None), k
        if w is not None:
            assert tuple(key[k]) == w, k


@pytest.mark.parametrize("shape", [(1, 1), (5, 3), (7, 16), (17, 1), (1023, 1025)])
def test_level_shapes(shape):
    import sitrack_b200 as sit
    from oracle import deform_grid_ref as O
    G = sit.EulerianGrid((0.0, 0.0), 1.0, shape, 12)
    for s in range(12):
        want = tuple(len(np.unique(np.arange(n) >> s)) for n in shape)
        assert G.shapes[s] == want == O.grid_shape(shape, s), s
        y, x = G.centres(s)
        assert y.shape == (want[0],) and x.shape == (want[1],) and y[0] == 0.5 * 2.0 ** s
    assert G.field_size() == sum(7 * a * b for a, b in G.shapes)


@pytest.mark.parametrize("kw", [dict(L0_km=0.0), dict(L0_km=-3.0), dict(L0_km=np.nan), dict(L0_km=np.inf),
                                dict(origin_yx=(np.nan, 0.0)), dict(origin_yx=(0.0, np.inf)), dict(origin_yx=(1.0,)),
                                dict(shape=(0, 4)), dict(shape=(4, 2 ** 20 + 1)), dict(shape=(4.5, 4)), dict(shape=4),
                                dict(levels=0), dict(levels=21), dict(levels=2.5), dict(cover=0.0),
                                dict(bins=[1.0, 1.0]), dict(bins=[])])
def test_eulerian_grid_rejects(kw):
    import sitrack_b200 as sit
    a = dict(origin_yx=(0.0, 0.0), L0_km=5.0, shape=(4, 4), levels=3)
    a.update(kw)
    with pytest.raises(ValueError):
        sit.EulerianGrid(**a)


@pytest.mark.parametrize("case", [dict(nT=0), dict(nT=-1), dict(nT=2 ** 31), dict(levels=0), dict(levels=21),
                                  dict(nj=0), dict(ni=0), dict(nj=2 ** 20 + 1), dict(ni=-3), dict(nedge=0),
                                  dict(nedge=4097), dict(out=None)])
def test_grid_scratch_bytes_rejects(case):
    """st_deform_grid_scratch_bytes returns ST_EINVAL (-1) for each bad argument before any CUDA call, and leaves
    the output alone."""
    from sitrack_b200 import _lib
    a = dict(nT=1000, levels=3, nj=40, ni=50, nedge=61, out=True)
    a.update(case)
    out = C.c_int64(-5)
    rc = _lib.lib().st_deform_grid_scratch_bytes(a["nT"], a["levels"], a["nj"], a["ni"], a["nedge"],
                                                 C.byref(out) if a["out"] else None)
    assert rc == -1 and out.value == -5
    assert b"st_deform_grid_scratch_bytes" in _lib.lib().st_last_error(None)


def _writer_fields(G, jw):
    return [{n: np.full(G.shapes[s], 10 * jw + s + k, np.float32) for k, n in enumerate(NAMES)}
            for s in range(G.levels)]


def test_grid_writer_npz(tmp_path):
    import sitrack_b200 as sit
    G = sit.EulerianGrid((-30.0, 12.0), 6.0, (5, 3), 3, cover=0.25)
    f = str(tmp_path / "g.npz")
    with quiet(sit.DeformationGridWriter, f, 2, G, corigin="X") as w:
        for jw in range(2):
            w.write(jw, 100 + jw, 200 + jw, _writer_fields(G, jw))
    z = np.load(f)
    assert z["time_start"].tolist() == [100, 101] and z["time_end"].tolist() == [200, 201]
    assert z["time_end"].dtype == np.int32
    assert np.array_equal(z["L_km"], [6.0, 12.0, 24.0]) and float(z["cover"]) == 0.25
    assert z["origin"].tolist() == [-30.0, 12.0] and float(z["FillValue"]) == -9999.0
    for s in range(3):
        y, x = G.centres(s)
        assert np.array_equal(z["y%d" % (s + 1)], y) and np.array_equal(z["x%d" % (s + 1)], x)
        assert str(z["y%d_units" % (s + 1)]) == "km"
        for k, n in enumerate(NAMES):
            v = z["%s_%d" % (n, s + 1)]
            assert v.dtype == np.float32 and v.shape == (2,) + G.shapes[s]
            assert (v[1] == 10 + s + k).all() and (v[0] == s + k).all()
            assert str(z["%s_%d_units" % (n, s + 1)]) == ("km" if n in ("L_eff", "y_ctr", "x_ctr") else "day-1")
    assert G.shapes == [(5, 3), (3, 2), (2, 1)]
    assert not [p for p in os.listdir(tmp_path) if p != "g.npz"]          # the temporary members are gone


def test_grid_writer_netcdf_branch(monkeypatch, tmp_path):
    """The netCDF4 branch against the in-memory stand-in of test_cli: dimensions, variables, fill values, units
    and attributes."""
    import types
    import sitrack_b200 as sit
    from test_cli import _FakeNC
    fake = types.ModuleType("netCDF4"); fake.Dataset = _FakeNC.Dataset
    monkeypatch.setitem(sys.modules, "netCDF4", fake)
    G = sit.EulerianGrid((0.0, -4.0), 2.0, (3, 4), 2)
    f = str(tmp_path / "g.nc")
    with quiet(sit.DeformationGridWriter, f, 3, G, corigin="ORG") as w:
        for jw in range(3):
            w.write(jw, jw, jw + 1, _writer_fields(G, jw))
    ds = _FakeNC.files[f]
    assert ds._dims == {"time": None, "y1": 3, "x1": 4, "y2": 2, "x2": 2}
    assert ds.attrs["Origin"] == "ORG" and np.array_equal(ds.attrs["L_km"], [2.0, 4.0]) and ds.attrs["cover"] == 0.5
    assert np.array_equal(ds.attrs["origin"], [0.0, -4.0])
    v = ds.variables["shear_2"]
    assert v.a.shape == (3, 2, 2) and v.a.dtype == np.float32 and v.fill == -9999.0 and v.units == "day-1"
    assert (v.a[2] == 21 + 1).all()
    assert np.array_equal(ds.variables["x1"].a, G.centres(0)[1]) and ds.variables["x1"].units == "km"
    assert ds.variables["time_end"].a.tolist() == [1, 2, 3]


@pytest.mark.parametrize("extra", [["--deform-grid", "12", "3"], ["--deform", "6", "--deform-grid", "0", "3"],
                                   ["--deform", "6", "--deform-grid", "-1", "3"],
                                   ["--deform", "6", "--deform-grid", "12", "0"],
                                   ["--deform", "6", "--deform-grid", "12", "21"],
                                   ["--deform", "6", "--deform-grid", "12", "2.5"]])
def test_cli_deform_grid_argument_errors(tmp_path, monkeypatch, extra):
    """--deform-grid needs --deform, a positive L0 and 1..20 levels; each error is an ERROR line printed before
    anything is read or written."""
    import si3_part_tracker as cli
    monkeypatch.chdir(tmp_path)
    monkeypatch.setattr(sys, "argv", ["si3_part_tracker.py", "-i", "x.npz", "-m", "y.npz", "-s",
                                      "sitrack_seeding_nemoTsi3_19961215_00_HSS2.npz", "-F"] + extra)
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf), pytest.raises(SystemExit):
        cli.main()
    assert any(l.startswith("ERROR") and "--deform-grid" in l for l in buf.getvalue().splitlines())
    assert not os.listdir(tmp_path)


def test_cli_grid_over_the_model_grid():
    """The CLI's grid: origin floor(min / L0) L0, floor((max - origin) / L0) + 1 cells; more than 2^20 a side is an
    ERROR line."""
    import si3_part_tracker as cli
    Yt = np.array([[-25.0, 13.0], [7.0, 36.0]])
    Xt = np.array([[4.0, 59.9], [60.0, 11.0]])
    G = cli.deform_grid_over(Yt, Xt, 12.0, 3)
    assert G.origin.tolist() == [-36.0, 0.0] and G.shape == (7, 6) and G.levels == 3
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf), pytest.raises(SystemExit):
        cli.deform_grid_over(Yt, Xt, 60.0 / 2 ** 21, 3)
    assert buf.getvalue().startswith("ERROR") and "--deform-grid" in buf.getvalue()


# ---- GPU ---------------------------------------------------------------------------------------

def _bounds(G, nT):
    return [min(nT, nj * ni) for nj, ni in G.shapes]


def _device_grid(torch, G, yx0, yx1, m0, m1, tri, dt, slots=None):
    """The pass as GriddedRates launches it, plus the f8 box records from the front of its scratch (level s from the
    prefix sum of the bounds) and the box counts.  -> (per level (nbox,7) f8 sums, fields, mom, hist, nbox)."""
    from sitrack_b200 import deform_grid as DG
    dev = torch.device("cuda", 0)
    with torch.cuda.device(dev):
        t = lambda a, d: torch.from_numpy(np.ascontiguousarray(a, d)).to(dev)
        plan = DG._GridPlan(torch, dev, G, tri)
        mom, hist, fields, nbox = plan.outputs()
        plan.launch(None, t(yx0, np.float64), t(m0, np.int8), t(yx1, np.float64), t(m1, np.int8), dt, mom, hist,
                    fields, nbox, torch.cuda.current_stream(dev))
        torch.cuda.synchronize(dev)
        b = _bounds(G, tri.shape[0])
        rec = plan.scratch[:8 * sum(b)].cpu().numpy().reshape(-1, 8)[:, :7]
        fields, mom, hist, nbox = fields.cpu().numpy(), mom.cpu().numpy(), hist.cpu().numpy(), nbox.cpu().numpy()
    b0 = np.r_[0, np.cumsum(b)]
    S = [rec[b0[s]:b0[s] + nbox[s]] for s in range(G.levels)]
    return S, DG.split_fields(G, fields), mom, hist, nbox


def _check_grid(torch, G, yx0, yx1, m0, m1, tri, dt):
    """The pass against the oracle: box counts, f8 box sums bit for bit, f4 fields bit for bit, histograms and n
    exactly, moment sums within 1e-11; and a second pass gives the same bits.  -> (oracle E, stats, fields)."""
    E, boxes, rs, rf = _oracle(yx0, yx1, m0, m1, tri, dt, G)
    S, fields, mom, hist, nbox = _device_grid(torch, G, yx0, yx1, m0, m1, tri, dt)
    assert nbox.tolist() == [lv["key"].shape[0] for lv in E["levels"]]
    for s in range(G.levels):
        same = _same_bits(S[s], boxes[s]["S"])
        assert same.all(), "level %d: %d of %d box sums differ" % (s + 1, (~same).any(1).sum(), same.shape[0])
        for k in NAMES:
            assert fields[s][k].shape == G.shapes[s] and _same_bits(fields[s][k], rf[s][k]).all(), (s + 1, k)
        y, x = G.centres(s)
        assert np.array_equal(fields[s]["y_km"], y) and np.array_equal(fields[s]["x_km"], x)
    assert np.array_equal(hist, rs["hist"]) and np.array_equal(hist[:, 0].sum(1), rs["n"])
    assert rs["n"][0] == E["binned"].sum()
    assert (np.abs(mom - rs["sums"]) <= 1e-11 * np.abs(rs["sums"])).all()
    S2, fields2, mom2, hist2, nbox2 = _device_grid(torch, G, yx0, yx1, m0, m1, tri, dt)
    assert np.array_equal(mom2, mom) and np.array_equal(hist2, hist) and np.array_equal(nbox2, nbox)
    for s in range(G.levels):
        assert _same_bits(S2[s], S[s]).all()
        for k in NAMES:
            assert _same_bits(fields2[s][k], fields[s][k]).all()
    return E, rs, fields


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TRACK_CASES))
def test_grid_vs_oracle_golden(torch, sit, gold_track, name):
    """The golden rows on a 20 km grid that cuts the cloud (some triangles fall outside it)."""
    T, _ = gold_track
    posC, mask = T[name + "_posC"], T[name + "_mask"]
    tri = sit.TriangulateCloud(T["pos0"])
    G = sit.EulerianGrid((-60.0, -200.0), 20.0, (12, 11), 4)
    n = 0
    for k0, k1 in [(0, 6), (5, 29), (12, 48)]:
        E, rs, _ = _check_grid(torch, G, posC[k0], posC[k1], mask[k0], mask[k1], tri, (k1 - k0) * RDT / 86400.0)
        assert not E["binned"].all()
        n += rs["n"]
    assert n[0] > 30 and n[1] > 3


@pytest.mark.gpu
def test_grid_vs_oracle_lattice_large_drift(torch, sit):
    """~200 k buoys with 2 % masks, flipped triangles and a hole, a drift of up to 9 km against 12 km cells (many
    triangles change cells between windows), a grid that leaves part of the lattice outside."""
    rng = np.random.default_rng(21)
    yx0, tri = _lattice(450, hole=(600.0, 700.0, 90.0), seed=3)
    nP = yx0.shape[0]
    yx1 = yx0 + np.stack([6.0 * np.sin(yx0[:, 1] / 90.0), 9.0 * np.cos(yx0[:, 0] / 70.0)], 1)
    jump = rng.choice(nP, 300, replace=False)
    yx1[jump] += rng.choice([-1.0, 1.0], (300, 2)) * 7.0
    m0 = (rng.random(nP) >= 0.02).astype(np.int8)
    m1 = (rng.random(nP) >= 0.02).astype(np.int8)
    G = sit.EulerianGrid((-5.0, 30.0), 12.0, (110, 100), 6)
    from oracle import deform_grid_ref as O
    b_start, k_start = O.eulerian_binning(yx0, yx0, m0, m0, tri, G.origin, 12.0, G.shape)
    E, rs, fields = _check_grid(torch, G, yx0, yx1, m0, m1, tri, 0.25)
    both = E["binned"] & b_start
    k_mid = O.eulerian_binning(yx0, yx1, m0, m1, tri, G.origin, 12.0, G.shape)[1]
    assert (k_mid[both] != k_start[both]).any(1).sum() > 20000                    # membership moved with the drift
    assert (~E["binned"]).sum() > 20000 and (rs["n"] > 0).all()
    assert (fields[0]["total"] == FILL).any() and (fields[0]["total"] != FILL).sum() > 1000


@pytest.mark.gpu
def test_grid_cell_edges_and_nonfinite(torch, sit):
    """_edge_case on the device: the same cells, the same bins, the same bits."""
    yx, tri, want, _ = _edge_case()
    one = np.ones(yx.shape[0], np.int8)
    G = sit.EulerianGrid(levels=2, cover=1e-3, **EDGE_GRID)
    E, rs, fields = _check_grid(torch, G, yx, yx, one, one, tri, 0.25)
    assert E["binned"].tolist() == [w is not None for w in want]
    assert sorted(map(tuple, E["levels"][0]["key"])) == sorted(w for w in want if w is not None)


@pytest.mark.gpu
def test_grid_nothing_binned(torch, sit):
    """A grid away from the mesh: zero boxes, every field FillValue, n = 0, zero moments."""
    yx0, tri = _lattice(30, seed=4)
    yx1, m0, m1 = _drift(yx0, 5, jumps=5, masked=0.02)
    G = sit.EulerianGrid((5000.0, 5000.0), 10.0, (9, 7), 3)
    E, rs, fields = _check_grid(torch, G, yx0, yx1, m0, m1, tri, 0.25)
    assert not E["binned"].any() and (rs["n"] == 0).all()
    assert all((f[k] == FILL).all() for f in fields for k in NAMES)


@pytest.mark.gpu
@pytest.mark.parametrize("nT", [1, 255, 256, 257])
def test_grid_one_cell_and_block_sizes(torch, sit, nT):
    """nT around the block size, on a 1 x 1 grid holding every triangle and on a 5 km grid of 3 levels."""
    yx0, tri = _lattice(20, seed=13)
    yx1, m0, m1 = _drift(yx0, 14, jumps=12, masked=0.03)
    tri = tri[np.random.default_rng(15).permutation(tri.shape[0])[:nT]]
    G1 = sit.EulerianGrid((-10.0, -10.0), 100.0, (1, 1), 1, cover=1e-6)
    E, rs, _ = _check_grid(torch, G1, yx0, yx1, m0, m1, tri, 0.25)
    assert E["levels"][0]["key"].shape[0] == int(E["binned"].any())
    G = sit.EulerianGrid((-3.0, -3.0), 5.0, (13, 13), 3, cover=1e-3)
    _check_grid(torch, G, yx0, yx1, m0, m1, tri, 0.25)


@pytest.mark.gpu
def test_grid_levels20(torch, sit):
    """20 levels on a 300 x 300 lattice with 3 km cells: the top levels are single cells."""
    yx0, tri = _lattice(300, d=3.0, seed=9)
    yx1, m0, m1 = _drift(yx0, 10, jumps=200, masked=0.01)
    G = sit.EulerianGrid((-3.0, -3.0), 3.0, (302, 303), 20)
    E, rs, fields = _check_grid(torch, G, yx0, yx1, m0, m1, tri, 0.25)
    assert G.shapes[-1] == (1, 1) and E["levels"][-1]["key"].shape[0] == 1 and (rs["n"][:8] > 0).all()


@pytest.mark.gpu
def test_grid_device_segmentation_equals_host_hierarchy(torch, sit):
    """yx0 = yx1 = P on the grid of BoxHierarchy(P, ...): the device-sorted, device-segmented Eulerian pass gives the
    f8 box sums of the Lagrangian pass over the host-built hierarchy, at every level."""
    yx, tri = _lattice(200, hole=(300.0, 250.0, 60.0), seed=6)
    tri = tri[np.random.default_rng(8).permutation(tri.shape[0])]
    one = np.ones(yx.shape[0], np.int8)
    H = sit.BoxHierarchy(yx, tri, 9.0, 6)
    origin, shape = _covering(yx, tri, 9.0)
    G = sit.EulerianGrid(origin, 9.0, shape, 6)
    S_lag, _, mom_l, hist_l = _device_pass(torch, H, yx, yx, one, one, 0.25)
    S_eul, _, mom_e, hist_e, nbox = _device_grid(torch, G, yx, yx, one, one, tri, 0.25)
    assert nbox.tolist() == H.nbox.tolist()
    for s in range(6):
        assert _same_bits(S_eul[s], S_lag[s]).all(), s
    assert np.array_equal(hist_e, hist_l) and np.array_equal(mom_e, mom_l)


@pytest.mark.gpu
@pytest.mark.parametrize("rows", ["f8", "f4"])
@pytest.mark.parametrize("name", ["uv1", "win"])
def test_track_deform_grid(torch, sit, gold_track, name, rows):
    """track(deform=dict(..., grid=G)): per-window fields and statistics equal the oracle's, bit for bit the same
    whether the buoys are stored in the caller's order or sorted on the host or the device, with and without
    `scales`; the per-triangle outputs and the scales' statistics are those of the same call without `grid`."""
    T, g = gold_track
    every = 6
    sh = np.random.default_rng(7).permutation(T["pos0"].shape[0])
    pos0 = T["pos0"][sh]
    tri = sit.TriangulateCloud(pos0)
    G = sit.EulerianGrid((-60.0, -200.0), 20.0, (12, 11), 4)
    H = sit.BoxHierarchy(pos0, tri, 20.0, 3)
    posC, mask = T[name + "_posC"][:, sh], T[name + "_mask"][:, sh]
    ref = [_oracle(posC[k], posC[k + every], mask[k], mask[k + every], tri, every * RDT / 86400.0, G)
           for k in range(0, 48, every)]
    first = None
    for sort in ("none", "host", "dev"):
        for scales in (False, True):
            spec = dict(tri=tri, every=every, grid=G)
            if scales:
                spec["scales"] = H
            res, _ = _engine_run(T, g, name, sort, rows, every, spec)
            got = res["deform_grid"]
            assert len(got) == len(ref) == 8
            for (fl, st), (_, _, rs, rf) in zip(got, ref):
                _check_stats(st, rs, G)
                for s in range(G.levels):
                    for k in NAMES:
                        assert _same_bits(fl[s][k], rf[s][k]).all(), (sort, s, k)
            if first is None:
                first = got
                plain, _ = _engine_run(T, g, name, sort, rows, every, dict(tri=tri, every=every, scales=H))
            for (fl, st), (fl0, st0) in zip(got, first):
                for k in st:
                    assert np.array_equal(st[k], st0[k]), (sort, k)
                for a, b in zip(fl, fl0):
                    for k in a:
                        assert np.array_equal(a[k], b[k]), (sort, k)
            if scales and sort == "none":
                for a, b in zip(res["deform_scales"], plain["deform_scales"]):
                    for k in a:
                        assert np.array_equal(a[k], b[k])
                for a, b in zip(res["deform"], plain["deform"]):
                    for k in sit.DEFORM_NAMES:
                        assert np.array_equal(a[k], b[k])
            if not scales:
                assert "deform_scales" not in res
    assert sum(int(st["n"][1]) for _, st in first) > 5


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["keep", "sink"])
@pytest.mark.parametrize("every", [1, 48, 49])
def test_track_grid_windows(torch, sit, gold_track, every, mode):
    """every = 1, nrec and nrec + 1 over the 48 records of the uv1 case, rows kept or sunk, results collected or
    handed to grid_sink."""
    from conftest import engine_for
    T, g = gold_track
    posC, mask = T["uv1_posC"], T["uv1_mask"]
    nrec = 48
    tri = sit.TriangulateCloud(T["pos0"])
    G = sit.EulerianGrid((-100.0, -240.0), 25.0, (13, 13), 3)
    nwin = nrec // every
    ref = [_oracle(posC[w * every], posC[(w + 1) * every], mask[w * every], mask[(w + 1) * every], tri,
                   every * RDT / 86400.0, G) for w in range(nwin)]
    eng = engine_for(g, device=0)
    eng.set_buoys(T["pos0"], T["jiT0"].astype(np.int32))
    spec = dict(tri=tri, every=every, grid=G)
    if mode == "keep":
        res = eng.track((T["U"], T["V"], T["IC"]), nrec, pos0=T["pos0"], deform=spec)
        got = res["deform_grid"]
    else:
        seen = []
        spec["grid_sink"] = lambda w, fl, st: seen.append((w, fl, st))
        res = eng.track((T["U"], T["V"], T["IC"]), nrec, sink=lambda *a: None, deform=spec)
        assert "deform_grid" not in res and [w for w, _, _ in seen] == list(range(nwin))
        got = [(fl, st) for _, fl, st in seen]
    eng.close()
    assert len(got) == nwin
    for (fl, st), (_, _, rs, rf) in zip(got, ref):
        _check_stats(st, rs, G)
        for s in range(G.levels):
            for k in NAMES:
                assert _same_bits(fl[s][k], rf[s][k]).all()


@pytest.mark.gpu
def test_grid_entry_point_refuses_bad_dt_and_nT(torch, sit):
    """st_deform_grid_dev, given real, aligned device buffers, returns ST_EINVAL for dt_days <= 0 (and NaN) and
    nT < 0, and writes nothing; the same buffers with dt_days > 0 are accepted."""
    from sitrack_b200 import _lib
    from sitrack_b200 import deform_grid as DG
    L = _lib.lib()
    dev = torch.device("cuda", 0)
    yx0, tri = _lattice(8)
    yx1, m0, m1 = _drift(yx0, 16)
    G = sit.EulerianGrid((-3.0, -3.0), 6.0, (5, 5), 2)
    t = lambda a, d: torch.from_numpy(np.ascontiguousarray(a, d)).to(dev)
    with torch.cuda.device(dev):
        st = torch.cuda.current_stream(dev)
        a_t, b_t, m0_t, m1_t = t(yx0, np.float64), t(yx1, np.float64), t(m0, np.int8), t(m1, np.int8)
        plan = DG._GridPlan(torch, dev, G, tri)
        mom, hist, fields, nbox = plan.outputs()
        mom.fill_(7.0); hist.fill_(7); fields.fill_(7.0); nbox.fill_(7)
        p = lambda x: C.c_void_p(x.data_ptr())
        for n, dt in [(tri.shape[0], 0.0), (tri.shape[0], -0.25), (tri.shape[0], -0.0), (tri.shape[0], float("nan")),
                      (-1, 0.25)]:
            assert L.st_deform_grid_dev(
                None, n, p(plan.tri_t), p(a_t), p(m0_t), p(b_t), p(m1_t), dt, G.levels, G.shape[0], G.shape[1],
                float(G.origin[0]), float(G.origin[1]), G.L0_km, plan.min_area.ctypes.data, G.bin_edges.size,
                p(plan.edges_t), p(plan.scratch), plan.scratch_bytes, p(mom), p(hist), p(fields), p(nbox),
                C.c_void_p(st.cuda_stream)) == -1, (n, dt)
        torch.cuda.synchronize(dev)
        assert (mom == 7.0).all().item() and (hist == 7).all().item() and (fields == 7.0).all().item()
        assert (nbox == 7).all().item()
        plan.launch(None, a_t, m0_t, b_t, m1_t, 0.25, mom, hist, fields, nbox, st)
        torch.cuda.synchronize(dev)
        assert hist[0, 0].sum().item() > 0 and (nbox != 7).all().item() and (fields != 7.0).all().item()


@pytest.mark.gpu
def test_gridded_rates_public_call(sit):
    """sit.GriddedRates: the public host-array call gives the oracle's fields and statistics."""
    yx0, tri = _lattice(40, seed=2)
    yx1, m0, m1 = _drift(yx0, 3, jumps=10, masked=0.02)
    G = sit.EulerianGrid((10.0, -2.0), 7.0, (14, 18), 3)
    fields, st = sit.GriddedRates(yx0, yx1, m0, m1, tri, G, 0.25)
    _, _, rs, rf = _oracle(yx0, yx1, m0, m1, tri, 0.25, G)
    _check_stats(st, rs, G)
    for s in range(3):
        for k in NAMES:
            assert fields[s][k].dtype == np.float32 and _same_bits(fields[s][k], rf[s][k]).all()
    with pytest.raises(TypeError):
        sit.GriddedRates(yx0, yx1, m0, m1, tri, sit.BoxHierarchy(yx0, tri, 7.0, 2), 0.25)


@pytest.mark.gpu
def test_cli_deform_grid_end_to_end(tmp_path, monkeypatch):
    """si3_part_tracker.py -F --deform 6 --deform-grid 75 3 on the 'small' synthetic case: both new files' variables,
    shapes, units and attributes; values agree with the oracle applied to the tracking file's f4 rows; the tracking
    and per-triangle files are those of a run without --deform-grid."""
    import si3_part_tracker as cli
    from make_synth_case import write_case
    from oracle import deform_grid_ref as O
    r = write_case(str(tmp_path / "in"), grid="small", nrec=24, hss=3)
    runs = {}
    for tag, extra in (("plain", ["--deform", "6"]), ("grid", ["--deform", "6", "--deform-grid", "75", "3"])):
        d = tmp_path / tag
        d.mkdir()
        monkeypatch.chdir(d)
        monkeypatch.setattr(sys, "argv", _synth_argv(r, *extra))
        quiet(cli.main)
        runs[tag] = d / "nc"
    files = sorted(os.listdir(runs["plain"]))
    tail = "nemoTsi3_idlSeed_19961215h00_19961216h00.npz"
    gfiles = sorted(f for f in os.listdir(runs["grid"]) if "_deformation-grid" in f)
    assert gfiles == ["NEMO-SI3_SYNTH4_SYN00_deformation-grid-scaling_" + tail,
                      "NEMO-SI3_SYNTH4_SYN00_deformation-grid_" + tail], gfiles
    assert sorted(set(os.listdir(runs["grid"])) - set(gfiles)) == files
    for f in files:
        a, b = np.load(runs["plain"] / f), np.load(runs["grid"] / f)
        assert sorted(a.files) == sorted(b.files)
        for k in a.files:
            assert a[k].dtype == b[k].dtype and a[k].tobytes() == b[k].tobytes(), (f, k)
    trk = np.load(runs["plain"] / [f for f in files if "_tracking_" in f][0])
    dfm = np.load(runs["plain"] / [f for f in files if "_deformation_" in f][0])
    zf = np.load(runs["grid"] / gfiles[1])
    zs = np.load(runs["grid"] / gfiles[0])
    g = r["grid"]
    L0 = 75.0
    origin = np.array([np.floor(g["Yt"].min() / L0) * L0, np.floor(g["Xt"].min() / L0) * L0])
    shape = tuple(int(np.floor((A.max() - o) / L0)) + 1 for A, o in ((g["Yt"], origin[0]), (g["Xt"], origin[1])))
    assert np.array_equal(zf["origin"], origin) and zf["L_km"].tolist() == [75.0, 150.0, 300.0]
    assert zf["time_start"].tolist() == dfm["time_start"].tolist() == zs["time_start"].tolist()
    assert zs["scale_km"].tolist() == [-9999.0, 75.0, 150.0, 300.0]
    assert zf["divergence_1"].shape == (4,) + shape and zf["total_3"].dtype == np.float32
    for k in ("hist_total", "hist_divergence", "hist_shear"):
        assert zs[k].shape == (4, 4, 62) and np.array_equal(zs[k].sum(2), zs["n"])
    # the oracle on the tracking file's f4 rows (the device works on the f8 positions those rows round): counts
    # within a few cells, field values within 1e-3 where both count
    yx = np.stack([trk["y_pos"], trk["x_pos"]], -1).astype(np.float64)
    tri = dfm["vertices"]
    assert (zs["n"][:, 0] > 100).all() and (zs["n"][:, 1] > 3).all()
    for w in range(4):
        E = O.eulerian_hierarchy(yx[6 * w], yx[6 * w + 6], trk["mask"][6 * w], trk["mask"][6 * w + 6], tri, origin,
                                 L0, shape, 3)
        boxes, ref = O.coarse_grain(yx[6 * w], yx[6 * w + 6], trk["mask"][6 * w], trk["mask"][6 * w + 6], tri, 0.25,
                                    E, L0=L0)
        assert (np.abs(zs["n"][w] - ref["n"]) <= 1 + ref["n"] // 100).all(), w
        rf = O.grid_fields(boxes, shape)
        for s in range(3):
            a, b = zf["total_%d" % (s + 1)][w], rf[s]["total"]
            both = (a != FILL) & (b != FILL)
            assert both.sum() >= 0.9 * (b != FILL).sum()
            assert (np.abs(a[both] - b[both]) <= 1e-3 * np.abs(b[both]) + 1e-6).all(), (w, s)


@pytest.mark.gpu
def test_bench_deform_grid_small():
    """tools/bench_deform.py end to end on a small lattice: the grid pass's stage timings, sample exactness and
    run-to-run identity."""
    import json
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "bench_deform.py"), "--ny", "300", "--nx", "300",
                        "--seconds", "0.05"], stdout=subprocess.PIPE, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:]
    gr = json.loads(r.stdout.strip().splitlines()[-1])["grid"]
    assert gr["sample_cells_bit_identical"] and gr["run_to_run_identical"] and gr["sample_cells"] > 1000
    assert set(gr["stages"]) == {"key_us", "sort_us", "segmentation_us", "boxes_stats_fields_us"}
    assert gr["boxes_per_level"][0] > 1000 and gr["n_per_scale"][0] == gr["binned_triangles"]
