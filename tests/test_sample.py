"""SI3 T-cell fields sampled along the buoy trajectories (sitrack_b200.sample, csrc/st_sample.cu).

CPU: the oracle (oracle/sample_ref.py) on closed forms (linear fields on a regular and a rotated grid, corner values,
land and non-finite corners, the quadrant and parallelogram rules), the vectorised oracle against its per-buoy loop,
the host-side argument checks, both writer branches and the CLI's ERROR lines.  GPU: k_sample equals the oracle bit
for bit over the golden cases stepped record by record; track(sample=...) with f8 and f4 rows, sorted buoys,
physics, every > 1, rec_first windows and buoys killed at the border; siconc from the record slot equals siconc as an
extra field; st_sample_dev's refusals; the CLI end to end, alone and under torchrun; a small run of the benchmark."""
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
FILL = np.float32(-9999.0)


def _ref():
    from oracle import sample_ref as O
    return O


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def _regular(nj=12, ni=10, d=5.0, theta=0.0, y0=-300.0, x0=700.0):
    """T-points of a regular grid of spacing d, rotated by theta about its origin -> (Yt, Xt)."""
    jj, ii = np.meshgrid(np.arange(nj, dtype=np.float64), np.arange(ni, dtype=np.float64), indexing="ij")
    y, x = jj * d, ii * d
    c, s = np.cos(theta), np.sin(theta)
    return y0 + c * y + s * x, x0 - s * y + c * x


def _in_grid(rng, n, nj, ni, d, theta, y0=-300.0, x0=700.0):
    """n random positions in the cells 1..nj-2 x 1..ni-2 of _regular's grid -> (yx, cells)."""
    jy = rng.uniform(0.5, nj - 1.5, n)
    ix = rng.uniform(0.5, ni - 1.5, n)
    y, x = jy * d, ix * d
    c, s = np.cos(theta), np.sin(theta)
    yx = np.stack([y0 + c * y + s * x, x0 - s * y + c * x], 1)
    return yx, np.stack([np.round(jy), np.round(ix)], 1).astype(np.int64)


# ---- CPU: the oracle ---------------------------------------------------------------------------

@pytest.mark.parametrize("theta", [0.0, 0.3, -1.1])
def test_oracle_reproduces_linear_fields(theta):
    """A field linear in (x, y) is reproduced by "bilinear" to rounding on a regular and on a rotated grid (every
    T-quad is a parallelogram, where the bilinear map is exact), and equals the sample loop bit for bit."""
    O = _ref()
    nj, ni, d = 12, 10, 5.0
    Yt, Xt = _regular(nj, ni, d, theta)
    F = (2.5 + 0.01 * Xt - 0.02 * Yt).astype(np.float32)
    rng = np.random.default_rng(3)
    yx, cell = _in_grid(rng, 2000, nj, ni, d, theta)
    tm = np.ones((nj, ni), np.int8)
    got = O.sample(F, tm, cell, yx, np.ones(2000, np.int8), "bilinear", Yt, Xt)[0]
    exact = 2.5 + 0.01 * yx[:, 1] - 0.02 * yx[:, 0]
    # the T-values are f4: their rounding (< 2^-24 relative of |F| <= 20) bounds the error
    assert np.abs(got - exact).max() < 4e-6
    assert got.tobytes() == O.sample_loop(F, tm, cell, yx, np.ones(2000, np.int8), "bilinear", Yt, Xt)[0].tobytes()
    cellv = O.sample(F, tm, cell, yx, np.ones(2000, np.int8), "cell", Yt, Xt)[0]
    assert np.array_equal(cellv, F[cell[:, 0], cell[:, 1]])


def test_oracle_corner_values_at_the_corners():
    """P at a T-point of the 3 x 3 stencil gives that point's value exactly, whichever quad it picks."""
    O = _ref()
    Yt, Xt = _regular(8, 8, 4.0, 0.4)
    F = np.random.default_rng(1).uniform(-5, 5, (8, 8)).astype(np.float32)
    tm = np.ones((8, 8), np.int8)
    cells, yx, want = [], [], []
    for dj in (-1, 0, 1):
        for di in (-1, 0, 1):
            cells.append((4, 4)); yx.append((Yt[4 + dj, 4 + di], Xt[4 + dj, 4 + di])); want.append(F[4 + dj, 4 + di])
    got = O.sample(F, tm, np.array(cells), np.array(yx), np.ones(9, np.int8), "bilinear", Yt, Xt)[0]
    assert np.array_equal(got, np.array(want, np.float32))


def test_oracle_land_and_nonfinite_corners_renormalise():
    """A land or non-finite corner is dropped and the other weights renormalised; an all-dropped quad falls back to the
    cell value, and a non-finite cell value then gives FillValue; masked rows and cells outside the interior too."""
    O = _ref()
    Yt, Xt = _regular(6, 6, 10.0)
    F = np.arange(36, dtype=np.float32).reshape(6, 6)
    tm = np.ones((6, 6), np.int8)
    # P at xi = 0.25, eta = 0.5 of the quad SW = T[2,2] (cell (2,2): P north-east of T[2,2])
    P = np.array([[Yt[2, 2] + 5.0, Xt[2, 2] + 2.5]])
    c = np.array([[2, 2]])
    w = np.array([0.75 * 0.5, 0.25 * 0.5, 0.25 * 0.5, 0.75 * 0.5])
    v = np.array([F[2, 2], F[2, 3], F[3, 3], F[3, 2]], np.float64)
    one = np.ones(1, np.int8)
    assert O.sample(F, tm, c, P, one, "bilinear", Yt, Xt)[0, 0] == np.float32((w * v).sum())
    tm2 = tm.copy(); tm2[3, 3] = 0
    assert O.sample(F, tm2, c, P, one, "bilinear", Yt, Xt)[0, 0] == \
        np.float32((((w[0] * v[0]) + w[1] * v[1]) + w[3] * v[3]) / ((w[0] + w[1]) + w[3]))
    F2 = F.copy(); F2[3, 3] = np.nan
    assert O.sample(F2, tm, c, P, one, "bilinear", Yt, Xt)[0, 0] == O.sample(F, tm2, c, P, one, "bilinear", Yt, Xt)[0, 0]
    F3 = F.copy(); F3[2, 3] = np.inf
    tm3 = tm2.copy(); tm3[2, 2] = 0; tm3[3, 2] = 0
    assert O.sample(F3, tm3, c, P, one, "bilinear", Yt, Xt)[0, 0] == F[2, 2]            # all dropped: the cell value
    F4 = F3.copy(); F4[2, 2] = np.nan
    assert O.sample(F4, tm3, c, P, one, "bilinear", Yt, Xt)[0, 0] == FILL
    assert O.sample(F4, tm, c, P, one, "cell", Yt, Xt)[0, 0] == FILL
    # weights of the kept corners all zero (P on the dropped corner): the cell value
    P2 = np.array([[Yt[3, 3], Xt[3, 3]]])
    assert O.sample(F, tm2, c, P2, one, "bilinear", Yt, Xt)[0, 0] == F[2, 2]
    for cc, m in (([2, 2], 0), ([0, 2], 1), ([2, 5], 1), ([2 | (1 << 31), 2], 0)):
        assert O.sample(F, tm, np.array([cc]), P, np.array([m], np.int8), "bilinear", Yt, Xt)[0, 0] == FILL
    dead = np.array([[2 | (1 << 31), 2]])                                                 # bit 31 stripped
    assert O.sample(F, tm, dead, P, one, "cell", Yt, Xt)[0, 0] == F[2, 2]
    for a, b in ((F, tm2), (F2, tm), (F3, tm3), (F4, tm3)):
        for p in (P, P2):
            assert O.sample(a, b, c, p, one, "bilinear", Yt, Xt).tobytes() == \
                O.sample_loop(a, b, c, p, one, "bilinear", Yt, Xt).tobytes()


def test_oracle_quadrant_and_parallelogram_rules():
    """A point on a grid line through T[jT,iT] takes the quad of the higher index; NaN positions behave like ties.
    On a parallelogram k2 == 0 exactly and the linear root is taken; on a trapezoid (k2 != 0) the quadratic one."""
    O = _ref()
    Yt, Xt = _regular(6, 6, 10.0)
    jT, iT = np.array([2, 2, 2, 2, 2]), np.array([2, 2, 2, 2, 2])
    P = np.array([[Yt[2, 2], Xt[2, 2] - 3.0],      # on W->E, west: j0 = jT, i0 = iT-1
                  [Yt[2, 2] - 3.0, Xt[2, 2]],      # on S->N, south: j0 = jT-1, i0 = iT
                  [Yt[2, 2], Xt[2, 2]],            # both: the NE quad
                  [Yt[2, 2] - 1.0, Xt[2, 2] - 1.0],
                  [np.nan, np.nan]])
    j0, i0 = O.quad(P, jT, iT, Yt, Xt)
    assert j0.tolist() == [2, 1, 2, 1, 2] and i0.tolist() == [1, 2, 2, 1, 2]
    # parallelogram: a sheared quad, P at (xi, eta) = (0.25, 0.75)
    a, b, d = np.array([0.0, 0.0]), np.array([1.0, 8.0]), np.array([6.0, 2.0])         # [y, x]
    c = b + d - a
    P = a + 0.25 * (b - a) + 0.75 * (d - a)
    xi, eta = O.inv_bilinear(P[None], a[None], b[None], c[None], d[None])
    assert xi[0] == 0.25 and eta[0] == 0.75
    # trapezoid: c moved; P = the bilinear image of (0.3, 0.6) is found back to rounding
    c2 = c + np.array([1.5, 2.0])
    xi0, eta0 = 0.3, 0.6
    P2 = a + xi0 * (b - a) + eta0 * (d - a) + xi0 * eta0 * (a - b + c2 - d)
    xi, eta = O.inv_bilinear(P2[None], a[None], b[None], c2[None], d[None])
    assert abs(xi[0] - xi0) < 1e-14 and abs(eta[0] - eta0) < 1e-14
    # outside the quad: clamped to [0, 1]
    xi, eta = O.inv_bilinear((a - np.array([1.0, 1.0]))[None], a[None], b[None], c2[None], d[None])
    assert xi[0] == 0.0 and eta[0] == 0.0
    assert O.sampled_rows(48, 1).tolist() == list(range(49)) and O.sampled_rows(48, 7).tolist() == [0, 7, 14, 21, 28,
                                                                                                    35, 42]
    assert O.sampled_rows(5, 6).tolist() == [0] and [O.row_record(r, 3) for r in (0, 1, 2, 7)] == [3, 3, 4, 9]


def _curvy(rng, nj=30, ni=26, d=6.0):
    """A curvilinear grid (smooth distortion), land, NaNs -> (Yt, Xt, tmask, fields (3, nj, ni) f4)."""
    jj, ii = np.meshgrid(np.arange(nj, dtype=np.float64), np.arange(ni, dtype=np.float64), indexing="ij")
    Yt = jj * d + 1.7 * np.sin(ii / 3.0) + 0.9 * np.cos(jj / 2.3)
    Xt = ii * d + 1.3 * np.cos(jj / 2.7) - 0.8 * np.sin(ii / 4.1) + 0.15 * jj * d
    tm = (rng.random((nj, ni)) > 0.2).astype(np.int8)
    F = rng.normal(0, 3, (3, nj, ni)).astype(np.float32)
    F[0][rng.random((nj, ni)) < 0.05] = np.nan
    F[1][rng.random((nj, ni)) < 0.02] = np.inf
    return Yt, Xt, tm, F


def test_oracle_vectorised_equals_loop():
    """The vectorised oracle equals its per-buoy loop bit for bit on a curvilinear grid with land and non-finite
    values, positions anywhere in the 3 x 3 stencil (so some are clamped), masked buoys and out-of-range cells."""
    O = _ref()
    rng = np.random.default_rng(5)
    Yt, Xt, tm, F = _curvy(rng)
    n = 3000
    cell = np.stack([rng.integers(0, 30, n), rng.integers(0, 26, n)], 1)
    cell[rng.random(n) < 0.1, 0] |= 1 << 31
    jc, ic = np.clip(cell[:, 0] & 0x7fffffff, 1, 28), np.clip(cell[:, 1], 1, 24)
    yx = np.stack([Yt[jc, ic], Xt[jc, ic]], 1) + rng.uniform(-7, 7, (n, 2))
    m = (rng.random(n) > 0.1).astype(np.int8)
    for interp in ("cell", "bilinear"):
        a = O.sample(F, tm, cell, yx, m, interp, Yt, Xt)
        b = O.sample_loop(F, tm, cell, yx, m, interp, Yt, Xt)
        assert a.tobytes() == b.tobytes(), interp
        assert (a != FILL).sum() > n, interp


# ---- CPU: host-side checks, writers, CLI -------------------------------------------------------------

def test_host_side_checks():
    from sitrack_b200 import sample as S
    from sitrack_b200 import _lib
    assert S.check_interp("cell") == 0 and S.check_interp("bilinear") == 1
    for bad in ("nearest", None, 1):
        with pytest.raises(ValueError):
            S.check_interp(bad)
    with pytest.raises(ValueError):
        S.tpoints(None, 4, 5)
    with pytest.raises(ValueError):
        S.tpoints((np.zeros((4, 5)), np.zeros((5, 4))), 4, 5)
    Yt, Xt = _regular(4, 5, 3.0, 0.7)
    t = S.tpoints((Yt, Xt), 4, 5)
    assert t.shape == (20, 2) and t.flags["C_CONTIGUOUS"] and np.array_equal(t[:, 0], Yt.ravel()) and \
        np.array_equal(t[:, 1], Xt.ravel())
    # the quad pick assumes a right-handed grid: a mirrored one (i westward) and a degenerate one are refused, a grid
    # with a minority of inverted quads (a fold) is accepted
    for bad in ((Yt, -Xt), (Yt[::-1], Xt[::-1]), (np.full((4, 5), 1.0), np.full((4, 5), 2.0))):
        with pytest.raises(ValueError, match="right-handed"):
            S.tpoints(bad, 4, 5)
    Yf, Xf = _regular(8, 8, 3.0)
    Yf, Xf = Yf.copy(), Xf.copy()
    Yf[-1], Xf[-1] = Yf[-3], Xf[-3]                                     # the last row folded back
    assert S.tpoints((Yf, Xf), 8, 8).shape == (64, 2)
    # a NULL context is refused before anything else, on any machine
    L = _lib.lib()
    assert L.st_sample_dev(None, 1, 16, 100, None, 16, 0, None, 16, None) == -1
    assert b"st_sample_dev" in L.st_last_error(None)


def _wvals(js, nP):
    return dict(siconc=np.full(nP, 0.5 + js, np.float32), sithic=np.where(np.arange(nP) % 3, js, -9999.0))


def test_sample_writer_npz(tmp_path):
    import sitrack_b200 as sit
    f = str(tmp_path / "s.npz")
    ids = np.array([7, 3, 11, 5])
    with quiet(sit.SampleWriter, f, 3, ids, ["siconc", "sithic"], "bilinear", 6, units=dict(sithic="m"),
               corigin="X") as w:
        for js in range(3):
            w.write(js, 1000 + 6 * 3600 * js, _wvals(js, 4))
    z = np.load(f)
    assert sorted(z.files) == sorted(["time", "time_units", "id_buoy", "id_buoy_units", "siconc", "sithic",
                                      "sithic_units", "interp", "every", "FillValue"])
    assert z["time"].dtype == np.int32 and z["time"].tolist() == [1000, 22600, 44200]
    assert z["id_buoy"].dtype == np.int64 and z["id_buoy"].tolist() == ids.tolist()
    assert z["siconc"].dtype == np.float32 and z["siconc"].shape == (3, 4) and (z["siconc"][2] == 2.5).all()
    assert z["sithic"][1].tolist() == [-9999.0, 1.0, 1.0, -9999.0] and str(z["sithic_units"]) == "m"
    assert str(z["interp"]) == "bilinear" and int(z["every"]) == 6
    assert z["FillValue"].dtype == np.float32 and float(z["FillValue"]) == -9999.0


def test_sample_writer_netcdf_branch(monkeypatch, tmp_path):
    import types
    import sitrack_b200 as sit
    from test_cli import _FakeNC
    fake = types.ModuleType("netCDF4"); fake.Dataset = _FakeNC.Dataset
    monkeypatch.setitem(sys.modules, "netCDF4", fake)
    f = str(tmp_path / "s.nc")
    with quiet(sit.SampleWriter, f, 2, np.arange(5), ["siconc", "sithic"], "cell", 1,
               units=dict(siconc="1", sithic="m"), corigin="ORG") as w:
        for js in range(2):
            w.write(js, js, _wvals(js, 5))
    ds = _FakeNC.files[f]
    assert ds._dims == {"time": None, "buoy": 5}
    assert ds.attrs["Origin"] == "ORG" and ds.attrs["interp"] == "cell" and ds.attrs["every"] == 1
    v = ds.variables["sithic"]
    assert v.a.shape == (2, 5) and v.a.dtype == np.float32 and v.fill == np.float32(-9999.0) and v.units == "m"
    assert ds.variables["siconc"].units == "1" and ds.variables["time"].a.tolist() == [0, 1]
    assert ds.variables["id_buoy"].a.dtype == np.int64 and ds.variables["id_buoy"].a.tolist() == list(range(5))


def _add_var(r, name, arr):
    z = dict(np.load(r["si3"]))
    z[name] = arr
    np.savez(r["si3"], **z)


def _synth_argv(r, *extra):
    return ["si3_part_tracker.py", "-i", r["si3"], "-m", r["mesh"], "-s", r["seed"], "-F", "-N", "SYNTH4"] + list(extra)


@pytest.mark.parametrize("extra", [["--sample", "sinone"], ["--sample", "flat"], ["--sample", "short"],
                                   ["--sample", "siconc", "--sample-every", "1.5"],
                                   ["--sample", "siconc", "--sample-every", "0"],
                                   ["--sample", "siconc", "siconc"], ["--sample-every", "2"],
                                   ["--sample-interp", "bilinear"]])
def test_cli_sample_errors(tmp_path, monkeypatch, extra):
    """A variable missing from the SI3 file, a non-(t,y,x) variable, one of the wrong shape, HOURS that is not a
    multiple of the time step, a repeated variable and an option without --sample: ERROR lines printed before anything
    is written."""
    import si3_part_tracker as cli
    from make_synth_case import write_case
    r = write_case(str(tmp_path / "in"), grid="tiny", nrec=6, hss=3)
    U = r["records"][0]
    _add_var(r, "flat", U[0])
    _add_var(r, "short", U[:, :-1])
    d = tmp_path / "run"
    d.mkdir()
    monkeypatch.chdir(d)
    monkeypatch.setattr(sys, "argv", _synth_argv(r, *extra))
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf), pytest.raises(SystemExit):
        cli.main()
    assert any(l.startswith("ERROR") and "--sample" in l for l in buf.getvalue().splitlines()), buf.getvalue()[-800:]
    assert not os.listdir(d)


# ---- GPU ---------------------------------------------------------------------------------------

def _extra(T):
    """A second field on the golden grid: a smooth 'thickness' with NaNs on a few cells, one record per record."""
    IC = T["IC"]
    nrec, nj, ni = IC.shape
    jj, ii = np.meshgrid(np.arange(nj), np.arange(ni), indexing="ij")
    H = (1.0 + 0.5 * np.sin(jj / 4.0 + np.arange(nrec)[:, None, None] / 5.0) + 0.02 * ii).astype(np.float32)
    H[:, 7, 9] = np.nan
    H[:, 20:23, 15] = np.inf
    return H


def _stepped(T, g, name, physics=None, nrec=48):
    """The case stepped record by record with f8 rows, not chained: per row (0 .. nrec) the state's cells
    (get_state), the f8 row and its mask, in the caller's order -> (cells, yx, mask) lists."""
    c = TRACK_CASES[name]
    s = np.float32(c["scale"])
    import torch
    dev = torch.device("cuda", 0)
    first = T["win_first"] if c["win"] else None
    last = T["win_last"] if c["win"] else None
    eng = engine_for(g, uv_strategy=c["uv_strategy"], device=0)
    pos0, cell0 = T["pos0"], T["jiT0"].astype(np.int32)
    eng.set_buoys(pos0, cell0, first, last)
    m0 = np.ones(pos0.shape[0], np.int8) if first is None else (first - c["kstrt"] == 0).astype(np.int8)
    cells, rows, masks = [eng.get_state()[1]], [pos0.copy()], [m0]
    eng.record_slots(1)
    yx = torch.empty((pos0.shape[0], 2), dtype=torch.float64, device=dev)
    mk = torch.empty((pos0.shape[0],), dtype=torch.int8, device=dev)
    for k in range(nrec):
        st = eng.staging(0)
        st[0], st[1], st[2] = s * T["U"][k], s * T["V"][k], T["IC"][k]
        eng.submit_record(0)
        if physics:
            eng.step_ext(0, k + c["kstrt"], physics["scheme"], physics["interp"], physics["max_hops"], yx, None, mk)
        else:
            eng.step(0, k + c["kstrt"], yx, None, mk)
        torch.cuda.synchronize()
        cells.append(eng.get_state()[1]); rows.append(yx.cpu().numpy()); masks.append(mk.cpu().numpy())
    eng.close()
    return cells, rows, masks


def _oracle_rows(T, g, stepped, names, H, interp, every, nrec=48):
    O = _ref()
    cells, rows, masks = stepped
    out = {n: [] for n in names}
    for r in O.sampled_rows(nrec, every):
        k = O.row_record(r)
        F = np.stack([T["IC"][k] if n == "siconc" else H[k] for n in names])
        v = O.sample(F, g["tmask"], cells[r], rows[r], masks[r], interp, g["Yt"], g["Xt"])
        for i, n in enumerate(names):
            out[n].append(v[i])
    return {n: np.array(v) for n, v in out.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("interp", ["cell", "bilinear"])
@pytest.mark.parametrize("name", list(TRACK_CASES))
def test_sample_vs_oracle_stepped(torch, sit, gold_track, name, interp):
    """Every golden case stepped record by record: SampleFields on the engine's state, the f8 row and its mask (and
    on the state's own positions) equals the oracle on get_state()'s cells bit for bit, in both modes."""
    O = _ref()
    T, g = gold_track
    c = TRACK_CASES[name]
    s = np.float32(c["scale"])
    H = _extra(T)
    first = T["win_first"] if c["win"] else None
    eng = engine_for(g, uv_strategy=c["uv_strategy"], device=0)
    pos0 = T["pos0"]
    eng.set_buoys(pos0, T["jiT0"].astype(np.int32), first, T["win_last"] if c["win"] else None)
    eng.record_slots(1)
    dev = torch.device("cuda", 0)
    yx = torch.empty((pos0.shape[0], 2), dtype=torch.float64, device=dev)
    mk = torch.empty((pos0.shape[0],), dtype=torch.int8, device=dev)
    tyx = (g["Yt"], g["Xt"])
    m0 = np.ones(pos0.shape[0], np.int8) if first is None else (first - c["kstrt"] == 0).astype(np.int8)
    F0 = np.stack([T["IC"][0], H[0]])
    got = sit.SampleFields(eng, F0, m0, interp, tyx)
    ref = O.sample(F0, g["tmask"], eng.get_state()[1], pos0, m0, interp, g["Yt"], g["Xt"])
    assert got.tobytes() == ref.tobytes()
    valid = 0
    for k in range(48):
        st = eng.staging(0)
        st[0], st[1], st[2] = s * T["U"][k], s * T["V"][k], T["IC"][k]
        eng.submit_record(0)
        eng.step(0, k + c["kstrt"], yx, None, mk)
        torch.cuda.synchronize()
        row, m = yx.cpu().numpy(), mk.cpu().numpy()
        F = np.stack([T["IC"][k], H[k]])
        pos, cell, _ = eng.get_state()
        ref = O.sample(F, g["tmask"], cell, row, m, interp, g["Yt"], g["Xt"])
        got = sit.SampleFields(eng, F, m, interp, tyx, yx=row)
        assert got.tobytes() == ref.tobytes(), k
        got_state = sit.SampleFields(eng, F, m, interp, tyx)            # the state's positions: the same row
        assert got_state.tobytes() == ref.tobytes(), k
        valid += int((ref[0] != FILL).sum())
    eng.close()
    assert valid > 1000


def _track(T, g, name, rows, sample, sort=False, physics=None, nrec=48, sink=None):
    c = TRACK_CASES[name]
    s = np.float32(c["scale"])
    first = T["win_first"] if c["win"] else None
    last = T["win_last"] if c["win"] else None
    eng = engine_for(g, uv_strategy=c["uv_strategy"], device=0)
    eng.set_buoys(T["pos0"], T["jiT0"].astype(np.int32), first, last, sort=sort)
    res = eng.track((s * T["U"], s * T["V"], T["IC"]), nrec, kstrt=c["kstrt"], pos0=T["pos0"], rec_first=first,
                    row_dtype=rows, physics=physics, sample=sample, sink=sink)
    eng.close()
    return res


@pytest.mark.gpu
@pytest.mark.parametrize("interp", ["cell", "bilinear"])
@pytest.mark.parametrize("every", [1, 5, 48, 49])
@pytest.mark.parametrize("rows", ["f8", "f4"])
@pytest.mark.parametrize("name", ["uv1", "win", "fast"])
def test_track_sample(torch, sit, gold_track, name, rows, every, interp):
    """track(sample=...) equals the oracle over the stepped rows, bit for bit, with f8 (chained) and f4 rows, every
    n records, rec_first windows, buoys stored in the caller's order or sorted, kept or sent to a sink; the rows
    themselves are those of the same call without sampling."""
    T, g = gold_track
    H = _extra(T)
    names = ["sithic", "siconc"]
    ref = _oracle_rows(T, g, _stepped(T, g, name), names, H, interp, every)
    spec = dict(names=names, get=lambda k, n: H[k], every=every, interp=interp, tyx=(g["Yt"], g["Xt"]))
    plain = _track(T, g, name, rows, None)
    for sort in (False, True):
        res = _track(T, g, name, rows, spec, sort=sort)
        for n in names:
            assert res["sample"][n].shape == (48 // every + 1, 94) and res["sample"][n].dtype == np.float32
            assert res["sample"][n].tobytes() == ref[n].tobytes(), (n, sort)
        assert np.array_equal(res["posC"], plain["posC"]) and np.array_equal(res["mask"], plain["mask"])
    seen, order = [], []
    res = _track(T, g, name, rows, dict(spec, sink=lambda s, v: (seen.append((s, v)), order.append(("s", s)))),
                 sort=True, sink=lambda k, *a: order.append(("r", k + 1)))
    assert "sample" not in res and [s for s, _ in seen] == list(range(48 // every + 1))
    for s, v in seen:
        for n in names:
            assert v[n].tobytes() == ref[n][s].tobytes()
        assert order.index(("s", s)) < order.index(("r", max(s * every, 1)))   # a row's sample before its row


@pytest.mark.gpu
@pytest.mark.parametrize("interp", ["cell", "bilinear"])
def test_track_sample_physics(torch, sit, gold_track, interp):
    """With physics (RK4, C-grid linear, 3 hops) the samples equal the oracle over rows stepped with st_step_ext."""
    T, g = gold_track
    H = _extra(T)
    phys = dict(scheme=4, interp=1, max_hops=3)
    names = ["siconc", "sithic"]
    ref = _oracle_rows(T, g, _stepped(T, g, "fast", physics=phys), names, H, interp, 3)
    res = _track(T, g, "fast", "f8", dict(names=names, get=lambda k, n: H[k], every=3, interp=interp,
                                          tyx=(g["Yt"], g["Xt"])), physics=phys)
    for n in names:
        assert res["sample"][n].tobytes() == ref[n].tobytes(), n


@pytest.mark.gpu
def test_track_sample_siconc_slot_equals_extra_field(torch, sit, gold_track):
    """siconc read from the record slot equals siconc handed over as an extra field, in both modes; refusals."""
    T, g = gold_track
    for interp in ("cell", "bilinear"):
        res = _track(T, g, "win", "f4", dict(names=["siconc", "ic2"], get=lambda k, n: T["IC"][k], every=2,
                                             interp=interp, tyx=(g["Yt"], g["Xt"])))
        assert res["sample"]["siconc"].tobytes() == res["sample"]["ic2"].tobytes()
        assert (res["sample"]["siconc"] != FILL).sum() > 500
    eng = engine_for(g, device=0)
    eng.set_buoys(T["pos0"], T["jiT0"].astype(np.int32))
    rec = (T["U"], T["V"], T["IC"])
    with pytest.raises(ValueError, match="streaming record loop"):
        eng.track(rec, 48, chunk=8, sample=dict(names=["siconc"]))
    for bad in (dict(names=[]), dict(names=["siconc", "siconc"]), dict(names=["x"]), dict(names=["siconc"], every=0),
                dict(names=["siconc"], interp="nearest"), dict(names=["siconc"], interp="bilinear"),
                dict(names=["f%d" % i for i in range(17)], get=lambda k, n: T["IC"][k])):
        with pytest.raises(ValueError):
            eng.track(rec, 48, sink=lambda *a: None, sample=bad)
    eng.close()


@pytest.mark.gpu
def test_track_sample_killed_at_the_border(torch, sit, gold_track):
    """Four buoys one T-spacing from the four borders, pushed across by a uniform drift: the step kills them in
    cells jT = 1, jT = Nj-2, iT = 1, iT = Ni-2 with the row mask 1, and the bilinear stencil, which then reaches the
    grid's first or last row or column, equals the oracle."""
    O = _ref()
    T, g = gold_track
    Yt, Xt = g["Yt"], g["Xt"]
    Nj, Ni = Yt.shape
    cases = [((2, 20), (1, 20)), ((Nj - 3, 20), (Nj - 2, 20)), ((24, 2), (24, 1)), ((24, Ni - 3), (24, Ni - 2))]
    H = _extra(T)
    for (j, i), (j1, i1) in cases:
        dy, dx = Yt[j1, i1] - Yt[j, i], Xt[j1, i1] - Xt[j, i]
        U = np.full((1, Nj, Ni), dx * 1000.0 / 3600.0, np.float32)
        V = np.full((1, Nj, Ni), dy * 1000.0 / 3600.0, np.float32)
        IC = np.ones((1, Nj, Ni), np.float32)
        eng = engine_for(g, device=0)
        pos0 = np.array([[Yt[j, i], Xt[j, i]]])
        eng.set_buoys(pos0, np.array([[j, i]], np.int32))
        res = eng.track((U, V, IC), 1, pos0=pos0, sample=dict(names=["siconc", "h"], get=lambda k, n: H[5],
                                                               interp="bilinear", tyx=(Yt, Xt)))
        _, cell, alive = eng.get_state()
        eng.close()
        assert cell[0].tolist() == [j1, i1] and alive[0] == 0 and res["mask"][1, 0] == 1
        for r in (0, 1):
            ref = O.sample(np.stack([IC[0], H[5]]), g["tmask"], [[j, i]] if r == 0 else cell, res["posC"][r],
                           res["mask"][r], "bilinear", Yt, Xt)
            got = np.stack([res["sample"]["siconc"][r], res["sample"]["h"][r]])
            assert got.tobytes() == ref.tobytes() and (got != FILL).all()


@pytest.mark.gpu
def test_sample_entry_point_refusals(torch, sit, gold_track):
    """st_sample_dev refuses a NULL context, fields, mask or out, tyx NULL with interp 1, nF outside 1..16, a plane
    stride below Nj*Ni, an unknown interp and misaligned fields, out, yx or tyx; it writes nothing then."""
    from sitrack_b200 import _lib
    from sitrack_b200 import sample as S
    L = _lib.lib()
    T, g = gold_track
    dev = torch.device("cuda", 0)
    eng = engine_for(g, device=0)
    eng.set_buoys(T["pos0"], T["jiT0"].astype(np.int32))
    nP, plane = eng.nP, 48 * 40
    F = torch.from_numpy(np.ascontiguousarray(np.tile(T["IC"][0], (16, 1, 1)))).to(dev)
    mk = torch.ones((nP,), dtype=torch.int8, device=dev)
    yx = torch.from_numpy(T["pos0"]).to(dev)
    tyx = torch.from_numpy(S.tpoints((g["Yt"], g["Xt"]), 48, 40)).to(dev)
    out = torch.empty((17 * nP + 8,), dtype=torch.float32, device=dev)
    s = torch.cuda.current_stream(dev).cuda_stream

    def call(ctx=True, nF=2, fields=None, stride=plane, yx_p=None, mask=True, interp=1, tyx_p=None, out_p=None):
        out.fill_(3.0)
        torch.cuda.synchronize()
        rc = L.st_sample_dev(eng.h if ctx else None, nF, F.data_ptr() if fields is None else fields, stride,
                             yx.data_ptr() if yx_p is None else yx_p, mk.data_ptr() if mask else None, interp,
                             tyx.data_ptr() if tyx_p is None else tyx_p, out.data_ptr() if out_p is None else out_p, s)
        torch.cuda.synchronize()
        return rc

    assert call() == 0 and (out[:2 * nP] != 3.0).all()
    assert call(nF=16, interp=0, tyx_p=0) == 0 and call(nF=1, stride=10 ** 12) == 0
    for kw in (dict(ctx=False), dict(nF=0), dict(nF=17), dict(nF=-1), dict(fields=0), dict(mask=False),
               dict(out_p=0), dict(tyx_p=0), dict(interp=2), dict(interp=-1), dict(stride=plane - 1),
               dict(fields=F.data_ptr() + 2), dict(out_p=out.data_ptr() + 2), dict(yx_p=yx.data_ptr() + 8),
               dict(tyx_p=tyx.data_ptr() + 8)):
        assert call(**kw) == -1, kw
        assert (out == 3.0).all(), kw
    eng.close()


@pytest.mark.gpu
def test_cli_sample_end_to_end(tmp_path, monkeypatch):
    """si3_part_tracker.py -F --sort --sample siconc sithic --sample-every 3 --sample-interp bilinear on the 'small'
    synthetic case with a `sithic` variable added (NaN on masked cells): the file holds the oracle's values over the
    rows stepped on the same inputs, follows the tracking file's buoy axis, and the tracking files are byte-identical
    to a run without the flag."""
    import si3_part_tracker as cli
    import sitrack_b200 as sit
    from make_synth_case import write_case
    O = _ref()
    r = write_case(str(tmp_path / "in"), grid="small", nrec=24, hss=3)
    U, V, IC = r["records"]
    g0 = r["grid"]
    jj, ii = np.meshgrid(np.arange(U.shape[1]), np.arange(U.shape[2]), indexing="ij")
    sith = (1.5 + 0.3 * np.cos(jj / 7.0 + np.arange(24)[:, None, None] / 6.0) + 0.01 * ii).astype(np.float32)
    sith[:, g0["tmask"] == 0] = np.nan
    _add_var(r, "sithic", sith)
    runs = {}
    for tag, extra in (("plain", ["--sort"]), ("sample", ["--sort", "--sample", "siconc", "sithic", "--sample-every", "3",
                                                          "--sample-interp", "bilinear"])):
        d = tmp_path / tag
        d.mkdir()
        monkeypatch.chdir(d)
        monkeypatch.setattr(sys, "argv", _synth_argv(r, *extra))
        quiet(cli.main)
        runs[tag] = d
    files = sorted(os.listdir(runs["plain"] / "nc"))
    sfiles = [f for f in os.listdir(runs["sample"] / "nc") if "_sampled_" in f]
    assert sfiles == ["NEMO-SI3_SYNTH4_SYN00_sampled_nemoTsi3_idlSeed_19961215h00_19961216h00.npz"], sfiles
    assert sorted(set(os.listdir(runs["sample"] / "nc")) - set(sfiles)) == files
    for f in files:
        a, b = np.load(runs["plain"] / "nc" / f), np.load(runs["sample"] / "nc" / f)
        for k in a.files:
            assert a[k].tobytes() == b[k].tobytes(), (f, k)
    z = np.load(runs["sample"] / "nc" / sfiles[0])
    tr = np.load(runs["sample"] / "nc" / [f for f in files if "_tracking_" in f][0])
    assert np.array_equal(z["id_buoy"], tr["id_buoy"]) and np.array_equal(z["time"], tr["time"][::3])
    assert str(z["interp"]) == "bilinear" and int(z["every"]) == 3 and z["siconc"].shape == (9, tr["id_buoy"].size)
    # the oracle over the same buoys (the seeding cache, in the file's --sort order) stepped record by record
    cache = np.load(runs["sample"] / "seed" / os.listdir(runs["sample"] / "seed")[0])
    kmaskt, _, _, Yt, Xt, Yf, Xf, _ = quiet(sit.GetModelGrid, r["mesh"])
    Yv, Xv, Yu, Xu = quiet(sit.GetModelUVGrid, r["mesh"])
    vJ = cache["vJIt"]
    perm = np.argsort(vJ[:, 0].astype(np.int64) * U.shape[2] + vJ[:, 1], kind="stable")
    pos0, cell0 = cache["xPosC0"][perm], vJ[perm].astype(np.int32)
    assert np.array_equal(cache["IDs"][perm], tr["id_buoy"])
    import torch
    dev = torch.device("cuda", 0)
    with sit.TrackEngine(Yf, Xf, Yu, Xu, Yv, Xv, tmask=kmaskt, uv_strategy=1, rdt=3600.0, rmin_conc=sit.rmin_conc,
                         device=0) as eng:
        eng.set_buoys(pos0, cell0)
        eng.record_slots(1)
        n = pos0.shape[0]
        yx = torch.empty((n, 2), dtype=torch.float64, device=dev)
        mk = torch.empty((n,), dtype=torch.int8, device=dev)
        rows = [(eng.get_state()[1], pos0, np.ones(n, np.int8))]
        for k in range(24):
            st = eng.staging(0)
            st[0], st[1], st[2] = U[k], V[k], IC[k]
            eng.submit_record(0)
            eng.step(0, k, yx, None, mk)
            torch.cuda.synchronize()
            rows.append((eng.get_state()[1], yx.cpu().numpy(), mk.cpu().numpy()))
    for js, rr in enumerate(range(0, 25, 3)):
        k = O.row_record(rr)
        cell, p, m = rows[rr]
        ref = O.sample(np.stack([IC[k], sith[k]]), kmaskt, cell, p, m, "bilinear", Yt, Xt)
        assert z["siconc"][js].tobytes() == ref[0].tobytes() and z["sithic"][js].tobytes() == ref[1].tobytes(), js
    assert (z["sithic"] != FILL).sum() > 1000


@pytest.mark.gpu
@pytest.mark.timeout(300)
def test_cli_sample_under_torchrun(tmp_path):
    """`torchrun --nproc-per-node 2` (both ranks on cuda:0): each rank samples its block of buoys and rank 0 writes a
    _sampled_ file identical to the single-process run's, variable by variable."""
    import socket
    from make_synth_case import write_case
    r = write_case(str(tmp_path / "in"), grid="small", nrec=12, hss=2)
    _add_var(r, "sithic", (2.0 * r["records"][2]).astype(np.float32))
    cli = os.path.join(ROOT, "si3_part_tracker.py")
    common = ["-i", r["si3"], "-m", r["mesh"], "-s", r["seed"], "-F", "-N", "SYNTH4", "--device", "0",
              "--sample", "sithic", "siconc", "--sample-every", "2", "--sample-interp", "bilinear"]
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    one, two = tmp_path / "one", tmp_path / "two"
    one.mkdir(); two.mkdir()
    subprocess.run([sys.executable, cli] + common, cwd=one, env=env, check=True, stdout=subprocess.DEVNULL)
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                    "--master-addr", "127.0.0.1", "--master-port", str(port), cli] + common,
                   cwd=two, env=env, check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    files = sorted(os.listdir(one / "nc"))
    assert files == sorted(os.listdir(two / "nc")) and len(files) == 3
    f = [f for f in files if "_sampled_" in f][0]
    a, b = np.load(one / "nc" / f), np.load(two / "nc" / f)
    assert sorted(a.files) == sorted(b.files)
    for k in a.files:
        assert a[k].tobytes() == b[k].tobytes(), k
    assert a["sithic"].shape == (7, a["id_buoy"].size) and a["id_buoy"].size > 256
    assert (a["sithic"] != FILL).sum() > 1000


@pytest.mark.gpu
def test_bench_sample_small():
    """tools/bench_sample.py end to end on the small synthetic grid: exit 0, every configuration equal to the oracle."""
    import json
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_sample.py"), "--grid", "small", "--buoys",
                        "50000", "--check-buoys", "20000", "--seconds", "0.05"],
                       stdout=subprocess.PIPE, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    assert res["oracle_check_passed"] and res["step_us"] > 0 and set(res["sample"]) == {"cell_1", "cell_4",
                                                                                        "bilinear_1", "bilinear_4"}
