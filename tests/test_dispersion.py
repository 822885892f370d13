"""Two-particle (pair) dispersion over time lags, and its per-window statistics by initial separation
(sitrack_b200.dispersion, csrc/st_disperse.cu).

CPU: the oracle (oracle/dispersion_ref.py) against closed forms on dyadic inputs, MeshPairs and SeparationPairs, the
argument checks of the pairs, edges, lags and st_dispersion_scratch_bytes, both writer branches and the CLI's argument
errors.  GPU: the per-pair values bit for bit against the oracle, the statistics against the oracle (counts exact,
sums within 1e-11 of fsum) on the golden rows, a 200 k-buoy lattice and the edge cases, the fused multi-lag call
against one call per origin and two passes bit for bit, TrackEngine.track(dispersion=...) against the oracle in every
buoy storage order and row dtype, the entry point's refusals, the CLI end to end and a small run of the benchmark."""
import contextlib
import ctypes as C
import io
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import TRACK_CASES, engine_for
from test_deformation_scales import RDT, _lattice, _synth_argv, quiet

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FILL = -9999.0


def _pyth_cloud(scale=1.0):
    """Buoys on integer km positions, and pairs whose offsets are Pythagorean triples, so that every r0 is exact."""
    off = np.array([[3, 4], [4, 3], [5, 12], [12, 5], [8, 6], [-6, 8], [20, -21], [-9, -40], [7, 24], [0, 16],
                    [33, 56], [-48, 55], [65, -72], [0, -256], [-160, 231]], np.float64)
    base = np.stack(np.meshgrid(np.arange(0, 600.0, 37.0), np.arange(0, 900.0, 41.0), indexing="ij"), -1).reshape(-1, 2)
    yx = np.concatenate([base, (base[:, None] + off[None]).reshape(-1, 2)]) * scale
    nb = base.shape[0]
    a = np.repeat(np.arange(nb), off.shape[0])
    b = nb + np.arange(a.size)
    return yx, np.stack([a, b], 1).astype(np.int32)


# ---- CPU: the oracle ---------------------------------------------------------------------------

def test_oracle_translation_dilation_rotation():
    from oracle import dispersion_ref as O
    yx0, pairs = _pyth_cloud()
    one = np.ones(yx0.shape[0], np.int8)
    r0_exact = np.hypot(*(yx0[pairs[:, 0]] - yx0[pairs[:, 1]]).T)
    # a uniform translation by dyadic amounts: dr = dD2 = 0 exactly, every pair in the underflow stretch bin
    p = O.per_pair(yx0, yx0 + np.array([1.5, -2.25]), one, one, pairs)
    assert (p["dr"] == 0).all() and (p["dD2"] == 0).all() and np.array_equal(p["r0"], r0_exact)
    st = O.lag_stats(yx0, yx0 + np.array([1.5, -2.25]), one, one, pairs, 0.25)
    assert st["hist"][:, 0].sum() == pairs.shape[0] and st["hist"][:, 1:].sum() == 0
    # a dilation by 1 + 1/4 about the origin: dr = r0/4, dD2 = r0^2/16 exactly
    p = O.per_pair(yx0, yx0 * 1.25, one, one, pairs)
    assert np.array_equal(p["dr"], r0_exact / 4) and np.array_equal(p["dD2"], r0_exact ** 2 / 16)
    # a rotation by theta: |separation| is kept, dD2 = 2 r0^2 (1 - cos theta)
    th = 0.3
    R = np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]])
    p = O.per_pair(yx0, yx0 @ R.T, one, one, pairs)
    ref = 2 * r0_exact ** 2 * (1 - np.cos(th))
    assert (np.abs(p["dD2"] - ref) <= 1e-12 * ref).all() and (np.abs(p["dr"]) <= 1e-12 * r0_exact).all()


def test_oracle_classes_ties_and_zero_separation():
    """r0 exactly on a class edge goes to the upper class, s exactly on a bin edge to the upper bin, r0 = 0 to the
    overflow bin (s = inf or NaN)."""
    from oracle import dispersion_ref as O
    yx0 = np.array([[0.0, 0.0], [3.0, 4.0], [10.0, 10.0], [10.0, 10.0], [50.0, 50.0], [50.0, 50.0]])
    yx1 = np.array([[0.0, 0.0], [6.0, 8.0], [10.0, 10.0], [11.0, 10.0], [50.0, 50.0], [50.0, 50.0]])
    one = np.ones(6, np.int8)
    pairs = np.array([[0, 1], [2, 3], [4, 5]])
    st = O.lag_stats(yx0, yx1, one, one, pairs, 1.0, r_edges=[5.0, 20.0], bins=[0.5, 1.0, 2.0])
    # pair 0: r0 = 5 (class 1), r1 = 10, s = 5/5 = 1 (bin 2); pair 1: r0 = 0, s = inf; pair 2: s = NaN
    assert st["hist"].tolist() == [[0, 0, 0, 2], [0, 0, 1, 0], [0, 0, 0, 0]]


def test_mesh_pairs():
    import sitrack_b200 as sit
    yx, tri = _lattice(20)
    E = sit.MeshPairs(tri[np.random.default_rng(0).permutation(tri.shape[0])])
    ref = {tuple(sorted((int(t[j]), int(t[(j + 1) % 3])))) for t in tri for j in range(3)}
    assert E.dtype == np.int32 and sorted(ref) == [tuple(e) for e in E.tolist()]
    assert (E[:, 0] < E[:, 1]).all()
    n = 20
    assert E.shape[0] == 2 * n * (n - 1) + (n - 1) ** 2
    tri2 = sit.TriangulateCloud(np.random.default_rng(1).uniform(0, 100, (300, 2)))
    E2 = sit.MeshPairs(tri2)
    assert E2.shape[0] == len({tuple(sorted((int(t[j]), int(t[(j + 1) % 3])))) for t in tri2 for j in range(3)})


def test_separation_pairs():
    import sitrack_b200 as sit
    n = 400
    jj, ii = np.divmod(np.arange(n * n), n)
    yx = np.stack([jj * 2.5, ii * 2.5], 1).astype(np.float64)            # 1000 km a side
    P = sit.SeparationPairs(yx, 4.0, 400.0, 20000, seed=3)
    assert np.array_equal(P, sit.SeparationPairs(yx, 4.0, 400.0, 20000, seed=3))
    assert not np.array_equal(P, sit.SeparationPairs(yx, 4.0, 400.0, 20000, seed=4))
    assert P.dtype == np.int32 and (P[:, 0] != P[:, 1]).all() and P.min() >= 0 and P.max() < n * n
    assert (P[:, 0] < P[:, 1]).all() and np.unique(P, axis=0).shape[0] == P.shape[0]
    assert (np.lexsort(P.T[::-1]) == np.arange(P.shape[0])).all()         # sorted
    r = np.hypot(*(yx[P[:, 0]] - yx[P[:, 1]]).T)
    d1, d2 = ((r >= 4) & (r < 40)).sum(), ((r >= 40) & (r <= 400)).sum()
    assert P.shape[0] > 18000 and 0.8 < d1 / d2 < 1.25, (d1, d2)
    with pytest.raises(ValueError):
        sit.SeparationPairs(yx, 0.0, 10.0, 5)
    with pytest.raises(ValueError):
        sit.SeparationPairs(yx, 10.0, 10.0, 5)
    with pytest.raises(ValueError):
        sit.SeparationPairs(yx, 1.0, 10.0, 0)


@pytest.mark.parametrize("pairs", [np.zeros((0, 2), np.int32), [[0, 1, 2]], [0, 1], [[0, 10]], [[-1, 2]], [[3, 3]],
                                   [[0.5, 1.0]]])
def test_check_pairs_rejects(pairs):
    from sitrack_b200.dispersion import check_pairs
    with pytest.raises(ValueError):
        check_pairs(pairs, 10)


def test_edge_and_lag_checks():
    from sitrack_b200 import dispersion as P
    for bad in ([], [1.0, 1.0], [2.0, 1.0], [np.nan], np.arange(64.0) + 1):
        with pytest.raises(ValueError):
            P.check_edges(bad, P.DEFAULT_R_EDGES, P.MAX_CLASS_EDGES, "r_edges")
    with pytest.raises(ValueError):
        P.check_edges(np.arange(4097.0), P.DEFAULT_BIN_EDGES, P.MAX_EDGES, "bins")
    assert np.array_equal(P.check_edges(None, P.DEFAULT_R_EDGES, 63, "r_edges"), P.DEFAULT_R_EDGES)
    assert P.DEFAULT_R_EDGES[0] == 10.0 and P.DEFAULT_R_EDGES[-1] == 1000.0 and P.DEFAULT_R_EDGES.size == 9
    for bad in (0, 65, 2.5, -1):
        with pytest.raises(ValueError):
            P.check_lags(bad)
    assert P.check_lags(64) == 64 and P.check_lags(1.0) == 1


@pytest.mark.parametrize("case", [dict(nQ=0), dict(nQ=2 ** 31), dict(lags=0), dict(lags=65), dict(ncls=0),
                                  dict(ncls=64), dict(nedge=0), dict(nedge=4097), dict(ncls=13, nedge=3511),
                                  dict(lags=64, ncls=63, nedge=61), dict(out=None)])
def test_dispersion_scratch_bytes_rejects(case):
    """st_dispersion_scratch_bytes returns ST_EINVAL (-1) for each bad argument before any CUDA call, and leaves the
    output alone; the shared-memory limit is exact (13 class edges: 3510 bins fit, 3511 do not)."""
    from sitrack_b200 import _lib
    a = dict(nQ=1000, lags=1, ncls=9, nedge=61, out=True)
    a.update(case)
    out = C.c_int64(-5)
    rc = _lib.lib().st_dispersion_scratch_bytes(a["nQ"], a["lags"], a["ncls"], a["nedge"],
                                                C.byref(out) if a["out"] else None)
    assert rc == -1 and out.value == -5
    assert b"st_dispersion_scratch_bytes" in _lib.lib().st_last_error(None)


def test_dispersion_scratch_bytes_accepts():
    from sitrack_b200 import _lib
    out = C.c_int64(0)
    for nQ, lags, ncls, nedge in ((1, 1, 1, 1), (1000, 1, 13, 3510), (10 ** 8, 64, 9, 61)):
        assert _lib.lib().st_dispersion_scratch_bytes(nQ, lags, ncls, nedge, C.byref(out)) == 0
        grid = min(max(1, -(-nQ // 256)), 1184)
        assert out.value == grid * lags * (ncls + 1) * 4 * 8


def _writer_stats(jw, m, Cn, NB):
    return dict(n=np.full((m, Cn), jw + 1), sum_r0=np.full((m, Cn), 1.5 * jw), sum_dr=np.full((m, Cn), -0.5),
                sum_dr2=np.full((m, Cn), 0.25), sum_dD2=np.full((m, Cn), 2.0 + jw),
                hist_stretch=np.full((m, Cn, NB), jw))


def test_dispersion_writer_npz(tmp_path):
    import sitrack_b200 as sit
    lag, re, be = np.array([0.25, 0.5, 0.75]), np.array([10.0, 100.0]), np.array([0.01, 0.1, 1.0, 10.0])
    f = str(tmp_path / "d.npz")
    with quiet(sit.DispersionWriter, f, 2, lag, re, be, corigin="X") as w:
        for jw in range(2):
            w.write(jw, 100 + jw, 200 + jw, _writer_stats(jw, 3, 3, 5))
    z = np.load(f)
    assert z["time_start"].tolist() == [100, 101] and z["time_end"].dtype == np.int32
    assert np.array_equal(z["lag_days"], lag) and np.array_equal(z["r_edges"], re) and np.array_equal(z["bin_edges"], be)
    assert z["n"].dtype == np.int64 and z["n"].shape == (2, 3, 3) and (z["n"][1] == 2).all()
    assert z["hist_stretch"].shape == (2, 3, 3, 5) and z["hist_stretch"].dtype == np.int64 and (z["hist_stretch"][1] == 1).all()
    assert z["sum_dD2"].dtype == np.float64 and (z["sum_dD2"][1] == 3.0).all() and (z["sum_dr"] == -0.5).all()
    units = dict(lag_days="day", r_edges="km", bin_edges="day-1", n="1", sum_r0="km", sum_dr="km", sum_dr2="km2",
                 sum_dD2="km2", hist_stretch="1")
    for k, u in units.items():
        assert str(z[k + "_units"]) == u, k
    assert "FillValue" not in z.files


def test_dispersion_writer_netcdf_branch(monkeypatch, tmp_path):
    """The netCDF4 branch against the in-memory stand-in of test_cli: dimensions, variables, no fill values, units."""
    import types
    import sitrack_b200 as sit
    from test_cli import _FakeNC
    fake = types.ModuleType("netCDF4"); fake.Dataset = _FakeNC.Dataset
    monkeypatch.setitem(sys.modules, "netCDF4", fake)
    f = str(tmp_path / "d.nc")
    with quiet(sit.DispersionWriter, f, 3, [0.25, 0.5], [10.0, 100.0, 1000.0], [1.0, 2.0], corigin="ORG") as w:
        for jw in range(3):
            w.write(jw, jw, jw + 1, _writer_stats(jw, 2, 4, 3))
    ds = _FakeNC.files[f]
    assert ds._dims == {"time": None, "lag": 2, "class": 4, "bin": 3, "class_edge": 3, "bin_edge": 2}
    assert ds.attrs["Origin"] == "ORG"
    v = ds.variables["hist_stretch"]
    assert v.a.shape == (3, 2, 4, 3) and v.a.dtype == np.int64 and v.fill is None and (v.a[2] == 2).all()
    assert ds.variables["sum_r0"].fill is None and ds.variables["sum_r0"].units == "km"
    assert ds.variables["n"].a.tolist()[2] == [[3] * 4] * 2 and ds.variables["lag_days"].a.tolist() == [0.25, 0.5]
    assert ds.variables["time_end"].a.tolist() == [1, 2, 3]


@pytest.mark.parametrize("extra,env", [(["--dispersion", "0", "2"], {}), (["--dispersion", "1.5", "2"], {}),
                                       (["--dispersion", "6", "0"], {}), (["--dispersion", "6", "65"], {}),
                                       (["--dispersion", "6", "2.5"], {}),
                                       (["--dispersion", "6", "2", "--dispersion-pairs", "0", "10", "100"], {}),
                                       (["--dispersion", "6", "2", "--dispersion-pairs", "10", "0", "100"], {}),
                                       (["--dispersion", "6", "2", "--dispersion-pairs", "10", "50", "50"], {}),
                                       (["--dispersion-pairs", "10", "10", "100"], {}),
                                       (["--dispersion", "6", "2"], {"WORLD_SIZE": "2"})])
def test_cli_dispersion_argument_errors(tmp_path, monkeypatch, extra, env):
    """Each bad --dispersion / --dispersion-pairs argument is an ERROR line printed before anything is read or
    written."""
    import si3_part_tracker as cli
    monkeypatch.chdir(tmp_path)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    monkeypatch.setattr(sys, "argv", ["si3_part_tracker.py", "-i", "x.npz", "-m", "y.npz", "-s",
                                      "sitrack_seeding_nemoTsi3_19961215_00_HSS2.npz", "-F"] + extra)
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf), pytest.raises(SystemExit):
        cli.main()
    assert any(l.startswith("ERROR") and "--dispersion" in l for l in buf.getvalue().splitlines())
    assert not os.listdir(tmp_path)


def test_cli_dispersion_run_shorter_than_a_window(tmp_path, monkeypatch):
    import si3_part_tracker as cli
    from make_synth_case import write_case
    r = write_case(str(tmp_path / "in"), grid="tiny", nrec=6, hss=3)
    d = tmp_path / "run"
    d.mkdir()
    monkeypatch.chdir(d)
    monkeypatch.setattr(sys, "argv", _synth_argv(r, "--dispersion", "12", "2"))
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf), pytest.raises(SystemExit):
        cli.main()
    assert any(l.startswith("ERROR") and "--dispersion" in l for l in buf.getvalue().splitlines())
    assert not os.listdir(d)


# ---- GPU ---------------------------------------------------------------------------------------

def _bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.int64)


def _check_stats(got, ref_hist, ref_sums, ref_abs):
    """Counts and histograms exact, sums within 1e-11 fsum(|terms|)."""
    assert got["hist_stretch"].dtype == np.int64 and np.array_equal(got["hist_stretch"], ref_hist)
    assert np.array_equal(got["n"], ref_hist.sum(-1))
    for q, k in enumerate(("sum_r0", "sum_dr", "sum_dr2", "sum_dD2")):
        err = np.abs(got[k] - ref_sums[..., q])
        assert (err <= 1e-11 * ref_abs[..., q]).all(), (k, err.max())


def _vs_oracle(sit, yx0, yx1, m0, m1, pairs, dt, r_edges=None, bins=None):
    from oracle import dispersion_ref as O
    kw = {}
    if r_edges is not None:
        kw["r_edges"] = r_edges
    if bins is not None:
        kw["bins"] = bins
    pp, st = sit.PairDispersion(yx0, yx1, m0, m1, pairs, dt, **kw)
    ref = O.per_pair_filled(yx0, yx1, m0, m1, pairs)
    for j, k in enumerate(sit.PAIR_NAMES):
        assert np.array_equal(_bits(pp[k]), _bits(ref[j])), k
    rs = O.lag_stats(yx0, yx1, m0, m1, pairs, dt, **kw)
    _check_stats(st, rs["hist"][None], rs["sums"][None], rs["absum"][None])
    pp2, st2 = sit.PairDispersion(yx0, yx1, m0, m1, pairs, dt, **kw)          # two passes: the same bits
    for k in st:
        assert np.array_equal(_bits(st[k]) if st[k].dtype == np.float64 else st[k],
                              _bits(st2[k]) if st2[k].dtype == np.float64 else st2[k]), k
    return pp, st


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TRACK_CASES))
def test_pairs_vs_oracle_golden(sit, gold_track, name):
    """Every pair of the 94 golden buoys, both orders, between several pairs of golden rows: per-pair values bit for
    bit, statistics against the oracle."""
    T, _ = gold_track
    posC, mask = T[name + "_posC"], T[name + "_mask"]
    n = posC.shape[1]
    a, b = np.triu_indices(n, 1)
    pairs = np.concatenate([np.stack([a, b], 1), np.stack([b, a], 1)]).astype(np.int32)
    nv = 0
    for k0, k1 in [(0, 1), (0, 6), (5, 29), (12, 48), (47, 48)]:
        _, st = _vs_oracle(sit, posC[k0], posC[k1], mask[k0], mask[k1], pairs, (k1 - k0) * RDT / 86400.0,
                           r_edges=[1.0, 3.0, 10.0, 30.0, 100.0])
        nv += int(st["n"].sum())
    assert nv > 5000


def _lattice_case(rng, n=450):
    yx0, tri = _lattice(n, hole=(600.0, 700.0, 90.0), seed=3)
    nP = yx0.shape[0]
    yx1 = yx0 + 1.2 + np.stack([np.sin(yx0[:, 1] / 40.0), np.cos(yx0[:, 0] / 55.0)], 1) * 0.7
    jump = rng.choice(nP, 300, replace=False)
    yx1[jump] += rng.choice([-1.0, 1.0], (300, 2)) * 7.0
    m0 = (rng.random(nP) >= 0.02).astype(np.int8)
    m1 = m0 * (rng.random(nP) >= 0.03).astype(np.int8)                 # deaths: masked at the lag row only
    return yx0, yx1, m0, m1, tri


@pytest.mark.gpu
def test_pairs_vs_oracle_lattice(sit):
    """~200 k buoys with masks and deaths, mesh pairs and sampled pairs (10 to 1000 km)."""
    rng = np.random.default_rng(11)
    yx0, yx1, m0, m1, tri = _lattice_case(rng)
    pairs = np.concatenate([sit.MeshPairs(tri), sit.SeparationPairs(yx0, 10.0, 1000.0, 200000, seed=5)])
    _, st = _vs_oracle(sit, yx0, yx1, m0, m1, pairs, 0.25)
    assert (st["n"][0, 1:-1] > 1000).all() and st["n"][0, 0] > 400000
    assert st["n"].sum() < pairs.shape[0]


@pytest.mark.gpu
def test_pairs_ties_zero_separation_and_limits(sit):
    """r0 exactly on a class edge (a 3-4-5 pair against edge 5.0), s exactly on a bin edge, r0 = 0; then the largest
    class/bin shape the shared memory holds (13 class edges, 3510 bins) and one bin more refused."""
    yx0 = np.array([[0.0, 0.0], [3.0, 4.0], [10.0, 10.0], [10.0, 10.0], [50.0, 50.0], [50.0, 50.0]])
    yx1 = np.array([[0.0, 0.0], [6.0, 8.0], [10.0, 10.0], [11.0, 10.0], [50.0, 50.0], [50.0, 50.0]])
    one = np.ones(6, np.int8)
    pp, st = _vs_oracle(sit, yx0, yx1, one, one, [[0, 1], [2, 3], [4, 5]], 1.0, r_edges=[5.0, 20.0],
                        bins=[0.5, 1.0, 2.0])
    assert st["hist_stretch"][0].tolist() == [[0, 0, 0, 2], [0, 0, 1, 0], [0, 0, 0, 0]]
    assert pp["r0"].tolist() == [5.0, 0.0, 0.0] and pp["dr"].tolist() == [5.0, 1.0, 0.0]
    rng = np.random.default_rng(2)
    yx0, yx1, m0, m1, tri = _lattice_case(rng, 120)
    pairs = np.concatenate([sit.MeshPairs(tri), sit.SeparationPairs(yx0, 2.0, 300.0, 20000, seed=1)])
    from oracle import dispersion_ref as O
    p = O.per_pair(yx0, yx1, m0, m1, pairs)
    s = np.abs(p["dr"]) / (p["r0"] * 0.25)
    vals = np.unique(s[p["valid"] & np.isfinite(s)])
    # 1000 edges exactly on stretch rates that occur (ties), the rest spread over 1e-7 .. 1e4
    bins = np.unique(np.r_[vals[::max(1, vals.size // 1000)][:1000], 10.0 ** np.linspace(-7, 4, 3510)])[:3510]
    r0v = np.unique(p["r0"][p["valid"]])
    r_edges = r0v[::r0v.size // 14][1:14]                              # 13 edges exactly on separations that occur
    assert bins.size == 3510 and r_edges.size == 13
    _vs_oracle(sit, yx0, yx1, m0, m1, pairs, 0.25, r_edges=r_edges, bins=bins)
    with pytest.raises(sit.SitrackCudaError):
        sit.PairDispersion(yx0, yx1, m0, m1, pairs, 0.25, r_edges=r_edges, bins=np.r_[bins, bins[-1] * 2])


@pytest.mark.gpu
@pytest.mark.parametrize("nQ", [1, 255, 256, 257])
def test_pairs_vs_oracle_small_counts(sit, nQ):
    rng = np.random.default_rng(nQ)
    yx0 = rng.uniform(0, 2000.0, (600, 2))
    yx1 = yx0 + rng.normal(0, 3.0, yx0.shape)
    m0, m1 = (rng.random(600) > 0.05).astype(np.int8), (rng.random(600) > 0.05).astype(np.int8)
    a = rng.integers(0, 600, nQ)
    pairs = np.stack([a, (a + 1 + rng.integers(0, 599, nQ)) % 600], 1)
    _vs_oracle(sit, yx0, yx1, m0, m1, pairs, 0.5)


def _fused_and_single(torch, yx_rows, mk_rows, pairs, lags, dt, r_edges=None, bins=None):
    """Closing row = the last row; origins = the rows before it at lags 1..len-1.  -> (fused (hist, sums), single
    calls' (hist, sums) accumulated per lag)."""
    from sitrack_b200 import dispersion as P
    dev = torch.device("cuda", 0)
    t = lambda a, d: torch.from_numpy(np.ascontiguousarray(a, d)).to(dev)
    plan = P._Plan(torch, dev, pairs, lags, r_edges, bins)
    Y = [t(y, np.float64) for y in yx_rows]
    M = [t(m, np.int8) for m in mk_rows]
    nact = len(yx_rows) - 1
    s = torch.cuda.current_stream(dev)
    origins = [(Y[-1 - l], M[-1 - l], l) for l in range(1, nact + 1)]
    h, su = plan.outputs()
    plan.launch(None, Y[-1], M[-1], origins, dt, h, su, None, s)
    fused = (h.cpu().numpy(), su.cpu().numpy())
    hs, ss = np.zeros_like(fused[0]), np.zeros_like(fused[1])
    for o in origins:
        h1, s1 = plan.outputs()
        plan.launch(None, Y[-1], M[-1], [o], dt, h1, s1, None, s)
        h1, s1 = h1.cpu().numpy(), s1.cpu().numpy()
        assert not np.delete(h1, o[2] - 1, 0).any() and not np.delete(s1, o[2] - 1, 0).any()   # other lags zero
        hs[o[2] - 1], ss[o[2] - 1] = h1[o[2] - 1], s1[o[2] - 1]
    return fused, (hs, ss), plan


@pytest.mark.gpu
@pytest.mark.parametrize("lags,nact", [(1, 1), (8, 5), (64, 64)])
def test_fused_equals_single_origin_calls(torch, sit, lags, nact):
    """The fused call over nact origins gives, lag by lag, the bits of one single-origin call per lag, and the oracle's
    statistics; lags not active stay zero; two fused passes give the same bits."""
    from oracle import dispersion_ref as O
    rng = np.random.default_rng(lags)
    nP = 3000
    rows = [rng.uniform(0, 1500.0, (nP, 2))]
    for _ in range(nact):
        rows.append(rows[-1] + rng.normal(0.2, 2.0, (nP, 2)))
    masks = [np.ones(nP, np.int8)]
    for _ in range(nact):
        masks.append(masks[-1] * (rng.random(nP) > 0.01).astype(np.int8))
    pairs = sit.SeparationPairs(rows[0], 5.0, 1000.0, 20000, seed=lags)
    dt = 0.125
    fused, single, _ = _fused_and_single(torch, rows, masks, pairs, lags, dt)
    assert np.array_equal(fused[0], single[0]) and np.array_equal(_bits(fused[1]), _bits(single[1]))
    again, _, _ = _fused_and_single(torch, rows, masks, pairs, lags, dt)
    assert np.array_equal(again[0], fused[0]) and np.array_equal(_bits(again[1]), _bits(fused[1]))
    ref = O.window_stats(rows, masks, nact - 1, lags, dt, pairs=pairs)
    _check_stats(dict(hist_stretch=fused[0], n=fused[0].sum(-1), sum_r0=fused[1][..., 0], sum_dr=fused[1][..., 1],
                      sum_dr2=fused[1][..., 2], sum_dD2=fused[1][..., 3]), ref["hist"], ref["sums"], ref["absum"])
    assert fused[0][:nact].sum() > 0 and not fused[0][nact:].any() and not fused[1][nact:].any()


@pytest.mark.gpu
def test_entry_point_refusals(torch, sit):
    """st_dispersion_dev on real, aligned buffers refuses nQ < 1, dt_days <= 0 or NaN, no active lag, more active lags
    than `lags`, a repeated or out-of-range lag number and per-pair outputs with two origins; it writes nothing then."""
    from sitrack_b200 import _lib
    from sitrack_b200 import dispersion as P
    L = _lib.lib()
    dev = torch.device("cuda", 0)
    nP = 100
    yx = torch.zeros((nP, 2), dtype=torch.float64, device=dev)
    mk = torch.ones((nP,), dtype=torch.int8, device=dev)
    plan = P._Plan(torch, dev, np.stack([np.arange(50), np.arange(50, 100)], 1), 4)
    h, s = plan.outputs()
    pp = torch.full((4, 50), 7.0, dtype=torch.float64, device=dev)
    yp = (C.c_void_p * 5)(*[yx.data_ptr()] * 5)
    mp = (C.c_void_p * 5)(*[mk.data_ptr()] * 5)

    def call(nQ=50, nact=1, lag=(1,), dt=0.25, per_pair=False):
        h.fill_(-3); s.fill_(-3.0)
        torch.cuda.synchronize()
        lg = (C.c_int * 5)(*(list(lag) + [1] * (5 - len(lag))))
        rc = L.st_dispersion_dev(None, nQ, plan.pairs_t.data_ptr(), yx.data_ptr(), mk.data_ptr(), nact,
                                 C.cast(yp, C.c_void_p), C.cast(mp, C.c_void_p), C.cast(lg, C.c_void_p), dt, 4,
                                 plan.r_edges.size, plan.r_edges_t.data_ptr(), plan.bins.size, plan.bins_t.data_ptr(),
                                 plan.scratch.data_ptr(), plan.scratch_bytes, h.data_ptr(), s.data_ptr(),
                                 pp.data_ptr() if per_pair else None, None)
        torch.cuda.synchronize()
        return rc

    assert call() == 0 and int(h.sum()) == 50                           # every pair at r0 = 0: the overflow bin
    for kw in (dict(nQ=0), dict(nQ=-1), dict(dt=0.0), dict(dt=-1.0), dict(dt=float("nan")), dict(nact=0),
               dict(nact=5, lag=(1, 2, 3, 4, 1)), dict(nact=2, lag=(1, 1)), dict(lag=(5,)), dict(lag=(0,)),
               dict(nact=2, lag=(1, 2), per_pair=True)):
        assert call(**kw) == -1, kw
        assert (h.cpu().numpy() == -3).all() and (s.cpu().numpy() == -3.0).all() and (pp.cpu().numpy() == 7.0).all(), kw
    assert call(per_pair=True) == 0 and (pp.cpu().numpy()[0] == 0.0).all()


def _series_ref(posC, mask, pairs, every, lags, r_edges):
    from oracle import dispersion_ref as O
    return O.series_stats(posC, mask, pairs, every, lags, RDT, r_edges=r_edges)


def _engine(T, g, name, sort, rows, dispersion, deform=None):
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
                    row_dtype=rows, deform=deform, dispersion=dispersion)
    eng.close()
    return res, sh


@pytest.mark.gpu
@pytest.mark.parametrize("every,lags", [(6, 3), (1, 5), (12, 9)])
@pytest.mark.parametrize("rows", ["f8", "f4"])
@pytest.mark.parametrize("name", ["uv1", "win"])
def test_track_dispersion(torch, sit, gold_track, name, rows, every, lags):
    """track(dispersion=...): per-window statistics equal the oracle's over the series' rows, bit-identical whether
    the buoys are stored in the caller's order or sorted on the host or the device; lags past the number of windows
    stay zero."""
    T, g = gold_track
    sh = np.random.default_rng(7).permutation(T["pos0"].shape[0])
    posC, mask = T[name + "_posC"][:, sh], T[name + "_mask"][:, sh]
    n = sh.size
    a, b = np.triu_indices(n, 1)
    pairs = np.stack([a, b], 1).astype(np.int32)[::3]
    ref = _series_ref(posC, mask, pairs, every, lags, [1.0, 3.0, 10.0])
    first = None
    for sort in ("none", "host", "dev"):
        res, _ = _engine(T, g, name, sort, rows, dict(pairs=pairs, every=every, lags=lags, r_edges=[1.0, 3.0, 10.0]))
        got = res["dispersion"]
        assert len(got) == len(ref) == 48 // every and "deform" not in res
        for w, (st, rf) in enumerate(zip(got, ref)):
            assert np.array_equal(st["lag_days"], np.arange(1, lags + 1) * (every * RDT / 86400.0))
            assert st["hist_stretch"].shape == (lags, 4, 62)
            _check_stats(st, rf["hist"], rf["sums"], rf["absum"])
            assert not st["hist_stretch"][w + 1:].any() and not st["sum_r0"][w + 1:].any()
        if first is None:
            first = got
        for st, f in zip(got, first):
            for k in st:
                assert np.array_equal(st[k], f[k]), (sort, k)
    assert sum(int(st["n"].sum()) for st in first) > 1000


@pytest.mark.gpu
def test_track_dispersion_with_deform_and_sink(torch, sit, gold_track):
    """dispersion together with deform: the per-triangle outputs are those of the same call without dispersion, the
    dispersion statistics those of the call without deform; with a sink the windows arrive in order."""
    T, g = gold_track
    sh = np.random.default_rng(7).permutation(T["pos0"].shape[0])
    pos0 = T["pos0"][sh]
    tri = sit.TriangulateCloud(pos0)
    pairs = np.concatenate([sit.MeshPairs(tri), sit.SeparationPairs(pos0, 1.0, 30.0, 500)])
    disp = dict(pairs=pairs, every=6, lags=4)
    both, _ = _engine(T, g, "uv1", "host", "f8", disp, dict(tri=tri, every=4))
    plain, _ = _engine(T, g, "uv1", "host", "f8", None, dict(tri=tri, every=4))
    alone, _ = _engine(T, g, "uv1", "host", "f8", disp)
    assert "dispersion" not in plain and len(both["deform"]) == len(plain["deform"]) == 12
    for a, b in zip(both["deform"], plain["deform"]):
        for k in sit.DEFORM_NAMES:
            assert np.array_equal(a[k], b[k]), k
    for a, b in zip(both["dispersion"], alone["dispersion"]):
        for k in a:
            assert np.array_equal(a[k], b[k]), k
    seen = []
    eng = engine_for(g, device=0)
    eng.set_buoys(pos0, T["jiT0"][sh].astype(np.int32))
    r = eng.track((T["U"], T["V"], T["IC"]), 48, sink=lambda *a: None,
                  dispersion=dict(disp, sink=lambda w, st: seen.append((w, st))))
    assert [w for w, _ in seen] == list(range(8)) and "dispersion" not in r
    for (_, a), b in zip(seen, alone["dispersion"]):
        for k in a:
            assert np.array_equal(a[k], b[k]), k
    with pytest.raises(ValueError):
        eng.track((T["U"], T["V"], T["IC"]), 48, chunk=8, dispersion=disp)
    with pytest.raises(ValueError):
        eng.track((T["U"], T["V"], T["IC"]), 48, sink=lambda *a: None, dispersion=dict(disp, lags=65))
    eng.close()


@pytest.mark.gpu
def test_cli_dispersion_end_to_end(tmp_path, monkeypatch):
    """si3_part_tracker.py -F --dispersion 6 3 on the 'small' synthetic case: the file's statistics are those of the
    engine API on the same inputs bit for bit, and the tracking files are byte-identical to a run without the flag."""
    import si3_part_tracker as cli
    import sitrack_b200 as sit
    from make_synth_case import write_case
    r = write_case(str(tmp_path / "in"), grid="small", nrec=24, hss=3)
    runs = {}
    for tag, extra in (("plain", []), ("disp", ["--dispersion", "6", "3", "--dispersion-pairs", "3000", "5", "500"])):
        d = tmp_path / tag
        d.mkdir()
        monkeypatch.chdir(d)
        monkeypatch.setattr(sys, "argv", _synth_argv(r, *extra))
        quiet(cli.main)
        runs[tag] = d
    files = sorted(os.listdir(runs["plain"] / "nc"))
    dfiles = [f for f in os.listdir(runs["disp"] / "nc") if "_dispersion_" in f]
    assert dfiles == ["NEMO-SI3_SYNTH4_SYN00_dispersion_nemoTsi3_idlSeed_19961215h00_19961216h00.npz"], dfiles
    assert sorted(set(os.listdir(runs["disp"] / "nc")) - set(dfiles)) == files
    for f in files:
        a, b = np.load(runs["plain"] / "nc" / f), np.load(runs["disp"] / "nc" / f)
        assert sorted(a.files) == sorted(b.files)
        for k in a.files:
            assert a[k].dtype == b[k].dtype and a[k].tobytes() == b[k].tobytes(), (f, k)
    z = np.load(runs["disp"] / "nc" / dfiles[0])
    assert z["time_start"].shape == (4,) and z["hist_stretch"].shape == (4, 3, 10, 62)
    assert np.array_equal(z["lag_days"], [0.25, 0.5, 0.75]) and np.array_equal(z["r_edges"], sit.DEFAULT_R_EDGES)
    # the engine API on the CLI's inputs: seeds from its cache, the same pairs, grid and records
    seed = [f for f in os.listdir(runs["disp"] / "seed")][0]
    cache = np.load(runs["disp"] / "seed" / seed)
    imaskt, _, _, _, _, Yf, Xf, _ = quiet(sit.GetModelGrid, r["mesh"])
    Yv, Xv, Yu, Xu = quiet(sit.GetModelUVGrid, r["mesh"])
    U, V, IC = r["records"]
    pos0 = cache["xPosC0"]
    pairs = sit.SeparationPairs(pos0, 5.0, 500.0, 3000, seed=0)
    seen = []
    with sit.TrackEngine(Yf, Xf, Yu, Xu, Yv, Xv, tmask=imaskt, uv_strategy=1, rdt=3600.0, rmin_conc=sit.rmin_conc,
                         device=0) as eng:
        eng.set_buoys(pos0, cache["vJIt"])
        eng.track((U[:24], V[:24], IC[:24]), 24, sink=lambda *a: None, row_dtype="f4",
                  dispersion=dict(pairs=pairs, every=6, lags=3, sink=lambda w, st: seen.append(st)))
    assert len(seen) == 4
    for w, st in enumerate(seen):
        assert np.array_equal(z["n"][w], st["n"]) and np.array_equal(z["hist_stretch"][w], st["hist_stretch"])
        for k in ("sum_r0", "sum_dr", "sum_dr2", "sum_dD2"):
            assert np.array_equal(_bits(z[k][w]), _bits(st[k])), (w, k)
    assert z["n"][3].sum() > 1000 and z["n"][0, 1:].sum() == 0


@pytest.mark.gpu
def test_bench_dispersion_small():
    """tools/bench_dispersion.py end to end on a small lattice: exit 0, fused statistics bit-identical to the single
    calls and to a second pass."""
    import json
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_dispersion.py"), "--ny", "300", "--nx", "300",
                        "--sep-pairs", "100000", "--seconds", "0.05"], stdout=subprocess.PIPE, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    assert res["fused_equals_single_calls"] and res["run_to_run_identical"] and res["lags"] == 8
