"""Buoy transits between regions: per-buoy connectivity state, transitions, source-to-region counts and first-arrival
times (sitrack_b200.connect, csrc/st_connect.cu).

CPU: the oracle (oracle/connect_ref.py) on closed forms, the vectorised oracle against its per-buoy loop, the label
checks, st_connect_state_bytes at its limits, RegionConnectivity's argument checks, both writer branches and every CLI
ERROR line.  GPU: the per-buoy state after every sample and every window's statistics equal the oracle's exactly, on
the golden cases stepped record by record, a 200 k-buoy lattice, small and grid-saturating buoy counts, the shape
limits, a single hot bin and warps of distinct bins; the entry point's refusals; TrackEngine.track(connect=...) in
every buoy storage order and row dtype, with physics and next to every other analysis; the CLI end to end, alone and
under torchrun; a small run of the benchmark."""
import contextlib
import ctypes as C
import io
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from conftest import TRACK_CASES, engine_for
from test_sample import _stepped, _synth_argv, quiet

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("n_start", "n_end", "count", "trans", "n_arrive", "sum_tau", "sum_tau2", "hist_tau")
EDGES = [1.0, 2.0, 3.0, 5.0, 8.0]


def _ref():
    from oracle import connect_ref as O
    return O


def _same(a, b):
    for k in NAMES:
        assert np.asarray(a[k]).dtype == np.int64 and np.array_equal(a[k], b[k]), k


def _both(cells, masks, labels, R, tau_edges=EDGES, every=1):
    """The oracle run, checked against its per-buoy loop."""
    O = _ref()
    s1, w1 = O.run(cells, masks, labels, R, tau_edges, every)
    s2, w2 = O.run(cells, masks, labels, R, tau_edges, every, step=O.sample_loop)
    assert np.array_equal(s1, s2)
    for a, b in zip(w1, w2):
        _same(a, b)
    return s1, w1


def _total(wins):
    return {k: sum(w[k] for w in wins) for k in NAMES if k != "count"}


def _stripes(Nj=6, Ni=14, width=2):
    """Vertical stripes in i: region 1 + (i-1)//width on the interior columns."""
    lab = np.zeros((Nj, Ni), np.int64)
    lab[:, 1:Ni - 1] = 1 + (np.arange(Ni - 2) // width)
    return lab


def _one(path, masks=None, labels=None, R=None, nj=2):
    """One buoy through the cells (nj, i) for i in path (a cell (j, i) tuple passes through): -> oracle (states, wins)."""
    labels = _stripes() if labels is None else labels
    R = int(labels.max()) if R is None else R
    cells = [np.array([c if isinstance(c, tuple) else (nj, c)], np.int64) for c in path]
    masks = [np.ones(1, np.int8)] * len(path) if masks is None else [np.array([m], np.int8) for m in masks]
    return _both(cells, masks, labels, R)


# ---- CPU: the oracle ---------------------------------------------------------------------------

def test_oracle_stripe_walk_arrives_at_the_stripe_times():
    """One cell per sample eastward across stripes two cells wide: region r is first reached at t = 2(r-1)."""
    st, w = _one(list(range(1, 13)))
    tot = _total(w)
    assert tot["n_arrive"][1].tolist() == [0, 1, 1, 1, 1, 1]
    assert tot["sum_tau"][1].tolist() == [0, 2, 4, 6, 8, 10] and tot["sum_tau2"][1, 5] == 100
    assert tot["hist_tau"][1, 1].tolist() == [0, 0, 1, 0, 0, 0] and tot["hist_tau"][1, 5, 5] == 1
    assert tot["trans"][1, 1] == 1 and all(tot["trans"][r, r + 1] == 1 for r in range(1, 6))
    assert tot["n_start"].tolist() == [0, 1, 0, 0, 0, 0, 0] and tot["n_end"].sum() == 0
    assert st[-1, 0].tolist() == [1, 1, 6, 0, 0b111111]
    assert w[0]["n_start"][1] == 1 and w[1]["n_arrive"][1, 1] == 1 and w[0]["n_arrive"].sum() == 0
    assert w[4]["count"][1, 3] == 1 and w[4]["count"].sum() == 1                    # a snapshot at sample 5


def test_oracle_reentry_and_return_are_not_arrivals():
    """Regions 1, 2, 1, 2, 3: arrivals in 2 at t = 1 and in 3 at t = 4 only."""
    st, w = _one([1, 3, 1, 3, 5])
    tot = _total(w)
    assert tot["n_arrive"][1].tolist() == [0, 1, 1, 0, 0, 0] and tot["sum_tau"][1, 1:3].tolist() == [1, 4]
    assert tot["trans"][1, 2] == 2 and tot["trans"][2, 1] == 1 and tot["trans"][2, 3] == 1
    assert st[-1, 0].tolist() == [1, 1, 3, 0, 0b111]


def test_oracle_region_zero_gives_transitions_and_counts_only():
    lab = _stripes()
    lab[:, 1:5] = 0
    st, w = _one([1, 2, 3, 4, 3], labels=lab)
    tot = _total(w)
    assert tot["n_start"][0] == 1 and tot["trans"][0, 0] == 4 and tot["trans"].sum() == 4
    assert tot["n_arrive"].sum() == 0 and all(x["count"][0, 0] == 1 for x in w)
    assert st[-1, 0].tolist() == [1, 0, 0, 0, 0]
    st, w = _one([2, 5, 6, 2], labels=lab)                                 # 0 -> 3: an arrival from source 0
    assert _total(w)["n_arrive"][0, 2] == 1 and _total(w)["sum_tau"][0, 2] == 1 and w[2]["count"][0, 0] == 1


def test_oracle_late_start_times_from_its_own_start():
    st, w = _one([1, 1, 1, 3, 5], masks=[0, 0, 1, 1, 1])
    tot = _total(w)
    assert st[0, 0, 0] == 0 and st[1, 0].tolist() == [1, 1, 1, 2, 1] and w[1]["n_start"][1] == 1
    assert tot["sum_tau"][1, 1:3].tolist() == [1, 2] and w[0]["count"].sum() == 0 and w[1]["count"][1, 1] == 1


def test_oracle_death_ends_for_good():
    st, w = _one([1, 3, 3, 5, 7], masks=[1, 1, 0, 1, 1])
    tot = _total(w)
    assert tot["n_end"].tolist() == [0, 1, 0, 0, 0, 0, 0] and tot["n_arrive"].sum() == 1
    assert st[1, 0, 0] == 2 and st[-1, 0].tolist() == st[1, 0].tolist()
    assert all(x["count"].sum() == 0 and x["trans"].sum() == 0 for x in w[1:])


def test_oracle_cell_outside_the_interior_ends_a_buoy():
    for bad in ((0, 3), (5, 3), (2, 0), (2, 13), (-1, 3), (2, 99)):
        st, w = _one([1, bad, 3])
        assert st[0, 0, 0] == 2 and _total(w)["n_end"][1] == 1, bad
    st, w = _one([(0, 1), 1, 3])                                           # not valid before the start: a late start
    assert st[0, 0].tolist() == [1, 1, 1, 1, 1]


def test_oracle_bit31_cell_is_read_stripped():
    dead = np.int64(-2 ** 31)
    st, w = _one([(2 | dead, 1), (2 | dead, 3), (2, 5)])
    assert st[-1, 0].tolist() == [1, 1, 3, 0, 0b111] and _total(w)["sum_tau"][1, 1:3].tolist() == [1, 2]


def test_oracle_sample_zero_adds_no_count():
    O = _ref()
    cells = [np.array([[2, 1], [2, 3], [0, 0]])] * 2
    s0, e0 = O.sample(O.new_state(3), _stripes(), 6, cells[0], np.ones(3), 0)
    assert e0["count"].sum() == 0 and e0["n_start"].tolist() == [0, 1, 1, 0, 0, 0, 0]
    _, w = _both(cells, [np.ones(3, np.int8)] * 2, _stripes(), 6)
    assert np.array_equal(w[0]["count"], np.diag(w[0]["n_start"]))


def _walk(rng, nP, S, Nj, Ni, out=True):
    """Random cell walks with deaths, late starts, cells off the interior and bit-31 cells."""
    cells = [np.stack([rng.integers(1, Nj - 1, nP), rng.integers(1, Ni - 1, nP)], 1)]
    for s in range(S):
        c = cells[-1] + rng.integers(-1, 2, (nP, 2))
        if out:
            c[:, 0], c[:, 1] = c[:, 0].clip(-1, Nj), c[:, 1].clip(-1, Ni)
        else:
            c[:, 0], c[:, 1] = c[:, 0].clip(1, Nj - 2), c[:, 1].clip(1, Ni - 2)
        cells.append(c)
    cells = [c.copy() for c in cells]
    if out:
        for c in cells:
            c[rng.choice(nP, max(1, nP // 50), replace=False), 0] |= np.int64(-2 ** 31)
    masks = [(rng.random(nP) > 0.2).astype(np.int8)]
    for s in range(S):
        masks.append(((masks[-1] | (rng.random(nP) < 0.2)) & (rng.random(nP) > 0.02)).astype(np.int8))
    return cells, masks


def _labels(rng, Nj, Ni, R):
    lab = rng.integers(0, R + 1, (Nj, Ni))
    lab[rng.random((Nj, Ni)) < 0.3] = R                                    # some blocks of one region
    return lab


@pytest.mark.parametrize("R", [1, 31])
def test_oracle_vectorised_equals_loop_on_random_walks(R):
    rng = np.random.default_rng(R)
    Nj, Ni = 14, 18
    cells, masks = _walk(rng, 500, 30, Nj, Ni)
    lab = _labels(rng, Nj, Ni, R)
    for every in (1, 4):
        st, w = _both(cells, masks, lab, R, every=every)
    tot = _total(w)
    assert tot["n_end"].sum() > 100 and tot["n_start"].sum() > 400 and (R == 1 or tot["n_arrive"].sum() > 300)


def test_check_labels():
    from sitrack_b200 import connect as K
    lab, R = K.check_labels(np.array([[0, 1], [3, 2.0]]), 2, 2)
    assert lab.dtype == np.uint8 and lab.flags["C_CONTIGUOUS"] and R == 3 and lab.tolist() == [[0, 1], [3, 2]]
    m = np.ma.masked_array([[np.nan, 5.0], [1.0, 40.0]], mask=[[True, False], [False, True]])
    lab, R = K.check_labels(m, 2, 2)
    assert lab.tolist() == [[0, 5], [1, 0]] and R == 5
    assert K.check_labels(np.full((2, 3), 31), 2, 3)[1] == 31 and K.check_labels(np.ones((1, 1), bool), 1, 1)[1] == 1
    for bad in (np.ones((2, 3)), np.ones((3, 2)), np.ones(6), [[0, -1], [1, 1]], [[0, 32], [1, 1]], [[0, 1.5], [1, 1]],
                [[0, np.nan], [1, 1]], [[0, np.inf], [1, 1]], np.zeros((2, 2)), [["a", "b"], ["c", "d"]]):
        with pytest.raises(ValueError):
            K.check_labels(bad, 2, 2)


@pytest.mark.parametrize("case", [dict(nP=0), dict(nP=2 ** 31), dict(R=0), dict(R=32), dict(ntau=0), dict(ntau=513),
                                  dict(out=None)])
def test_connect_state_bytes_rejects(case):
    """st_connect_state_bytes returns ST_EINVAL (-1) one past each limit, before any CUDA call, and leaves the output
    alone."""
    from sitrack_b200 import _lib
    a = dict(nP=1000, R=31, ntau=17, out=True)
    a.update(case)
    out = C.c_int64(-5)
    rc = _lib.lib().st_connect_state_bytes(a["nP"], a["R"], a["ntau"], C.byref(out) if a["out"] else None)
    assert rc == -1 and out.value == -5
    assert b"st_connect_state_bytes" in _lib.lib().st_last_error(None)


def test_connect_state_bytes_accepts():
    """Each limit exactly; 31 regions need 28 288 B of shared-memory counters, inside the 48 KB of a block."""
    from sitrack_b200 import _lib
    out = C.c_int64(0)
    for nP, R, ntau in ((1, 1, 1), (2 ** 31 - 1, 31, 512), (1000, 5, 17)):
        assert _lib.lib().st_connect_state_bytes(nP, R, ntau, C.byref(out)) == 0
        assert out.value == 8 * nP
    R1 = 32
    assert 16 * R1 * 31 + 4 * (2 * R1 + 2 * R1 * R1 + R1 * 31) == 28288 < 48 * 1024


def test_region_connectivity_refusals():
    import sitrack_b200 as sit
    rng = np.random.default_rng(0)
    cells, masks = _walk(rng, 20, 3, 8, 9, out=False)
    ok = dict(cells=np.array(cells), masks=np.array(masks), labels=np.ones((8, 9)), sample_days=0.5)
    for bad in (dict(cells=np.array(cells)[:1], masks=np.array(masks)[:1]), dict(cells=np.array(cells)[..., :1]),
                dict(cells=np.array(cells)[:, :0], masks=np.array(masks)[:, :0]), dict(masks=np.array(masks)[:, :5]),
                dict(cells=np.array(cells).astype(float)), dict(sample_days=0.0), dict(sample_days=np.nan),
                dict(labels=np.zeros((8, 9))), dict(labels=np.ones(72)), dict(labels=np.full((8, 9), 32))):
        kw = dict(ok)
        kw.update(bad)
        with pytest.raises(ValueError):
            sit.RegionConnectivity(**kw)


def _writer_stats(jw, R, NB):
    R1 = R + 1
    return dict(n_start=np.full(R1, jw), n_end=np.full(R1, jw + 1), count=np.full((R1, R1), jw + 2),
                trans=np.full((R1, R1), 3), n_arrive=np.full((R1, R), 4), sum_tau=np.full((R1, R), 7 * jw),
                sum_tau2=np.full((R1, R), 2 ** 40 + jw), hist_tau=np.full((R1, R, NB), jw + 5))


def test_connectivity_writer_npz(tmp_path):
    import sitrack_b200 as sit
    te = np.array([1.0, 2.0, 4.0])
    f = str(tmp_path / "c.npz")
    with quiet(sit.ConnectivityWriter, f, 2, 3, te, 0.25, corigin="X") as w:
        for jw in range(2):
            w.write(jw, 100 + jw, 200 + jw, _writer_stats(jw, 3, 4))
    z = np.load(f)
    assert z["time_start"].tolist() == [100, 101] and z["time_end"].dtype == np.int32
    assert np.array_equal(z["tau_edges"], te) and float(z["sample_days"]) == 0.25
    shapes = dict(n_start=(2, 4), n_end=(2, 4), count=(2, 4, 4), trans=(2, 4, 4), n_arrive=(2, 4, 3),
                  sum_tau=(2, 4, 3), sum_tau2=(2, 4, 3), hist_tau=(2, 4, 3, 4))
    for k, sh in shapes.items():
        assert z[k].shape == sh and z[k].dtype == np.int64, k
    assert (z["sum_tau2"][1] == 2 ** 40 + 1).all() and (z["hist_tau"][1] == 6).all() and (z["count"][0] == 2).all()
    units = dict(tau_edges="sample", n_start="1", n_end="1", count="1", trans="1", n_arrive="1", sum_tau="sample",
                 sum_tau2="sample2", hist_tau="1", time_start=sit.tunits_default)
    for k, u in units.items():
        assert str(z[k + "_units"]) == u, k
    assert "FillValue" not in z.files


def test_connectivity_writer_netcdf_branch(monkeypatch, tmp_path):
    """The netCDF4 branch against the in-memory stand-in of test_cli: dimensions, variables, no fill values, units,
    the sample_days attribute."""
    import types
    import sitrack_b200 as sit
    from test_cli import _FakeNC
    fake = types.ModuleType("netCDF4"); fake.Dataset = _FakeNC.Dataset
    monkeypatch.setitem(sys.modules, "netCDF4", fake)
    f = str(tmp_path / "c.nc")
    with quiet(sit.ConnectivityWriter, f, 3, 2, [1.0, 2.0], 0.5, corigin="ORG") as w:
        for jw in range(3):
            w.write(jw, jw, jw + 1, _writer_stats(jw, 2, 3))
    ds = _FakeNC.files[f]
    assert ds._dims == {"time": None, "region": 3, "dest": 2, "tau_bin": 3, "tau_edge": 2}
    assert ds.attrs["Origin"] == "ORG" and ds.attrs["sample_days"] == 0.5
    v = ds.variables["hist_tau"]
    assert v.a.shape == (3, 3, 2, 3) and v.a.dtype == np.int64 and v.fill is None and (v.a[2] == 7).all()
    assert ds.variables["count"].a.shape == (3, 3, 3) and ds.variables["count"].fill is None
    assert ds.variables["sum_tau"].units == "sample" and ds.variables["sum_tau2"].units == "sample2"
    assert ds.variables["time_end"].a.tolist() == [1, 2, 3] and ds.variables["tau_edges"].a.tolist() == [1.0, 2.0]


def _regions_file(tmp_path, r, **arrays):
    fn = str(tmp_path / "regions.npz")
    np.savez(fn, **arrays)
    return fn


@pytest.mark.parametrize("extra", [["--connect", "2"], ["--connect-regions", "REG", "lab"],
                                   ["--connect", "1.5", "--connect-regions", "REG", "lab"],
                                   ["--connect", "0", "--connect-regions", "REG", "lab"],
                                   ["--connect", "2", "--connect-regions", "nofile.npz", "lab"],
                                   ["--connect", "2", "--connect-regions", "REG", "nolab"],
                                   ["--connect", "2", "--connect-regions", "REG", "flat"],
                                   ["--connect", "2", "--connect-regions", "REG", "short"],
                                   ["--connect", "2", "--connect-regions", "REG", "big"],
                                   ["--connect", "2", "--connect-regions", "REG", "neg"],
                                   ["--connect", "2", "--connect-regions", "REG", "half"],
                                   ["--connect", "2", "--connect-regions", "REG", "zero"],
                                   ["--connect", "12", "--connect-regions", "REG", "lab"],
                                   ["--connect", "1", "--connect-regions", "REG", "lab"]])
def test_cli_connect_errors(tmp_path, monkeypatch, extra):
    """One flag without the other, HOURS that is not a multiple of the time step, a missing file or variable, a
    variable that is not (y,x) after its first plane, bad labels, a run shorter than one window and (with MAX_SAMPLES
    lowered to 5) more windows than a run may have: ERROR lines printed before anything is written."""
    import si3_part_tracker as cli
    import sitrack_b200 as sit
    from make_synth_case import write_case
    r = write_case(str(tmp_path / "in"), grid="tiny", nrec=6, hss=3)
    nj, ni = r["records"][0].shape[1:]
    lab = np.ones((nj, ni), np.int16)
    reg = _regions_file(tmp_path, r, lab=lab[None, None], flat=lab[0], short=lab[:, :-1], big=lab * 32, neg=-lab,
                        half=lab * 0.5, zero=lab * 0)
    extra = [reg if a == "REG" else a for a in extra]
    d = tmp_path / "run"
    d.mkdir()
    monkeypatch.chdir(d)
    if extra[1] == "1":
        monkeypatch.setattr(sit, "MAX_SAMPLES", 5)                        # 6 windows of one record
    monkeypatch.setattr(sys, "argv", _synth_argv(r, *extra))
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf), pytest.raises(SystemExit):
        cli.main()
    assert any(l.startswith("ERROR") and "--connect" in l for l in buf.getvalue().splitlines()), buf.getvalue()[-800:]
    assert not os.listdir(d)


# ---- GPU ---------------------------------------------------------------------------------------

def _c32(torch, dev, cells):
    a = (np.asarray(cells).astype(np.int64) & 0xffffffff).astype(np.uint32).view(np.int32)
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _device_run(torch, cells, masks, labels, R, tau_edges=EDGES, every=1):
    """One st_connect_dev per sample through connect._Plan on explicit cells, as the engine drives it: -> (states
    (S, nP, 5) after each window, the windows' stats)."""
    from sitrack_b200 import connect as K
    dev = torch.device("cuda", 0)
    g = lambda a: torch.from_numpy(np.ascontiguousarray(np.asarray(a) != 0, np.int8)).to(dev)
    lab = np.ascontiguousarray(labels, np.uint8)
    plan = K._Plan(torch, dev, lab, R, lab.shape[0], lab.shape[1], len(cells[0]), tau_edges, 0.25)
    s = torch.cuda.current_stream(dev)
    o0 = plan.outputs()
    plan.start(None, g(masks[0]), o0, s, cell_t=_c32(torch, dev, cells[0]))
    states, wins = [], []
    for w in range((len(cells) - 1) // every):
        k = (w + 1) * every
        o = o0 if w == 0 else plan.outputs()
        plan.window(None, None, None, g(masks[k]), 0.25, o, s, cell_t=_c32(torch, dev, cells[k]))
        d = plan.state_dict()
        states.append(np.stack([d[n] for n in ("status", "src", "prev", "start", "visited")], 1))
        wins.append(plan.results((o[0].cpu(),))[0])
    return np.array(states), wins


def _vs_oracle(torch, cells, masks, labels, R, tau_edges=EDGES, every=1):
    O = _ref()
    st, wins = _device_run(torch, cells, masks, labels, R, tau_edges, every)
    rs, rw = O.run(cells, masks, labels, R, tau_edges, every)
    assert st.shape == rs.shape and np.array_equal(st, rs)
    assert len(wins) == len(rw)
    for a, b in zip(wins, rw):
        _same(a, b)
        assert a["nreg"] == R and np.array_equal(a["tau_edges"], tau_edges)
    return _total(wins)


def _gold_maps(g):
    Nj, Ni = g["tmask"].shape
    jj, ii = np.meshgrid(np.arange(Nj), np.arange(Ni), indexing="ij")
    return {"i": (1 + ii % 7, 7), "j": (np.where(jj % 9 == 4, 0, 1 + jj % 31), 31)}


@pytest.mark.gpu
@pytest.mark.parametrize("stripes", ["i", "j"])
@pytest.mark.parametrize("name", list(TRACK_CASES))
def test_connect_vs_oracle_golden(torch, gold_track, name, stripes):
    """Every golden case stepped record by record, cells from get_state(): state after each sample and each window's
    statistics equal the oracle's, on stripe maps in i and in j that the golden buoys cross."""
    T, g = gold_track
    cells, _, masks = _stepped(T, g, name)
    lab, R = _gold_maps(g)[stripes]
    tot = _vs_oracle(torch, cells, masks, lab, R)
    assert tot["n_arrive"].sum() > 20 and tot["n_start"].sum() > 50


@pytest.mark.gpu
@pytest.mark.parametrize("every", [1, 2])
def test_connect_vs_oracle_lattice(torch, every):
    """The 200 k-buoy lattice of DESIGN section 11 moving over a 5 km cell grid, with deaths, late starts and buoys
    that leave the grid, on 31 block regions."""
    from test_deformation_scales import _lattice
    rng = np.random.default_rng(11)
    yx, _ = _lattice(450, hole=(600.0, 700.0, 90.0), seed=3)
    nP = yx.shape[0]
    Nj, Ni = 290, 290
    cells, masks = [], [(rng.random(nP) >= 0.02).astype(np.int8)]
    for s in range(7):
        cells.append(np.stack([np.floor(yx[:, 0] / 5.0), np.floor(yx[:, 1] / 5.0)], 1).astype(np.int64) + 1)
        yx = yx * 1.01 + 1.2 + rng.normal(0.0, 2.5, yx.shape)
        masks.append(masks[-1] * (rng.random(nP) >= 0.01).astype(np.int8))
    masks = masks[:7]
    masks[2][rng.choice(nP, 500, replace=False)] = 1                      # late starts
    jj, ii = np.meshgrid(np.arange(Nj), np.arange(Ni), indexing="ij")
    lab = 1 + ((jj // 50) * 6 + ii // 50) % 31
    lab[100:120, :] = 0
    tot = _vs_oracle(torch, cells, masks, lab, 31, every=every)
    assert tot["n_arrive"].sum() > 1000 and tot["n_end"].sum() > 1000


@pytest.mark.gpu
@pytest.mark.parametrize("nP", [1, 255, 256, 257, 700001])
def test_connect_vs_oracle_buoy_counts(torch, nP):
    """One buoy, a block's edges and more buoys than one wave of resident blocks holds (grid-strided)."""
    rng = np.random.default_rng(nP)
    cells, masks = _walk(rng, nP, 10, 30, 40)
    tot = _vs_oracle(torch, cells, masks, _labels(rng, 30, 40, 12), 12)
    assert nP < 256 or tot["n_arrive"].sum() > nP // 4


@pytest.mark.gpu
@pytest.mark.parametrize("R,ntau", [(1, 1), (1, 512), (31, 1), (31, 512)])
def test_connect_vs_oracle_shape_limits(torch, R, ntau):
    rng = np.random.default_rng(R * 1000 + ntau)
    cells, masks = _walk(rng, 40000, 30, 20, 24)
    tau_edges = np.arange(1.0, ntau + 1) * (30.0 / ntau)
    tot = _vs_oracle(torch, cells, masks, _labels(rng, 20, 24, R), R, tau_edges)
    assert tot["n_end"].sum() > 1000 and (R == 1 or tot["n_arrive"].sum() > 10000)


@pytest.mark.gpu
def test_connect_hot_bin_and_distinct_bins(torch):
    """One region everywhere, buoys stored cell-major: every lane of every warp in one bin.  Then warps whose 32
    lanes have 32 distinct sources, transitions and arrivals."""
    rng = np.random.default_rng(3)
    Nj, Ni = 60, 70
    cells, masks = _walk(rng, 300000, 8, Nj, Ni, out=False)
    order = np.argsort(cells[0][:, 0] * Ni + cells[0][:, 1], kind="stable")
    cells = [c[order] for c in cells]
    masks = [np.ones(300000, np.int8)] + [m[order] | 1 for m in masks[1:]]
    masks[5][::97] = 0
    tot = _vs_oracle(torch, cells, masks, np.ones((Nj, Ni), np.int64), 1)
    assert tot["trans"][1, 1] > 1_000_000 and tot["n_arrive"].sum() == 0
    nP, Ni = 32 * 4000, 70
    lab = np.zeros((8, Ni), np.int64)
    lab[:, 1:Ni - 1] = np.arange(Ni - 2) % 32                             # column i: region (i-1) % 32
    lane = np.arange(nP) % 32
    cells = [np.stack([np.full(nP, 3), 1 + (lane + 3 * t) % 64], 1) for t in range(12)]
    tot = _vs_oracle(torch, cells, [np.ones(nP, np.int8)] * 12, lab, 31)
    assert tot["n_start"].tolist() == [nP // 32] * 32 and tot["n_arrive"].sum() > nP * 5


@pytest.mark.gpu
def test_region_connectivity(sit):
    """The host entry point: final state and windows equal the oracle's."""
    O = _ref()
    rng = np.random.default_rng(4)
    cells, masks = _walk(rng, 3000, 12, 16, 20)
    lab = _labels(rng, 16, 20, 9)
    state, stats = sit.RegionConnectivity(np.array(cells), np.array(masks), lab, 0.5, tau_edges=EDGES)
    rs, rw = O.run(cells, masks, lab, 9, EDGES)
    for i, n in enumerate(("status", "src", "prev", "start", "visited")):
        assert np.array_equal(state[n], rs[-1][:, i]), n
    assert len(stats) == 12
    for a, b in zip(stats, rw):
        _same(a, b)
        assert a["sample_days"] == 0.5 and a["nreg"] == 9


@pytest.mark.gpu
def test_connect_entry_point_refusals(torch, sit, gold_track):
    """st_connect_dev on real, aligned buffers refuses t outside 0..65535, shapes past the limits, NULL pointers, a
    context's cell state that does not match and misaligned cells, state, edges or stats; it writes nothing then."""
    from sitrack_b200 import _lib
    from sitrack_b200 import connect as K
    L = _lib.lib()
    T, g = gold_track
    dev = torch.device("cuda", 0)
    eng = engine_for(g, device=0)
    eng.set_buoys(T["pos0"], T["jiT0"].astype(np.int32))
    Nj, Ni, nP = eng.Nj, eng.Ni, eng.nP
    lab = np.ascontiguousarray(_gold_maps(g)["i"][0], np.uint8)
    plan = K._Plan(torch, dev, lab, 7, Nj, Ni, nP)
    (st,) = plan.outputs()
    big = torch.zeros((plan.nstat + 1,), dtype=torch.int64, device=dev)
    cell = torch.from_numpy(np.ascontiguousarray(T["jiT0"], np.int32)).to(dev)
    cbig = torch.zeros((2 * nP + 2,), dtype=torch.int32, device=dev)
    mk = torch.ones((nP,), dtype=torch.int8, device=dev)

    def call(ctx=True, Nj_=Nj, Ni_=Ni, labels=None, R=7, n=nP, cell_p=None, m=True, t=0, state=None, ntau=17,
             tau=None, stats=None):
        st.fill_(-3)
        plan.state.fill_(-7)
        torch.cuda.synchronize()
        rc = L.st_connect_dev(eng.h if ctx else None, Nj_, Ni_, plan.labels_t.data_ptr() if labels is None else labels,
                              R, n, cell_p, mk.data_ptr() if m else None, t,
                              plan.state.data_ptr() if state is None else state, ntau,
                              plan.tau_edges_t.data_ptr() if tau is None else tau,
                              st.data_ptr() if stats is None else stats, None)
        torch.cuda.synchronize()
        return rc

    assert call() == 0 and int((st[:8] + 3).sum()) > 50 and (plan.state.cpu().numpy() != -7).all()
    assert call(cell_p=cell.data_ptr(), ctx=False, t=65535) == 0
    assert call(cell_p=cell.data_ptr(), Nj_=Nj + 3) == 0
    for kw in (dict(t=-1), dict(t=65536), dict(R=0), dict(R=32), dict(ntau=0), dict(ntau=513), dict(n=0),
               dict(n=2 ** 31), dict(Nj_=0), dict(Ni_=0), dict(Nj_=2 ** 16, Ni_=2 ** 15, cell_p=cell.data_ptr()),
               dict(labels=0), dict(m=False), dict(state=0), dict(tau=0), dict(stats=0), dict(ctx=False),
               dict(n=nP - 1), dict(Nj_=Nj + 1), dict(Ni_=Ni - 1), dict(cell_p=cbig.data_ptr() + 4),
               dict(state=plan.state.data_ptr() + 4), dict(tau=plan.tau_edges_t.data_ptr() + 4),
               dict(stats=big.data_ptr() + 4)):
        assert call(**kw) == -1, kw
        assert (st.cpu().numpy() == -3).all() and (plan.state.cpu().numpy() == -7).all(), kw
    eng.close()


def _engine(T, g, name, sort, rows, connect=None, sink=None, physics=None, **other):
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
                    row_dtype=rows, sink=sink, physics=physics, connect=connect, **other)
    eng.close()
    return res


@pytest.mark.gpu
@pytest.mark.parametrize("every", [1, 48, 49])
@pytest.mark.parametrize("rows", ["f8", "f4"])
@pytest.mark.parametrize("name", ["uv1", "win"])
def test_track_connect(torch, sit, gold_track, name, rows, every):
    """track(connect=...): every window's statistics equal the oracle run over the stepped cells (row 0 masked by
    rec_first on the `win` case), whether the buoys are stored in the caller's order or sorted on the host or the
    device, with the rows kept or sent to a sink; every = 49 > 48 records gives no window."""
    O = _ref()
    T, g = gold_track
    cells, _, masks = _stepped(T, g, name)
    lab, R = _gold_maps(g)["i"]
    _, ref = O.run(cells, masks, lab, R, EDGES, every)
    spec = dict(labels=lab, every=every, tau_edges=EDGES)
    for sort in ("none", "host", "dev"):
        got = _engine(T, g, name, sort, rows, spec)["connect"]
        assert len(got) == len(ref) == 48 // every
        for st, rf in zip(got, ref):
            _same(st, rf)
            assert st["sample_days"] == every * 3600.0 / 86400.0 and st["nreg"] == R
    seen = []
    res = _engine(T, g, name, "host", rows, dict(spec, sink=lambda w, st: seen.append((w, st))), sink=lambda *a: None)
    assert "connect" not in res and [w for w, _ in seen] == list(range(len(ref)))
    for (_, st), rf in zip(seen, ref):
        _same(st, rf)
    if every == 1:
        assert _total(ref)["n_arrive"].sum() > 20


@pytest.mark.gpu
def test_track_connect_physics(torch, sit, gold_track):
    """With physics (RK4, C-grid linear, 3 hops) on the `fast` case, kept and sunk, against the cells stepped with
    st_step_ext."""
    O = _ref()
    T, g = gold_track
    phys = dict(scheme=4, interp=1, max_hops=3)
    cells, _, masks = _stepped(T, g, "fast", physics=phys)
    lab, R = _gold_maps(g)["j"]
    _, ref = O.run(cells, masks, lab, R, EDGES, 3)
    res = _engine(T, g, "fast", "host", "f8", dict(labels=lab, every=3, tau_edges=EDGES), physics=phys)
    for st, rf in zip(res["connect"], ref):
        _same(st, rf)
    assert len(res["connect"]) == 16 and _total(ref)["n_arrive"].sum() > 20


@pytest.mark.gpu
def test_track_connect_with_every_other_analysis(torch, sit, gold_track):
    """connect together with deform, dispersion, fsle and sample: their outputs and the rows are those of the same
    call without connect, bit for bit, and the connect statistics those of the call without them; refusals before
    anything runs."""
    T, g = gold_track
    sh = np.random.default_rng(7).permutation(T["pos0"].shape[0])
    pos0 = T["pos0"][sh]
    tri = sit.TriangulateCloud(pos0)
    pairs = np.concatenate([sit.MeshPairs(tri), sit.SeparationPairs(pos0, 1.0, 30.0, 500)])
    lab, R = _gold_maps(g)["j"]
    others = dict(deform=dict(tri=tri, every=4), dispersion=dict(pairs=pairs, every=6, lags=4),
                  fsle=dict(pairs=pairs, every=2), sample=dict(names=["siconc"], every=3))
    con = dict(labels=lab, every=2)
    for rows in ("f8", "f4"):
        both = _engine(T, g, "uv1", "host", rows, con, **others)
        plain = _engine(T, g, "uv1", "host", rows, None, **others)
        alone = _engine(T, g, "uv1", "host", rows, con)
        assert "connect" not in plain and len(both["connect"]) == 24
        for k in ("posC", "posG", "mask", "n_alive"):
            assert np.ascontiguousarray(both[k]).tobytes() == np.ascontiguousarray(plain[k]).tobytes(), k
        for key in ("deform", "dispersion", "fsle"):
            for a, b in zip(both[key], plain[key]):
                for k in a:
                    if isinstance(a[k], np.ndarray):
                        assert np.ascontiguousarray(a[k]).tobytes() == np.ascontiguousarray(b[k]).tobytes(), (key, k)
        assert both["sample"]["siconc"].tobytes() == plain["sample"]["siconc"].tobytes()
        for a, b in zip(both["connect"], alone["connect"]):
            _same(a, b)
    eng = engine_for(g, device=0)
    eng.set_buoys(pos0, T["jiT0"][sh].astype(np.int32))
    rec = (T["U"], T["V"], T["IC"])
    with pytest.raises(ValueError, match="streaming record loop"):
        eng.track(rec, 48, chunk=8, connect=con)
    for bad in (dict(con, labels=lab[:, :-1]), dict(con, labels=lab * 0), dict(con, every=0),
                dict(con, tau_edges=[2.0, 1.0])):
        with pytest.raises(ValueError):
            eng.track(rec, 48, sink=lambda *a: None, connect=bad)
    from sitrack_b200 import fsle as F
    F_max = F.MAX_SAMPLES
    try:
        F.MAX_SAMPLES = 23                                             # 24 windows: refused before anything runs
        with pytest.raises(ValueError, match="windows"):
            eng.track(rec, 48, sink=lambda *a: None, connect=con)
    finally:
        F.MAX_SAMPLES = F_max
    eng.close()


def _two_d_time(r):
    """Give the seed file of a synthetic case per-buoy record windows (time_pos) for a run without -F, keeping only the
    seeds SeedInit keeps, as test_cli does."""
    import sitrack_b200 as sit
    from synth.records import T0_EPOCH
    z = dict(np.load(r["seed"]))
    kmaskt, latT, lonT, _, _, Yf, Xf, ResKM = quiet(sit.GetModelGrid, r["mesh"])
    _, zid, XG, XC = quiet(sit.LoadNCdata, r["seed"], krec=0)
    ok = quiet(sit.SeedInit, zid, XG, XC, latT, lonT, Yf, Xf, ResKM, kmaskt,
               xIceConc=np.asarray(r["records"][2][2], np.float64))[6]
    z["id_buoy"] = z["id_buoy"][ok]
    for k in ("latitude", "longitude", "y_pos", "x_pos"):
        z[k] = z[k][:, ok]
    nP = z["id_buoy"].size
    rng = np.random.default_rng(5)
    tm = T0_EPOCH + 1800 + 3600 * np.arange(r["records"][0].shape[0])
    first = rng.integers(2, 7, nP); first[0] = 2
    last = rng.integers(14, 21, nP); last[1] = 20
    tpos = np.stack([tm[first] - 1799, tm[last]]).astype("i4")
    z["time"] = np.array([tpos[0].min(), tpos[1].max()], "i4")
    for k in ("latitude", "longitude", "y_pos", "x_pos"):
        z[k] = np.concatenate([z[k], z[k]], axis=0)
    z["time_pos"] = tpos
    os.remove(r["seed"])
    np.savez(r["seed"], **z)


def _synth_regions(r, tmp_path):
    nj, ni = r["records"][0].shape[1:]
    jj, ii = np.meshgrid(np.arange(nj), np.arange(ni), indexing="ij")
    lab = (1 + (ii // 6) % 9 + 9 * ((jj // 10) % 2)).astype(np.float32)
    lab[:, : ni // 5] = 0
    fn = str(tmp_path / "regions.npz")
    np.savez(fn, reg=lab[None])
    return fn, lab


@pytest.mark.gpu
@pytest.mark.parametrize("extra", [["-F"], ["-F", "--sort"], []])
def test_cli_connect_end_to_end(tmp_path, monkeypatch, extra):
    """si3_part_tracker.py --connect 2 --connect-regions on the 'small' synthetic case, with and without -F and after
    --sort: the file holds the engine API's statistics on the same inputs and the tracking files are byte-identical to
    a run without the flags."""
    import si3_part_tracker as cli
    import sitrack_b200 as sit
    from make_synth_case import write_case
    r = write_case(str(tmp_path / "in"), grid="small", nrec=24, hss=3)
    if "-F" not in extra:
        _two_d_time(r)
    reg, lab = _synth_regions(r, tmp_path)
    argv = ["si3_part_tracker.py", "-i", r["si3"], "-m", r["mesh"], "-s", r["seed"], "-N", "SYNTH4"] + extra
    runs = {}
    for tag, more in (("plain", []), ("connect", ["--connect", "2", "--connect-regions", reg, "reg"])):
        d = tmp_path / tag
        d.mkdir()
        monkeypatch.chdir(d)
        monkeypatch.setattr(sys, "argv", argv + more)
        quiet(cli.main)
        runs[tag] = d
    files = sorted(os.listdir(runs["plain"] / "nc"))
    cfiles = [f for f in os.listdir(runs["connect"] / "nc") if "_connectivity_" in f]
    assert len(cfiles) == 1 and sorted(set(os.listdir(runs["connect"] / "nc")) - set(cfiles)) == files
    for f in files:
        a, b = np.load(runs["plain"] / "nc" / f), np.load(runs["connect"] / "nc" / f)
        assert sorted(a.files) == sorted(b.files)
        for k in a.files:
            assert a[k].dtype == b[k].dtype and a[k].tobytes() == b[k].tobytes(), (f, k)
    z = np.load(runs["connect"] / "nc" / cfiles[0])
    nw = z["time_start"].shape[0]
    assert nw >= 8 and z["count"].shape == (nw, 19, 19) and z["hist_tau"].shape == (nw, 19, 18, 18)
    assert float(z["sample_days"]) == 2 * 3600.0 / 86400.0
    cache = np.load(runs["connect"] / "seed" / os.listdir(runs["connect"] / "seed")[0])
    imaskt, _, _, _, _, Yf, Xf, _ = quiet(sit.GetModelGrid, r["mesh"])
    Yv, Xv, Yu, Xu = quiet(sit.GetModelUVGrid, r["mesh"])
    U, V, IC = r["records"]
    seen = []
    with sit.TrackEngine(Yf, Xf, Yu, Xu, Yv, Xv, tmask=imaskt, uv_strategy=1, rdt=3600.0, rmin_conc=sit.rmin_conc,
                         device=0) as eng:
        eng.set_buoys(cache["xPosC0"], cache["vJIt"])
        eng.track((U[:24], V[:24], IC[:24]), 24, sink=lambda *a: None, row_dtype="f4",
                  connect=dict(labels=lab, every=2, sink=lambda w, st: seen.append(st)))
    if "-F" in extra:                                                       # no per-buoy windows: the same buoys
        assert len(seen) == 12 == nw
        for w, st in enumerate(seen):
            for k in NAMES:
                assert np.array_equal(z[k][w], st[k]), (w, k)
    assert z["n_start"].sum() > 100 and z["trans"].sum() > 500


@pytest.mark.gpu
@pytest.mark.timeout(300)
def test_cli_connect_under_torchrun(tmp_path):
    """`torchrun --nproc-per-node 2` (both ranks on cuda:0): each rank counts its block of buoys, the windows are summed
    on rank 0, and the _connectivity_ file equals the single-process run's, variable by variable."""
    from make_synth_case import write_case
    r = write_case(str(tmp_path / "in"), grid="small", nrec=12, hss=2)
    reg, _ = _synth_regions(r, tmp_path)
    cli = os.path.join(ROOT, "si3_part_tracker.py")
    common = ["-i", r["si3"], "-m", r["mesh"], "-s", r["seed"], "-F", "-N", "SYNTH4", "--device", "0",
              "--connect", "2", "--connect-regions", reg, "reg"]
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
    f = [f for f in files if "_connectivity_" in f][0]
    a, b = np.load(one / "nc" / f), np.load(two / "nc" / f)
    assert sorted(a.files) == sorted(b.files)
    for k in a.files:
        assert a[k].tobytes() == b[k].tobytes(), k
    assert a["n_start"].sum() > 256 and a["trans"].sum() > 1000


@pytest.mark.gpu
def test_bench_connect_small():
    """tools/bench_connect.py end to end on the small synthetic grid: exit 0, both maps equal to the oracle."""
    import json
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_connect.py"), "--grid", "small", "--buoys",
                        "50000", "--seconds", "0.05"], stdout=subprocess.PIPE, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    assert res["oracle_check_passed"] and res["step_us"] > 0 and set(res["connect"]) == {"blocks_31", "one_region"}
    for c in res["connect"].values():
        assert c["started"] > 40000 and c["ended"] > 100 and c["state_writes"] >= c["ended"]
