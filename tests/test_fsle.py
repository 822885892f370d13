"""Finite-size Lyapunov exponents of buoy pairs: per-pair first-passage state and exit times between separation
thresholds (sitrack_b200.fsle, csrc/st_fsle.cu).

CPU: the oracle (oracle/fsle_ref.py) on closed forms, the vectorised oracle against its per-pair loop, the argument
checks of st_fsle_state_bytes and of the thresholds, both writer branches and the CLI's argument errors.  GPU: the
per-pair state after every sample and every window's statistics equal the oracle's exactly, on the golden rows, a
200 k-buoy lattice, small and grid-saturating pair counts and the shape limits; two runs give the same bits;
FiniteSizeLyapunov; the entry point's refusals; TrackEngine.track(fsle=...) in every buoy storage order and row dtype,
with and next to deform and dispersion; the CLI end to end and a small run of the benchmark."""
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
POW2 = 2.0 ** np.arange(16)                                   # 1 ... 32768 km
GOLD_DELTAS = 20.0 * 2.0 ** (np.arange(64) / 32.0)            # 20 ... 79 km: the golden buoys' separations grow by a few %


def _ref():
    from oracle import fsle_ref as O
    return O


def _same(a, b):
    assert set(a) >= {"n_start", "hist_tau", "n", "sum_tau", "sum_tau2", "n_censored"}
    for k in ("n_start", "hist_tau", "n", "sum_tau", "sum_tau2", "n_censored"):
        assert np.asarray(a[k]).dtype == np.int64 and np.array_equal(a[k], b[k]), k


def _one_pair(seps, masks=None, deltas=(1.0, 2.0, 4.0, 8.0, 16.0), tau_edges=(1.0, 2.0, 4.0)):
    """One pair along the x axis at separations `seps` (one per sample): -> (states (S, 1, 2), windows) of the oracle,
    checked against the per-pair loop."""
    O = _ref()
    rows = [np.array([[0.0, 0.0], [0.0, s]]) for s in seps]
    masks = [np.ones(2, np.int8)] * len(seps) if masks is None else [np.array([m, 1], np.int8) for m in masks]
    st, w = O.run(rows, masks, [[0, 1]], deltas, tau_edges)
    st2, w2 = O.run(rows, masks, [[0, 1]], deltas, tau_edges, step=O.sample_loop)
    assert np.array_equal(st, st2)
    for a, b in zip(w, w2):
        _same(a, b)
    return st, w


def _total(wins):
    return {k: sum(w[k] for w in wins) for k in wins[0]}


# ---- CPU: the oracle ---------------------------------------------------------------------------

@pytest.mark.parametrize("m", [1, 3, 4])
def test_oracle_doubling_every_m_samples(m):
    """Separations that double exactly every m samples (Pythagorean and power-of-two offsets scaled by 2^(s//m)) on
    deltas = 2^j: every timed exit time is m, no zero, and fsle_lambda = ln 2 / (m sample_days) exactly."""
    import sitrack_b200 as sit
    O = _ref()
    off = np.array([[3, 4], [4, 3], [5, 12], [0, 4], [8, 6], [-20, 21], [0, 1], [7, 24], [-2, 0]], np.float64)
    base = np.stack([np.arange(off.shape[0]) * 3000.0, np.arange(off.shape[0]) * -700.0], 1)
    pairs = np.stack([np.arange(off.shape[0]), off.shape[0] + np.arange(off.shape[0])], 1)
    S = 8 * m
    rows = [np.concatenate([base, base + off * 2.0 ** (s // m)]) for s in range(S + 1)]
    masks = [np.ones(2 * off.shape[0], np.int8)] * (S + 1)
    tau_edges = O.DEFAULT_TAU_EDGES
    _, wins = O.run(rows, masks, pairs, POW2, tau_edges)
    _, wins2 = O.run(rows, masks, pairs, POW2, tau_edges, step=O.sample_loop)
    for a, b in zip(wins, wins2):
        _same(a, b)
    tot = _total(wins)
    n = tot["n"]
    assert n.sum() == off.shape[0] * 7                                  # 8 doublings, the first one untimed
    assert (tot["sum_tau"] == m * n).all() and (tot["sum_tau2"] == m * m * n).all()
    kb = np.searchsorted(tau_edges, m, side="right")
    assert tot["hist_tau"][:, kb].sum() == n.sum() and tot["hist_tau"][:, 0].sum() == 0
    assert tot["n_start"].sum() == off.shape[0] and tot["n_censored"].sum() == 0
    sd = 0.125
    lam = sit.fsle_lambda([dict(w, deltas_km=POW2, sample_days=sd) for w in wins])
    assert np.array_equal(lam[n > 0], np.full((n > 0).sum(), np.log(2.0) / (m * sd)))
    assert np.isnan(lam[n == 0]).all()


def test_oracle_jump_over_three_thresholds():
    """0.5 -> 1.5 (level 1 at t = 1) -> 9 at t = 3: one timed tau = 2 for transition 0 and tau = 0 for 1 and 2."""
    st, w = _one_pair([0.5, 1.5, 1.7, 9.0])
    tot = _total(w)
    assert tot["n"].tolist() == [1, 1, 1, 0] and tot["sum_tau"].tolist() == [2, 0, 0, 0]
    assert tot["hist_tau"][0].tolist() == [0, 0, 1, 0] and tot["hist_tau"][1:3, 0].tolist() == [1, 1]
    assert st[-1, 0].tolist() == [4, 3] and tot["n_start"].tolist() == [1, 0, 0, 0, 0, 0]
    assert w[0]["n_start"][0] == 1 and w[2]["n"].sum() == 3                # events land in their window


def test_oracle_start_above_a_threshold_is_not_timed():
    """Starting at 5 (level 3, above delta_2 = 4): 9 is reached untimed, then 17 is timed (tau = 3)."""
    st, w = _one_pair([5.0, 6.0, 9.0, 10.0, 12.0, 17.0])
    tot = _total(w)
    assert tot["n_start"].tolist() == [0, 0, 0, 1, 0, 0] and tot["n"].tolist() == [0, 0, 0, 1]
    assert tot["sum_tau"][3] == 3 and st[1, 0].tolist() == [4, 2] and st[-1, 0].tolist() == [5, 5]


def test_oracle_tie_reaches_and_decrease_holds():
    """r exactly on a threshold reaches it; a decreasing r keeps the level and records nothing."""
    st, w = _one_pair([1.0, 4.0, 3.0, 0.5, 8.0])
    assert st[0, 0].tolist() == [3, 1] and st[1, 0].tolist() == [3, 1] and st[2, 0].tolist() == [3, 1]
    tot = _total(w)
    assert tot["n"].tolist() == [0, 1, 1, 0] and tot["sum_tau"][2] == 3      # 4 -> 8 timed: t 4 - 1
    assert w[1]["n"].sum() == 0 and w[2]["n"].sum() == 0


def test_oracle_deaths_censor_only_anchored_pairs():
    O = _ref()
    # anchored (level 3 reached at t = 1), dies at t = 2: transition 2 censored
    st, w = _one_pair([1.5, 4.0, 4.5, 9.0], masks=[1, 1, 0, 1])
    assert _total(w)["n_censored"].tolist() == [0, 0, 1, 0] and st[1, 0].tolist() == [-2, 1]
    assert st[2, 0].tolist() == [-2, 1]                                    # an ended pair stays ended
    # no anchor (started at level 3, never rose): not censored
    st, w = _one_pair([4.5, 5.0, 5.0], masks=[1, 1, 0])
    assert _total(w)["n_censored"].sum() == 0 and st[-1, 0].tolist() == [-2, -1]
    # anchored at the last level K: nothing left to censor
    st, w = _one_pair([9.0, 17.0, 17.0], masks=[1, 1, 0])
    assert _total(w)["n_censored"].sum() == 0 and st[0, 0].tolist() == [5, 1]
    # a non-finite separation on valid masks ends a started pair like a death
    for bad in (np.nan, np.inf, -np.inf):
        st, w = _one_pair([1.5, 4.0, bad])
        assert st[-1, 0, 0] == -2 and _total(w)["n_censored"].tolist() == [0, 0, 1, 0]
    assert O.DEFAULT_DELTAS.size == 19 and O.DEFAULT_DELTAS[0] == 2.0 and O.DEFAULT_DELTAS[-1] == 1024.0


def test_oracle_late_start_and_nonfinite_delay():
    """A pair masked at row 0 (rec_first later than the run's start) starts at its first valid sample; NaN, +inf or
    -inf coordinates on valid masks delay a pair that has not started and are never binned."""
    st, w = _one_pair([3.0, 3.0, 5.0, 9.0], masks=[0, 0, 1, 1])
    assert st[0, 0].tolist() == [-1, -1] and st[1, 0].tolist() == [3, -1] and w[1]["n_start"][3] == 1
    for bad in (np.nan, np.inf, -np.inf):
        st, w = _one_pair([bad, bad, 3.0, 5.0])
        assert st[0, 0].tolist() == [-1, -1] and st[1, 0].tolist() == [2, -1] and st[2, 0].tolist() == [3, 3]
        assert _total(w)["n_start"].sum() == 1 and _total(w)["n"].sum() == 0


def _walk(rng, nP=400, S=30, spread=1.5, dmask=0.01, nonfinite=True):
    rows = [rng.uniform(0, 60.0, (nP, 2))]
    for s in range(S):
        rows.append(rows[-1] * 1.02 + rng.normal(0, spread, (nP, 2)))
    rows = [r.copy() for r in rows]
    masks = [(rng.random(nP) > 0.1).astype(np.int8)]
    for s in range(S):
        masks.append((masks[-1] | (rng.random(nP) < 0.2)) & (rng.random(nP) > dmask))
    masks = [m.astype(np.int8) for m in masks]
    if nonfinite:
        for s in (3, 9, 17)[:S // 6]:
            k = rng.choice(nP, 4, replace=False)
            rows[s][k[0], 0], rows[s][k[1], 1], rows[s][k[2], 0], rows[s][k[3], 1] = np.nan, np.inf, -np.inf, 1e300
    return rows, masks


def test_oracle_vectorised_equals_loop_on_random_walks():
    O = _ref()
    rng = np.random.default_rng(5)
    rows, masks = _walk(rng)
    a = rng.integers(0, 400, 3000)
    pairs = np.stack([a, (a + 1 + rng.integers(0, 399, 3000)) % 400], 1)
    deltas = 2.0 ** (np.arange(24) / 3.0)
    for every in (4, 1):
        s1, w1 = O.run(rows, masks, pairs, deltas, [1.0, 2.0, 3.0, 5.0, 8.0], every=every)
        s2, w2 = O.run(rows, masks, pairs, deltas, [1.0, 2.0, 3.0, 5.0, 8.0], every=every, step=O.sample_loop)
        assert np.array_equal(s1, s2)
        for x, y in zip(w1, w2):
            _same(x, y)
    tot = _total(w1)
    assert tot["n"].sum() > 500 and tot["n_censored"].sum() > 20 and tot["hist_tau"][:, 0].sum() > 10


def test_threshold_checks_and_lambda_edges():
    import sitrack_b200 as sit
    from sitrack_b200 import fsle as F
    for bad in ([1.0], [1.0, 1.0], [2.0, 1.0], [0.0, 1.0], [-1.0, 1.0], [1.0, np.inf], [np.nan, 1.0],
                np.arange(1.0, 66.0)):
        with pytest.raises(ValueError):
            F.check_deltas(bad)
    assert np.array_equal(F.check_deltas(None), F.DEFAULT_DELTAS) and F.check_deltas(np.arange(1.0, 65.0)).size == 64
    assert np.array_equal(F.DEFAULT_DELTAS, 2.0 ** (1 + np.arange(19) / 2))
    assert F.DEFAULT_TAU_EDGES.tolist() == [2.0 ** k for k in range(17)]
    d = np.array([1.0, 2.0, 4.0, 8.0])
    st = dict(deltas_km=d, sample_days=0.5, n=np.array([0, 3, 2]), sum_tau=np.array([0, 0, 4]))
    lam = sit.fsle_lambda([st, st])
    assert np.isnan(lam[0]) and lam[1] == np.inf and lam[2] == np.log(2.0) / (0.5 * 2.0)


@pytest.mark.parametrize("case", [dict(nQ=0), dict(nQ=2 ** 31), dict(K=1), dict(K=65), dict(ntau=0), dict(ntau=513),
                                  dict(out=None)])
def test_fsle_state_bytes_rejects(case):
    """st_fsle_state_bytes returns ST_EINVAL (-1) for each bad argument, one past each limit, before any CUDA call,
    and leaves the output alone."""
    from sitrack_b200 import _lib
    a = dict(nQ=1000, K=19, ntau=17, out=True)
    a.update(case)
    out = C.c_int64(-5)
    rc = _lib.lib().st_fsle_state_bytes(a["nQ"], a["K"], a["ntau"], C.byref(out) if a["out"] else None)
    assert rc == -1 and out.value == -5
    assert b"st_fsle_state_bytes" in _lib.lib().st_last_error(None)


def test_fsle_state_bytes_accepts():
    """Each limit exactly; the largest shape (64 thresholds, 512 exit-time edges) needs 135 404 B of shared memory,
    inside the 227 KB a block may have."""
    from sitrack_b200 import _lib
    out = C.c_int64(0)
    for nQ, K, ntau in ((1, 2, 1), (2 ** 31 - 1, 64, 512), (1000, 19, 17)):
        assert _lib.lib().st_fsle_state_bytes(nQ, K, ntau, C.byref(out)) == 0
        assert out.value == 8 * nQ
    J = 63
    assert (64 + 512 + 2 * J) * 8 + (65 + J * 513 + J) * 4 == 135404 < 227 * 1024


def _writer_stats(jw, K, NB):
    return dict(n_start=np.full(K + 1, jw), hist_tau=np.full((K - 1, NB), jw + 2), n=np.full(K - 1, jw + 1),
                sum_tau=np.full(K - 1, 7 * jw), sum_tau2=np.full(K - 1, 2 ** 40 + jw), n_censored=np.full(K - 1, 3))


def test_fsle_writer_npz(tmp_path):
    import sitrack_b200 as sit
    d, te = np.array([2.0, 4.0, 8.0, 16.0]), np.array([1.0, 2.0, 4.0])
    f = str(tmp_path / "f.npz")
    with quiet(sit.FsleWriter, f, 2, d, te, 0.25, corigin="X") as w:
        for jw in range(2):
            w.write(jw, 100 + jw, 200 + jw, _writer_stats(jw, 4, 4))
    z = np.load(f)
    assert z["time_start"].tolist() == [100, 101] and z["time_end"].dtype == np.int32
    assert np.array_equal(z["delta_km"], d) and np.array_equal(z["tau_edges"], te) and float(z["sample_days"]) == 0.25
    assert z["n_start"].shape == (2, 5) and z["hist_tau"].shape == (2, 3, 4) and z["n"].shape == (2, 3)
    for k in ("n_start", "n", "sum_tau", "sum_tau2", "n_censored", "hist_tau"):
        assert z[k].dtype == np.int64, k
    assert (z["sum_tau2"][1] == 2 ** 40 + 1).all() and (z["hist_tau"][1] == 3).all() and (z["n_start"][1] == 1).all()
    units = dict(delta_km="km", tau_edges="sample", n_start="1", n="1", sum_tau="sample", sum_tau2="sample2",
                 n_censored="1", hist_tau="1")
    for k, u in units.items():
        assert str(z[k + "_units"]) == u, k
    assert "FillValue" not in z.files


def test_fsle_writer_netcdf_branch(monkeypatch, tmp_path):
    """The netCDF4 branch against the in-memory stand-in of test_cli: dimensions, variables, no fill values, units,
    the sample_days attribute."""
    import types
    import sitrack_b200 as sit
    from test_cli import _FakeNC
    fake = types.ModuleType("netCDF4"); fake.Dataset = _FakeNC.Dataset
    monkeypatch.setitem(sys.modules, "netCDF4", fake)
    f = str(tmp_path / "f.nc")
    with quiet(sit.FsleWriter, f, 3, [2.0, 4.0, 8.0], [1.0, 2.0], 0.5, corigin="ORG") as w:
        for jw in range(3):
            w.write(jw, jw, jw + 1, _writer_stats(jw, 3, 3))
    ds = _FakeNC.files[f]
    assert ds._dims == {"time": None, "threshold": 3, "transition": 2, "tau_bin": 3, "level": 4, "tau_edge": 2}
    assert ds.attrs["Origin"] == "ORG" and ds.attrs["sample_days"] == 0.5
    v = ds.variables["hist_tau"]
    assert v.a.shape == (3, 2, 3) and v.a.dtype == np.int64 and v.fill is None and (v.a[2] == 4).all()
    assert ds.variables["sum_tau"].fill is None and ds.variables["sum_tau"].units == "sample"
    assert ds.variables["n_start"].a.tolist()[2] == [2] * 4 and ds.variables["delta_km"].a.tolist() == [2.0, 4.0, 8.0]
    assert ds.variables["time_end"].a.tolist() == [1, 2, 3]


@pytest.mark.parametrize("extra,env", [(["--fsle", "0"], {}), (["--fsle", "1.5"], {}),
                                       (["--fsle", "6", "--fsle-deltas", "2", "1.4142", "1"], {}),
                                       (["--fsle", "6", "--fsle-deltas", "2", "1.4142", "65"], {}),
                                       (["--fsle", "6", "--fsle-deltas", "2", "1.4142", "2.5"], {}),
                                       (["--fsle", "6", "--fsle-deltas", "0", "1.4142", "19"], {}),
                                       (["--fsle", "6", "--fsle-deltas", "2", "1", "19"], {}),
                                       (["--fsle", "6", "--fsle-deltas", "1e300", "1e10", "64"], {}),
                                       (["--fsle", "6", "--fsle-pairs", "0", "10", "100"], {}),
                                       (["--fsle", "6", "--fsle-pairs", "10", "0", "100"], {}),
                                       (["--fsle", "6", "--fsle-pairs", "10", "50", "50"], {}),
                                       (["--fsle-pairs", "10", "10", "100"], {}),
                                       (["--fsle-deltas", "2", "2", "10"], {}),
                                       (["--fsle", "6"], {"WORLD_SIZE": "2"})])
def test_cli_fsle_argument_errors(tmp_path, monkeypatch, extra, env):
    """Each bad --fsle / --fsle-deltas / --fsle-pairs argument is an ERROR line printed before anything is read or
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
    assert any(l.startswith("ERROR") and "--fsle" in l for l in buf.getvalue().splitlines())
    assert not os.listdir(tmp_path)


@pytest.mark.parametrize("hours", ["12", "1"])
def test_cli_fsle_window_count(tmp_path, monkeypatch, hours):
    """A run shorter than one window, and (with MAX_SAMPLES lowered to 5) more windows than a run may have, are
    ERROR lines printed before anything is written."""
    import si3_part_tracker as cli
    import sitrack_b200 as sit
    from make_synth_case import write_case
    r = write_case(str(tmp_path / "in"), grid="tiny", nrec=6, hss=3)
    d = tmp_path / "run"
    d.mkdir()
    monkeypatch.chdir(d)
    if hours == "1":
        monkeypatch.setattr(sit, "MAX_SAMPLES", 5)                   # 6 windows of one record
    monkeypatch.setattr(sys, "argv", _synth_argv(r, "--fsle", hours))
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf), pytest.raises(SystemExit):
        cli.main()
    assert any(l.startswith("ERROR") and "--fsle" in l for l in buf.getvalue().splitlines()), buf.getvalue()[-500:]
    assert not os.listdir(d)


# ---- GPU ---------------------------------------------------------------------------------------

def _device_run(torch, rows, masks, pairs, deltas=None, tau_edges=None, every=1):
    """One st_fsle_dev per sample through fsle._Plan, as the engine drives it: -> (states (S, nQ, 2) after each
    window, the windows' stats)."""
    from sitrack_b200 import fsle as F
    dev = torch.device("cuda", 0)
    g = lambda a, d: torch.from_numpy(np.ascontiguousarray(a, d)).to(dev)
    plan = F._Plan(torch, dev, pairs, deltas, tau_edges, 0.25)
    s = torch.cuda.current_stream(dev)
    origin = [(g(rows[0], np.float64), g(masks[0], np.int8), 1)]
    states, wins = [], []
    for w in range((len(rows) - 1) // every):
        k = (w + 1) * every
        o = plan.outputs()
        plan.window(None, origin, g(rows[k], np.float64), g(masks[k], np.int8), 0.25, o, s)
        states.append(plan.state.cpu().numpy())
        wins.append(plan.results((o[0].cpu(),))[0])
    return np.array(states), wins, plan


def _vs_oracle(torch, rows, masks, pairs, deltas=None, tau_edges=None, every=1, again=False):
    O = _ref()
    kw = {}
    if deltas is not None:
        kw["deltas"] = deltas
    if tau_edges is not None:
        kw["tau_edges"] = tau_edges
    st, wins, plan = _device_run(torch, rows, masks, pairs, deltas, tau_edges, every)
    rs, rw = O.run(rows, masks, pairs, every=every, **kw)
    assert st.shape == rs.shape and np.array_equal(st, rs)
    assert len(wins) == len(rw)
    for a, b in zip(wins, rw):
        _same(a, b)
    if again:
        st2, wins2, _ = _device_run(torch, rows, masks, pairs, deltas, tau_edges, every)
        assert np.array_equal(st2, st)
        for a, b in zip(wins2, wins):
            _same(a, b)
    return _total(wins), plan


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TRACK_CASES))
def test_fsle_vs_oracle_golden(torch, gold_track, name):
    """Every ordered pair of the 94 golden buoys over every row of each golden case: state after each sample and
    each window's statistics equal the oracle's."""
    T, _ = gold_track
    posC, mask = T[name + "_posC"], T[name + "_mask"]
    n = posC.shape[1]
    a, b = np.triu_indices(n, 1)
    pairs = np.concatenate([np.stack([a, b], 1), np.stack([b, a], 1)]).astype(np.int32)
    tot, _ = _vs_oracle(torch, list(posC), list(mask), pairs, GOLD_DELTAS, [1.0, 2.0, 3.0, 6.0, 12.0, 24.0],
                        again=True)
    assert tot["n"].sum() > 200 and tot["n_start"].sum() > 5000 and tot["n_censored"].sum() > 50


def _lattice_rows(rng, n=450, S=6):
    yx0, tri = _lattice(n, hole=(600.0, 700.0, 90.0), seed=3)
    nP = yx0.shape[0]
    rows, masks = [yx0], [(rng.random(nP) >= 0.02).astype(np.int8)]
    for s in range(S):
        y = rows[-1]
        rows.append(y * 1.01 + 1.2 + np.stack([np.sin(y[:, 1] / 40.0 + s), np.cos(y[:, 0] / 55.0 - s)], 1) * 0.7
                    + rng.normal(0.0, 0.3, y.shape))
        jump = rng.choice(nP, 300, replace=False)
        rows[-1][jump] += rng.choice([-1.0, 1.0], (300, 2)) * 7.0
        masks.append(masks[-1] * (rng.random(nP) >= 0.01).astype(np.int8))
    masks[2][rng.choice(nP, 500, replace=False)] = 1                    # late starts
    return rows, masks, tri


@pytest.mark.gpu
def test_fsle_vs_oracle_lattice(torch, sit):
    """~200 k buoys with masks, deaths and late starts, mesh pairs and sampled pairs (10 to 1000 km), every = 1 and 2."""
    rng = np.random.default_rng(11)
    rows, masks, tri = _lattice_rows(rng)
    pairs = np.concatenate([sit.MeshPairs(tri), sit.SeparationPairs(rows[0], 10.0, 1000.0, 200000, seed=5)])
    deltas = 2.0 ** (np.arange(64) / 6.0)                             # 1 ... 1500 km
    tot, _ = _vs_oracle(torch, rows, masks, pairs, deltas, [1.0, 2.0, 3.0, 4.0, 5.0])
    assert tot["n"].sum() > 100000 and tot["n_censored"].sum() > 1000 and tot["hist_tau"][:, 0].sum() > 1000
    _vs_oracle(torch, rows, masks, pairs, deltas, every=2)


@pytest.mark.gpu
@pytest.mark.parametrize("nQ", [1, 255, 256, 257, 700001])
def test_fsle_vs_oracle_pair_counts(torch, nQ):
    """One pair, a block's edges and more pairs than one wave of resident blocks holds (grid-strided)."""
    rng = np.random.default_rng(nQ)
    rows, masks = _walk(rng, nP=600, S=12)
    a = rng.integers(0, 600, nQ)
    pairs = np.stack([a, (a + 1 + rng.integers(0, 599, nQ)) % 600], 1)
    tot, _ = _vs_oracle(torch, rows, masks, pairs, 2.0 ** (np.arange(30) / 3.0), again=nQ == 700001)
    assert nQ < 256 or tot["n"].sum() > nQ // 4


@pytest.mark.gpu
@pytest.mark.parametrize("K,ntau", [(2, 1), (2, 512), (64, 1), (64, 512)])
def test_fsle_vs_oracle_shape_limits(torch, K, ntau):
    """K = 2 and 64 thresholds, 1 and 512 exit-time edges (the largest shape: 135 KB of shared-memory counters)."""
    rng = np.random.default_rng(K * 1000 + ntau)
    rows, masks = _walk(rng, nP=800, S=40)
    a = rng.integers(0, 800, 40000)
    pairs = np.stack([a, (a + 1 + rng.integers(0, 799, 40000)) % 800], 1)
    deltas = np.array([20.0, 30.0]) if K == 2 else np.geomspace(1.0, 300.0, K)
    tau_edges = np.arange(1.0, ntau + 1) * (40.0 / ntau)
    tot, _ = _vs_oracle(torch, rows, masks, pairs, deltas, tau_edges)
    assert tot["n"].sum() > 1000


@pytest.mark.gpu
def test_finite_size_lyapunov(sit):
    """The host entry point: final state and windows equal the oracle's; bad shapes and sample_days are refused."""
    O = _ref()
    rng = np.random.default_rng(3)
    rows, masks = _walk(rng, nP=500, S=20)
    pairs = sit.SeparationPairs(rows[0], 1.0, 40.0, 5000, seed=2)
    deltas = 2.0 ** (np.arange(20) / 2.0)
    state, stats = sit.FiniteSizeLyapunov(np.array(rows), np.array(masks), pairs, 0.5, deltas=deltas)
    rs, rw = O.run(rows, masks, pairs, deltas)
    assert np.array_equal(state["level"], rs[-1][:, 0]) and np.array_equal(state["anchor"], rs[-1][:, 1])
    assert len(stats) == 20
    for a, b in zip(stats, rw):
        _same(a, b)
        assert a["sample_days"] == 0.5 and np.array_equal(a["deltas_km"], deltas)
    lam = sit.fsle_lambda(stats)
    n = _total(rw)["n"]
    assert np.isfinite(lam[(n > 0) & (_total(rw)["sum_tau"] > 0)]).all()
    for bad in (dict(pYX=np.array(rows)[:1]), dict(masks=np.array(masks)[:, :10]), dict(sample_days=0.0),
                dict(sample_days=np.nan), dict(pairs=[[0, 0]]), dict(deltas=[1.0])):
        kw = dict(pYX=np.array(rows), masks=np.array(masks), pairs=pairs, sample_days=0.5)
        kw.update(bad)
        with pytest.raises(ValueError):
            sit.FiniteSizeLyapunov(**kw)


@pytest.mark.gpu
def test_fsle_entry_point_refusals(torch, sit):
    """st_fsle_dev on real, aligned buffers refuses nQ < 1, t outside 1..65535, shapes past the limits, a NULL
    pointer, a start row without its mask and misaligned rows, pairs, state, edges or stats; it writes nothing then."""
    from sitrack_b200 import _lib
    from sitrack_b200 import fsle as F
    L = _lib.lib()
    dev = torch.device("cuda", 0)
    nP = 100
    yx = torch.zeros((nP + 1, 2), dtype=torch.float64, device=dev)
    yx[:, 1] = torch.arange(nP + 1, dtype=torch.float64)
    mk = torch.ones((nP,), dtype=torch.int8, device=dev)
    plan = F._Plan(torch, dev, np.stack([np.arange(50), np.arange(50, 100)], 1))
    (st,) = plan.outputs()
    big = torch.zeros((plan.nstat + 1,), dtype=torch.int64, device=dev)

    def call(nQ=50, t=1, K=19, ntau=17, yx_p=None, start=True, m0=True, pairs=None, state=None, deltas=None,
             tau=None, stats=None, m=True, poison=False):
        st.fill_(-3)
        if poison:                                                     # only for calls that must not launch
            plan.state.fill_(-7)
        torch.cuda.synchronize()
        y = yx.data_ptr() if yx_p is None else yx_p
        rc = L.st_fsle_dev(None, nQ, plan.pairs_t.data_ptr() if pairs is None else pairs,
                           plan.state.data_ptr() if state is None else state, y, mk.data_ptr() if m else None, t,
                           y if start else None, mk.data_ptr() if m0 else None, K,
                           plan.deltas_t.data_ptr() if deltas is None else deltas, ntau,
                           plan.tau_edges_t.data_ptr() if tau is None else tau,
                           st.data_ptr() if stats is None else stats, None)
        torch.cuda.synchronize()
        return rc

    assert call() == 0 and int(st[:20].sum()) == 50 and (plan.state.cpu().numpy()[:, 0] >= 0).all()
    assert call(start=False, m0=False, t=65535) == 0
    for kw in (dict(nQ=0), dict(nQ=-1), dict(t=0), dict(t=65536), dict(t=-1), dict(K=1), dict(K=65), dict(ntau=0),
               dict(ntau=513), dict(m=False), dict(m0=False), dict(start=False), dict(pairs=0), dict(state=0),
               dict(deltas=0), dict(tau=0), dict(stats=0), dict(yx_p=yx.data_ptr() + 8),
               dict(pairs=plan.pairs_t.data_ptr() + 4), dict(state=plan.state.data_ptr() + 4),
               dict(deltas=plan.deltas_t.data_ptr() + 4), dict(tau=plan.tau_edges_t.data_ptr() + 4),
               dict(stats=big.data_ptr() + 4)):
        if kw.get("start") is False:
            kw["m0"] = True                                            # a start mask without its row
        assert call(poison=True, **kw) == -1, kw
        assert (st.cpu().numpy() == -3).all() and (plan.state.cpu().numpy() == -7).all(), kw


def _engine(T, g, name, sort, rows, fsle=None, dispersion=None, deform=None, sink=None):
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
                    row_dtype=rows, sink=sink, deform=deform, dispersion=dispersion, fsle=fsle)
    eng.close()
    return res, sh


@pytest.mark.gpu
@pytest.mark.parametrize("every", [1, 48, 49])
@pytest.mark.parametrize("rows", ["f8", "f4"])
@pytest.mark.parametrize("name", ["uv1", "win"])
def test_track_fsle(torch, sit, gold_track, name, rows, every):
    """track(fsle=...): every window's statistics equal the oracle run over the series' rows (row 0 masked by
    rec_first on the `win` case), identical whether the buoys are stored in the caller's order or sorted on the host
    or the device, with the rows kept or sent to a sink; every = 49 > 48 records gives no window."""
    O = _ref()
    T, g = gold_track
    sh = np.random.default_rng(7).permutation(T["pos0"].shape[0])
    posC, mask = T[name + "_posC"][:, sh], T[name + "_mask"][:, sh]
    n = sh.size
    a, b = np.triu_indices(n, 1)
    pairs = np.concatenate([np.stack([a, b], 1), np.stack([b, a], 1)]).astype(np.int32)[::2]
    deltas = GOLD_DELTAS
    tau_edges = [1.0, 2.0, 4.0, 8.0]
    _, ref = O.run(list(posC), list(mask), pairs, deltas, tau_edges, every=every)
    spec = dict(pairs=pairs, every=every, deltas=deltas, tau_edges=tau_edges)
    for sort in ("none", "host", "dev"):
        res, _ = _engine(T, g, name, sort, rows, spec)
        got = res["fsle"]
        assert len(got) == len(ref) == 48 // every and "dispersion" not in res
        for st, rf in zip(got, ref):
            _same(st, rf)
            assert st["sample_days"] == every * RDT / 86400.0 and np.array_equal(st["deltas_km"], deltas)
        if rows == "f8" and sort == "host":
            _, kept = O.run(list(res["posC"]), list(res["mask"]), pairs, deltas, tau_edges, every=every)
            for st, rf in zip(got, kept):
                _same(st, rf)
    seen = []
    res, _ = _engine(T, g, name, "host", rows, dict(spec, sink=lambda w, st: seen.append((w, st))),
                     sink=lambda *a: None)
    assert "fsle" not in res and [w for w, _ in seen] == list(range(len(ref)))
    for (_, st), rf in zip(seen, ref):
        _same(st, rf)
    if every == 1:
        assert _total(ref)["n"].sum() > 100


@pytest.mark.gpu
def test_track_fsle_with_deform_and_dispersion(torch, sit, gold_track):
    """fsle together with deform and dispersion: their outputs are those of the same call without fsle, bit for bit,
    and the fsle statistics those of the call without them; refusals before anything runs."""
    T, g = gold_track
    sh = np.random.default_rng(7).permutation(T["pos0"].shape[0])
    pos0 = T["pos0"][sh]
    tri = sit.TriangulateCloud(pos0)
    pairs = np.concatenate([sit.MeshPairs(tri), sit.SeparationPairs(pos0, 1.0, 30.0, 500)])
    disp = dict(pairs=pairs, every=6, lags=4)
    fs = dict(pairs=pairs, every=2, deltas=GOLD_DELTAS)
    defo = dict(tri=tri, every=4)
    both, _ = _engine(T, g, "uv1", "host", "f8", fs, disp, defo)
    plain, _ = _engine(T, g, "uv1", "host", "f8", None, disp, defo)
    alone, _ = _engine(T, g, "uv1", "host", "f8", fs)
    assert "fsle" not in plain and len(both["fsle"]) == 24
    assert np.array_equal(both["posC"], plain["posC"]) and np.array_equal(both["mask"], plain["mask"])
    for a, b in zip(both["deform"], plain["deform"]):
        for k in sit.DEFORM_NAMES:
            assert np.array_equal(a[k], b[k]), k
    for a, b in zip(both["dispersion"], plain["dispersion"]):
        for k in a:
            assert np.ascontiguousarray(a[k]).tobytes() == np.ascontiguousarray(b[k]).tobytes(), k
    for a, b in zip(both["fsle"], alone["fsle"]):
        _same(a, b)
    assert sum(int(w["n"].sum()) for w in alone["fsle"]) > 50
    eng = engine_for(g, device=0)
    eng.set_buoys(pos0, T["jiT0"][sh].astype(np.int32))
    with pytest.raises(ValueError, match="streaming record loop"):
        eng.track((T["U"], T["V"], T["IC"]), 48, chunk=8, fsle=fs)
    with pytest.raises(ValueError):
        eng.track((T["U"], T["V"], T["IC"]), 48, sink=lambda *a: None, fsle=dict(fs, deltas=[1.0]))
    from sitrack_b200 import fsle as F
    F_max = F.MAX_SAMPLES
    try:
        F.MAX_SAMPLES = 23                                             # 24 windows: refused before anything runs
        with pytest.raises(ValueError, match="windows"):
            eng.track((T["U"], T["V"], T["IC"]), 48, sink=lambda *a: None, fsle=fs)
    finally:
        F.MAX_SAMPLES = F_max
    eng.close()


@pytest.mark.gpu
def test_cli_fsle_end_to_end(tmp_path, monkeypatch):
    """si3_part_tracker.py -F --fsle 2 on the 'small' synthetic case: the file's statistics are those of the engine
    API on the same inputs, and the tracking files are byte-identical to a run without the flag."""
    import si3_part_tracker as cli
    import sitrack_b200 as sit
    from make_synth_case import write_case
    r = write_case(str(tmp_path / "in"), grid="small", nrec=24, hss=3)
    runs = {}
    for tag, extra in (("plain", []), ("fsle", ["--fsle", "2", "--fsle-deltas", "1", "1.189207115", "40",
                                                "--fsle-pairs", "3000", "2", "200"])):
        d = tmp_path / tag
        d.mkdir()
        monkeypatch.chdir(d)
        monkeypatch.setattr(sys, "argv", _synth_argv(r, *extra))
        quiet(cli.main)
        runs[tag] = d
    files = sorted(os.listdir(runs["plain"] / "nc"))
    ffiles = [f for f in os.listdir(runs["fsle"] / "nc") if "_fsle_" in f]
    assert ffiles == ["NEMO-SI3_SYNTH4_SYN00_fsle_nemoTsi3_idlSeed_19961215h00_19961216h00.npz"], ffiles
    assert sorted(set(os.listdir(runs["fsle"] / "nc")) - set(ffiles)) == files
    for f in files:
        a, b = np.load(runs["plain"] / "nc" / f), np.load(runs["fsle"] / "nc" / f)
        assert sorted(a.files) == sorted(b.files)
        for k in a.files:
            assert a[k].dtype == b[k].dtype and a[k].tobytes() == b[k].tobytes(), (f, k)
    z = np.load(runs["fsle"] / "nc" / ffiles[0])
    deltas = 1.0 * 1.189207115 ** np.arange(40.0)
    assert z["time_start"].shape == (12,) and z["hist_tau"].shape == (12, 39, 18)
    assert np.array_equal(z["delta_km"], deltas) and np.array_equal(z["tau_edges"], sit.DEFAULT_TAU_EDGES)
    assert float(z["sample_days"]) == 2 * 3600.0 / 86400.0
    seed = [f for f in os.listdir(runs["fsle"] / "seed")][0]
    cache = np.load(runs["fsle"] / "seed" / seed)
    imaskt, _, _, _, _, Yf, Xf, _ = quiet(sit.GetModelGrid, r["mesh"])
    Yv, Xv, Yu, Xu = quiet(sit.GetModelUVGrid, r["mesh"])
    U, V, IC = r["records"]
    pos0 = cache["xPosC0"]
    pairs = sit.SeparationPairs(pos0, 2.0, 200.0, 3000, seed=0)
    seen = []
    with sit.TrackEngine(Yf, Xf, Yu, Xu, Yv, Xv, tmask=imaskt, uv_strategy=1, rdt=3600.0, rmin_conc=sit.rmin_conc,
                         device=0) as eng:
        eng.set_buoys(pos0, cache["vJIt"])
        eng.track((U[:24], V[:24], IC[:24]), 24, sink=lambda *a: None, row_dtype="f4",
                  fsle=dict(pairs=pairs, every=2, deltas=deltas, sink=lambda w, st: seen.append(st)))
    assert len(seen) == 12
    for w, st in enumerate(seen):
        for k in ("n_start", "n", "sum_tau", "sum_tau2", "n_censored", "hist_tau"):
            assert np.array_equal(z[k][w], st[k]), (w, k)
    assert z["n_start"].sum() > 1000


@pytest.mark.gpu
def test_bench_fsle_small():
    """tools/bench_fsle.py end to end on a small lattice: exit 0, state and statistics equal to the oracle."""
    import json
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_fsle.py"), "--ny", "300", "--nx", "300",
                        "--sep-pairs", "100000", "--check-pairs", "100000", "--seconds", "0.05"],
                       stdout=subprocess.PIPE, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    assert res["oracle_check_passed"] and res["fsle_us"] > 0 and res["dispersion_single_origin_us"] > 0
