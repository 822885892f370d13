"""Invariants the default step kernel relies on.

Cell bits as a constant: st_create reduces the cell bits over the cells a live buoy can occupy; where they are uniform
(6) the default chained step takes them from the instruction stream instead of gathering them per buoy.  A grid with
one odd cell in that domain must fall back to the gather, and either way the trajectories are the C oracle's, bit for
bit.
"""
import numpy as np
import pytest

from conftest import engine_for


def _run_oracle_and_track(corc, g, nrec=24, scale=3.0, seed_khss=2):
    import synth
    U, V, IC = synth.make_records(g, nrec, seed=1)
    U *= np.float32(scale); V *= np.float32(scale)
    ids, SG, SC = synth.hss_seeds(g, IC[0], khss=seed_khss)
    with engine_for(g) as eng:
        eng.set_locate_grid(g["latT"], g["lonT"], g["ResKM"])
        cell, near, keep = eng.seed_locate(SG, SC, IC[0])
        ik = np.flatnonzero(keep)
        pos0, cell0 = SC[ik], cell[ik]
        eng.set_buoys(pos0, cell0)
        bits = eng.cell_bits_uniform()
        r = eng.track((U, V, IC), nrec, pos0=pos0)
        p, c, a = eng.get_state()
    ref = corc.track(g, U, V, IC, pos0, cell0.astype(np.int64), do_latlon=False)
    return bits, r, (p, c, a), ref


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["uniform", "one_odd_cell"])
def test_constant_cell_bits_instance_vs_oracle(torch, corc, case):
    import synth
    g = synth.make_grid(**synth.GRID_PRESETS["small"], seed=0)
    if case == "one_odd_cell":
        # fold the four cells around one corner inside the buoy domain: their bit 2 (convex anticlockwise) goes
        Nj, Ni = g["tmask"].shape
        j, i = Nj // 2, Ni // 2
        g["Yf"] = g["Yf"].copy(); g["Xf"] = g["Xf"].copy()
        g["Yf"][j, i] += 0.9 * (g["Yf"][j + 1, i] - g["Yf"][j, i]) + 0.9 * (g["Yf"][j, i + 1] - g["Yf"][j, i])
        g["Xf"][j, i] += 0.9 * (g["Xf"][j + 1, i] - g["Xf"][j, i]) + 0.9 * (g["Xf"][j, i + 1] - g["Xf"][j, i])
    bits, r, (p, c, a), ref = _run_oracle_and_track(corc, g)
    assert bits == (6 if case == "uniform" else -1)
    assert ref["ncross"] > 100
    assert np.array_equal(r["posC"], ref["posC"])
    assert np.array_equal(r["mask"], ref["mask"]) and np.array_equal(r["n_alive"], ref["nalive"])
    assert np.array_equal(c, ref["jiT"]) and np.array_equal(a, ref["alive"])

