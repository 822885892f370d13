"""The pair-dispersion kernels (csrc/st_disperse.cu) pinned to their order-exact reference
(oracle/dispersion_ref.order_sums) where a kernel could be subtly wrong and still agree with fsum within 1e-11.

The fixed summation order of the moment sums is the contract that keeps the statistics identical run to run, on every
device and in every buoy storage order, so the f8 sums and the block partials (read from the front of the plan's
scratch, [block][origin][class][4]) are compared bit for bit; counts exactly.  Pinned: the golden rows; a 200
k-buoy lattice whose blocks run two or three tiles; nQ around a warp, a block and the 1184 x 256 pairs where the grid
saturates; 63 class edges with warps of 32 classes, of one class and of no valid lane, and classes with no pair; 64
fused origins; masked buoys whose positions are NaN, +-inf or 1e200; valid pairs with a NaN coordinate, r0 = inf and
r0 = 0; the largest class/bin shapes the shared memory holds with as many origins as lags (one bin more refused);
and track()'s ring of origin rows at one slot, 48 slots under 64 lags, a dropped partial window, one window and none.

CPU: order_sums against lag_stats' fsum, the premises of every GPU case, and the shared-memory shapes.  GPU: the
rest."""
import ctypes as C
import functools

import numpy as np
import pytest

from conftest import TRACK_CASES
from test_deformation_scales import RDT
from test_dispersion import _engine, _fused_and_single, _lattice_case

FILL = -9999.0
TILE, GRID = 256, 1184
SMEM = 227 * 1024                                     # the shared memory a block of k_disperse may opt into
GOLD_ROWS = [(0, 1), (0, 6), (5, 29), (12, 48), (47, 48)]
GOLD_EDGES = [1.0, 3.0, 10.0, 30.0, 100.0]
NQ = [1, 31, 32, 33, 255, 256, 257, 303103, 303104, 303105]


def _same_bits(a, b):
    """Element-wise: the same bit pattern, or both NaN.  -0.0 and +0.0 differ."""
    a, b = np.asarray(a), np.asarray(b)
    assert a.dtype == b.dtype and a.shape == b.shape, (a.dtype, b.dtype, a.shape, b.shape)
    u = {4: np.uint32, 8: np.uint64}[a.dtype.itemsize]
    return (a.view(u) == b.view(u)) | (np.isnan(a) & np.isnan(b))


def _nblk(nQ):
    return min(max(-(-nQ // TILE), 1), GRID)


def _tiles_per_block(nQ):
    """(nblk,) the number of tiles of 256 pairs each block of k_disperse runs."""
    nb, nt = _nblk(nQ), -(-nQ // TILE)
    return np.array([len(range(b, nt, nb)) for b in range(nb)])


def _smem(nact, ncedge, nedge):
    """DESIGN.md section 13: nact*C*(nedge+1) ints plus ncedge + nedge + 4*C*(nact + 16) doubles."""
    C_ = ncedge + 1
    return 4 * nact * C_ * (nedge + 1) + 8 * (ncedge + nedge + 4 * C_ * (nact + 16))


def _max_bins(nact, ncedge):
    nedge = 1
    while _smem(nact, ncedge, nedge + 1) <= SMEM:
        nedge += 1
    return nedge


# ---- the cases ------------------------------------------------------------------------------------

@functools.lru_cache(maxsize=1)
def _lattice_pairs():
    """The inputs of test_pairs_vs_oracle_lattice: ~200 k buoys with masks and deaths, mesh and sampled pairs."""
    import sitrack_b200 as sit
    yx0, yx1, m0, m1, tri = _lattice_case(np.random.default_rng(11))
    pairs = np.concatenate([sit.MeshPairs(tri), sit.SeparationPairs(yx0, 10.0, 1000.0, 200000, seed=5)])
    return yx0, yx1, m0, m1, pairs


def _count_case(nQ):
    """nQ random pairs of 5000 buoys over 2000 km, 5 % masked in each row; pair 0 joins buoys 0 and 1, which count."""
    rng = np.random.default_rng(nQ)
    nP = 5000
    yx0 = rng.uniform(0, 2000.0, (nP, 2))
    yx1 = yx0 + rng.normal(0, 3.0, yx0.shape)
    m0, m1 = (rng.random(nP) > 0.05).astype(np.int8), (rng.random(nP) > 0.05).astype(np.int8)
    m0[:2] = m1[:2] = 1
    a = rng.integers(0, nP, nQ)
    pairs = np.stack([a, (a + 1 + rng.integers(0, nP - 1, nQ)) % nP], 1).astype(np.int32)
    pairs[0] = (0, 1)
    return yx0, yx1, m0, m1, pairs


DENSE_EDGES = 2.0 * np.arange(1, 64)                  # 63 class edges: class c holds r0 in [2c, 2c + 2)


def _dense_case():
    """Pairs on their own buoys, r0 = 2c + 1 +- 0.8 for the class c wanted, in 4 tiles and a partial one.  Tile 0:
    warp 0 has classes 0 .. 31 lane by lane, warp 1 the odd classes 63, 61, ..., 1, warp 2 only class 17, warp 3 no
    valid lane (one mask byte off per pair, each of the four in turn); the other warps draw classes below 32 or odd
    at random, and 10 % of the pairs after tile 0 are masked.  The even classes 32 .. 62 have no pair."""
    rng = np.random.default_rng(31)
    nQ = 4 * TILE + 45
    want = np.where(rng.random(nQ) < 0.5, rng.integers(0, 32, nQ), 2 * rng.integers(0, 32, nQ) + 1)
    want[0:32] = np.arange(32)
    want[32:64] = np.arange(63, 0, -2)
    want[64:96] = 17
    r0 = 2.0 * want + 1.0 + rng.uniform(-0.8, 0.8, nQ)
    th = rng.uniform(0, 2 * np.pi, nQ)
    a = rng.uniform(0, 500.0, (nQ, 2))
    b = a + np.stack([r0 * np.sin(th), r0 * np.cos(th)], 1)
    yx0 = np.stack([a, b], 1).reshape(-1, 2)
    yx1 = yx0 + rng.normal(0.0, 0.3, yx0.shape)
    m0, m1 = np.ones(2 * nQ, np.int8), np.ones(2 * nQ, np.int8)
    off = np.flatnonzero(rng.random(nQ) < 0.1)
    off = off[off >= TILE]
    m0[2 * off + rng.integers(0, 2, off.size)] = 0
    for j, i in enumerate(range(96, 128)):
        (m0, m1)[j % 4 // 2][2 * i + j % 2] = 0
    pairs = np.arange(2 * nQ, dtype=np.int32).reshape(nQ, 2)
    return yx0, yx1, m0, m1, pairs


def _poisoned_case(poison):
    """A 120 x 120 lattice (2 % masked at the origin row, 3 % more at the closing row), mesh and sampled pairs; the
    positions of every masked buoy set to `poison` in both rows.  -> (poisoned rows, finite rows, masks, pairs)."""
    import sitrack_b200 as sit
    yx0, yx1, m0, m1, tri = _lattice_case(np.random.default_rng(2), 120)
    pairs = np.concatenate([sit.MeshPairs(tri), sit.SeparationPairs(yx0, 2.0, 300.0, 20000, seed=1)])
    dead = (m0 == 0) | (m1 == 0)
    p0, p1 = yx0.copy(), yx1.copy()
    p0[dead] = p1[dead] = poison
    return (p0, p1), (yx0, yx1), (m0, m1), pairs


NF_EDGES = [1.0, 10.0, 100.0, 1000.0]                 # classes: < 1, [1, 10), [10, 100), [100, 1000), >= 1000 and NaN
NF_CASES = {
    # name: (origin [y,x] of a and b, closing [y,x] of a and b, class, sums of that class finite (r0, dr, dr2, dD2))
    "nan_origin": ([[np.nan, 0.0], [3.0, 4.0]], [[0.0, 0.0], [3.0, 4.0]], 4, [False] * 4),
    "nan_closing": ([[0.0, 0.0], [3.0, 4.0]], [[0.0, np.nan], [3.0, 4.0]], 1, [True, False, False, False]),
    "r0_inf": ([[0.0, 0.0], [1e200, 0.0]], [[0.0, 0.0], [1e200, 0.0]], 4, [False, False, False, True]),
    "r1_inf": ([[0.0, 0.0], [30.0, 40.0]], [[0.0, 0.0], [1e200, 40.0]], 2, [True, False, False, False]),
    "r0_zero": ([[5.0, 5.0], [5.0, 5.0], [7.0, 7.0], [7.0, 7.0]],
                [[5.0, 5.0], [8.0, 9.0], [7.0, 7.0], [7.0, 7.0]], 0, [True] * 4),
}


def _nonfinite_case(name):
    """The special pair(s) of NF_CASES[name] at lanes 5 (and 20) of warp 0, among ordinary pairs drifting slowly,
    with r0 spread over every class (the overflow class at 1000 .. 2000 km).  -> (yx0, yx1, m0, m1, pairs, special
    pair indices, its class)."""
    o, c, cls, _ = NF_CASES[name]
    rng = np.random.default_rng(41)
    nQ = 64
    r0 = 10.0 ** rng.uniform(-1.0, 3.3, nQ)
    th = rng.uniform(0, 2 * np.pi, nQ)
    a = rng.uniform(0, 100.0, (nQ, 2))
    b = a + np.stack([r0 * np.sin(th), r0 * np.cos(th)], 1)
    yx0 = np.stack([a, b], 1).reshape(-1, 2)
    yx1 = yx0 + rng.normal(0.0, 0.01, yx0.shape)
    special = [5, 20][:len(o) // 2]
    for k, i in enumerate(special):
        yx0[2 * i:2 * i + 2], yx1[2 * i:2 * i + 2] = o[2 * k:2 * k + 2], c[2 * k:2 * k + 2]
    one = np.ones(2 * nQ, np.int8)
    return yx0, yx1, one, one.copy(), np.arange(2 * nQ, dtype=np.int32).reshape(nQ, 2), special, cls


def _limit_case(lags, ncedge):
    """The largest bins the shared memory holds at `lags` active origins and `ncedge` class edges: rows of 3000 buoys
    drifting over lags + 1 steps with 1 % dying per step, 20 000 sampled pairs, geometric class edges over 2 .. 1500
    km and bins over 1e-4 .. 1e2 day-1."""
    import sitrack_b200 as sit
    rng = np.random.default_rng(lags * 100 + ncedge)
    nP = 3000
    rows = [rng.uniform(0, 1500.0, (nP, 2))]
    masks = [np.ones(nP, np.int8)]
    for _ in range(lags):
        rows.append(rows[-1] + rng.normal(0.2, 2.0, (nP, 2)))
        masks.append(masks[-1] * (rng.random(nP) > 0.01).astype(np.int8))
    pairs = sit.SeparationPairs(rows[0], 2.0, 1500.0, 20000, seed=lags)
    r_edges = np.geomspace(5.0, 1000.0, ncedge) if ncedge > 1 else np.array([50.0])
    bins = np.geomspace(1e-4, 1e2, _max_bins(lags, ncedge))
    return rows, masks, pairs, r_edges, bins


LIMITS = [(64, 9, 79, 231104), (64, 63, 3, 229904), (64, 1, 436, 232360), (1, 63, 745, 232256)]


# ---- the device pass and its check ----------------------------------------------------------------

def _launch(torch, rows, masks, pairs, lags, dt, r_edges=None, bins=None, per_pair=False):
    """One st_dispersion_dev call: closing row rows[-1], origin rows[-1-l] at lag l = 1 .. len(rows)-1.  -> dict(hist
    (lags, C, NB), sums (lags, C, 4), part (nblk, nact, C, 4) from the front of the scratch, pp (4, nQ) or None, the
    plan's r_edges and bins)."""
    from sitrack_b200 import dispersion as P
    dev = torch.device("cuda", 0)
    t = lambda a, d: torch.from_numpy(np.ascontiguousarray(a, d)).to(dev)
    plan = P._Plan(torch, dev, pairs, lags, r_edges, bins)
    Y, M = [t(y, np.float64) for y in rows], [t(m, np.int8) for m in masks]
    nact = len(rows) - 1
    h, s = plan.outputs()
    pp = torch.empty((4, plan.nQ), dtype=torch.float64, device=dev) if per_pair else None
    plan.launch(None, Y[-1], M[-1], [(Y[-1 - l], M[-1 - l], l) for l in range(1, nact + 1)], dt, h, s, pp,
                torch.cuda.current_stream(dev))
    torch.cuda.synchronize(dev)
    nb = _nblk(plan.nQ)
    assert plan.scratch_bytes == nb * lags * plan.C * 4 * 8           # the grid depends on nQ only, capped at 1184
    part = plan.scratch[:nb * nact * plan.C * 4].cpu().numpy().reshape(nb, nact, plan.C, 4)
    return dict(hist=h.cpu().numpy(), sums=s.cpu().numpy(), part=part, pp=None if pp is None else pp.cpu().numpy(),
                r_edges=plan.r_edges, bins=plan.bins)


def _check(got, rows, masks, pairs, dt):
    """Every active lag l: sums and block partials bit for bit against order_sums, counts exactly against lag_hist;
    the lags not active all zero.  -> [(sums, part) of order_sums per lag]."""
    from oracle import dispersion_ref as O
    nact = len(rows) - 1
    ref = []
    for l in range(1, nact + 1):
        args = (rows[-1 - l], rows[-1], masks[-1 - l], masks[-1], pairs)
        s, part = O.order_sums(*args, r_edges=got["r_edges"])
        same = _same_bits(got["part"][:, l - 1], part)
        assert same.all(), "lag %d: %d of %d block partials differ" % (l, (~same).sum(), same.size)
        same = _same_bits(got["sums"][l - 1], s)
        assert same.all(), "lag %d: %d of %d sums differ" % (l, (~same).sum(), same.size)
        assert np.array_equal(got["hist"][l - 1], O.lag_hist(O.per_pair(*args), l * dt, got["r_edges"], got["bins"]))
        ref.append((s, part))
    assert not got["hist"][nact:].any() and not got["sums"][nact:].view(np.uint64).any()
    return ref


# ---- CPU: order_sums agrees with fsum -------------------------------------------------------------

def _fsum_case(name):
    if name == "lattice":
        return _lattice_pairs() + (None,)
    if name == "golden":
        from conftest import GOLD
        T = np.load(GOLD + "/track_tiny.npz")
        posC, mask = T["uv1_posC"], T["uv1_mask"]
        a, b = np.triu_indices(posC.shape[1], 1)
        pairs = np.concatenate([np.stack([a, b], 1), np.stack([b, a], 1)]).astype(np.int32)
        return posC[5], posC[29], mask[5], mask[29], pairs, GOLD_EDGES
    return _count_case(int(name[2:])) + (None,)


@pytest.mark.parametrize("name", ["lattice", "golden", "nQ1", "nQ257"])
def test_order_sums_within_fsum(name):
    """order_sums (the device's order) and lag_stats' math.fsum agree within 1e-11 fsum(|terms|); the block partials
    add up to the sums."""
    from oracle import dispersion_ref as O
    yx0, yx1, m0, m1, pairs, r_edges = _fsum_case(name)
    kw = {} if r_edges is None else dict(r_edges=r_edges)
    s, part = O.order_sums(yx0, yx1, m0, m1, pairs, **kw)
    st = O.lag_stats(yx0, yx1, m0, m1, pairs, 0.25, **kw)
    assert part.shape == (_nblk(pairs.shape[0]),) + s.shape
    err = np.abs(s - st["sums"])
    assert (err <= 1e-11 * st["absum"]).all(), err.max()
    assert (np.abs(part.sum(0) - st["sums"]) <= 1e-11 * st["absum"]).all()
    assert st["hist"].sum() > 0 and (st["sums"] != 0).any()


def _literal_order_sums(cls, v, C_, nblk):
    """DESIGN section 13's order one lane and one add at a time, in Python floats (IEEE f8, correctly rounded)."""
    nQ, ntile = cls.size, -(-cls.size // TILE)
    part = [[[0.0] * 4 for _ in range(C_)] for _ in range(nblk)]
    for b in range(nblk):
        for t in range(b, ntile, nblk):
            for w in range(8):
                lanes = [t * TILE + w * 32 + l for l in range(32)]
                for c in range(C_):
                    for q in range(4):
                        x = [float(v[i, q]) if i < nQ and cls[i] == c else 0.0 for i in lanes]
                        for sh in (16, 8, 4, 2, 1):
                            x = [x[l] + x[l ^ sh] for l in range(32)]
                        part[b][c][q] = part[b][c][q] + x[0]
    s = [[[0.0] * 4 for _ in range(C_)] for _ in range(TILE)]
    for t in range(TILE):
        for b in range(t, nblk, TILE):
            s[t] = [[s[t][c][q] + part[b][c][q] for q in range(4)] for c in range(C_)]
    w = TILE // 2
    while w:
        for t in range(w):
            s[t] = [[s[t][c][q] + s[t + w][c][q] for q in range(4)] for c in range(C_)]
        w //= 2
    return np.array(s[0]), np.array(part)


@pytest.mark.parametrize("grid,nQ,r_edges", [(3, 2000, None), (260, 261 * TILE + 7, [300.0])])
def test_order_sums_equals_literal_order(monkeypatch, grid, nQ, r_edges):
    """With the grid capped at 3 blocks (8 tiles: two rounds for every block, a third for blocks 0 and 1) and at 260
    (slots 0 .. 3 of the final sum add a second block partial), order_sums gives the bits of a lane-by-lane loop,
    on random values with a NaN and an inf among them."""
    from oracle import dispersion_ref as O
    yx0, yx1, m0, m1, pairs = _count_case(nQ)
    a, b = pairs[300]
    m0[[a, b]] = m1[[a, b]] = 1
    yx1[1, 1], yx1[a] = np.nan, (1e200, 0.0)                   # pair 0: dr NaN; pair 300: r1 = inf
    r_edges = O.DEFAULT_R_EDGES if r_edges is None else np.array(r_edges)
    monkeypatch.setattr(O, "MAX_GRID", grid)
    s, part = O.order_sums(yx0, yx1, m0, m1, pairs, r_edges)
    p = O.per_pair(yx0, yx1, m0, m1, pairs)
    cls = O.pair_class(p, r_edges)
    with np.errstate(all="ignore"):
        v = np.stack([p["r0"], p["dr"], p["dr"] * p["dr"], p["dD2"]], 1)
    assert (~np.isfinite(v[cls >= 0])).any() and part.shape[0] == grid
    ls, lp = _literal_order_sums(cls, v, r_edges.size + 1, grid)
    assert _same_bits(part, lp).all() and _same_bits(s, ls).all()


# ---- CPU: the premises of the GPU cases ------------------------------------------------------------

def test_premise_tiles_per_block():
    """The lattice's blocks run two or three tiles; nQ = 303 104 is the last count with one tile per block, 303 105
    gives block 0 a second tile of one pair."""
    tp = _tiles_per_block(_lattice_pairs()[4].shape[0])
    assert _lattice_pairs()[4].shape[0] > GRID * TILE and tp.size == GRID and tp.max() == 3 and tp.min() == 2
    for nQ in NQ:
        tp = _tiles_per_block(nQ)
        assert tp.size == min(-(-nQ // TILE), GRID)
        assert tp.tolist() == ([2] + [1] * (GRID - 1) if nQ == 303105 else [1] * tp.size), nQ
    assert 303104 == GRID * TILE


@pytest.mark.parametrize("nQ", NQ)
def test_premise_pair_counts(nQ):
    from oracle import dispersion_ref as O
    yx0, yx1, m0, m1, pairs = _count_case(nQ)
    assert pairs.shape == (nQ, 2) and (pairs[:, 0] != pairs[:, 1]).all()
    cls = O.pair_class(O.per_pair(yx0, yx1, m0, m1, pairs), O.DEFAULT_R_EDGES)
    assert cls[0] >= 0
    if nQ > 1:
        assert (cls < 0).any() and np.unique(cls[cls >= 0]).size >= 3


def test_premise_class_dense_warps():
    from oracle import dispersion_ref as O
    yx0, yx1, m0, m1, pairs = _dense_case()
    cls = O.pair_class(O.per_pair(yx0, yx1, m0, m1, pairs), DENSE_EDGES)
    w = cls[:TILE].reshape(8, 32)
    assert w[0].tolist() == list(range(32)) and w[1].tolist() == list(range(63, 0, -2))
    assert (w[2] == 17).all() and (w[3] == -1).all()
    assert {(m0[2 * i] == 0) + 2 * (m0[2 * i + 1] == 0) + 4 * (m1[2 * i] == 0) + 8 * (m1[2 * i + 1] == 0)
            for i in range(96, 128)} == {1, 2, 4, 8}
    assert all(np.unique(w[k][w[k] >= 0]).size > 8 for k in range(4, 8))
    empty = sorted(set(range(64)) - set(cls[cls >= 0].tolist()))
    assert empty == list(range(32, 64, 2))
    assert (cls[TILE:] < 0).sum() > 50 and pairs.shape[0] % TILE == 45


@pytest.mark.parametrize("poison", [np.nan, np.inf, -np.inf, 1e200])
def test_premise_poisoned_masks(poison):
    """The poisoned positions make the values of pairs that do not count non-finite (so that a multiply by 0 would
    reach the sums), in many warps; the finite run has pairs that do not count too."""
    from oracle import dispersion_ref as O
    (p0, p1), (yx0, yx1), (m0, m1), pairs = _poisoned_case(poison)
    p = O.per_pair(p0, p1, m0, m1, pairs)
    bad = ~p["valid"] & ~(np.isfinite(p["r0"]) & np.isfinite(p["dr"]) & np.isfinite(p["dD2"]))
    assert bad.sum() > 1000 and np.unique(np.flatnonzero(bad) // 32).size > 500
    q = O.per_pair(yx0, yx1, m0, m1, pairs)
    assert np.array_equal(p["valid"], q["valid"]) and 0 < (~q["valid"]).sum() < q["valid"].sum()
    for k in ("r0", "dr", "dD2"):
        assert _same_bits(p[k][p["valid"]], q[k][q["valid"]]).all()


@pytest.mark.parametrize("name", list(NF_CASES))
def test_premise_nonfinite_pairs(name):
    """The special pairs are valid with the non-finite values they are built for, in the class DESIGN section 13
    gives (NaN last) and the overflow stretch bin; every ordinary pair is finite, in a stretch bin below it, and
    every class has an ordinary pair."""
    from oracle import dispersion_ref as O
    yx0, yx1, m0, m1, pairs, special, cls = _nonfinite_case(name)
    p = O.per_pair(yx0, yx1, m0, m1, pairs)
    c = O.pair_class(p, np.array(NF_EDGES))
    assert p["valid"].all() and (c[special] == cls).all()
    with np.errstate(all="ignore"):
        s = np.abs(p["dr"]) / (p["r0"] * 0.25)
    r0, dr, dD2, s = p["r0"][special], p["dr"][special], p["dD2"][special], s[special]
    if name == "nan_origin":
        assert np.isnan([r0, dr, dD2, s]).all()
    elif name == "nan_closing":
        assert np.isfinite(r0).all() and np.isnan([dr, dD2, s]).all()
    elif name == "r0_inf":
        assert (r0 == np.inf).all() and np.isnan([dr, s]).all() and (dD2 == 0).all()
    elif name == "r1_inf":
        assert np.isfinite(r0).all() and (dr == np.inf).all() and (dD2 == np.inf).all() and (s == np.inf).all()
    else:
        assert (r0 == 0).all() and s[0] == np.inf and np.isnan(s[1]) and np.isfinite([dr, dD2]).all()
    rest = np.delete(np.arange(pairs.shape[0]), special)
    assert np.isfinite([p["r0"][rest], p["dr"][rest], p["dD2"][rest]]).all()
    with np.errstate(all="ignore"):
        sr = np.abs(p["dr"][rest]) / (p["r0"][rest] * 0.25)
    assert (sr < O.DEFAULT_BINS[-1]).all() and set(c[rest].tolist()) == set(range(len(NF_EDGES) + 1))


@pytest.mark.parametrize("lags,ncedge,nedge,smem", LIMITS)
def test_premise_shared_memory_limits(lags, ncedge, nedge, smem):
    """DESIGN section 13's formula against 227 KB gives the largest bins; st_dispersion_scratch_bytes accepts that
    shape with `lags` origins and refuses one bin more."""
    from sitrack_b200 import _lib
    assert _max_bins(lags, ncedge) == nedge and _smem(lags, ncedge, nedge) == smem
    assert smem <= SMEM < _smem(lags, ncedge, nedge + 1)
    out = C.c_int64(-5)
    assert _lib.lib().st_dispersion_scratch_bytes(20000, lags, ncedge, nedge, C.byref(out)) == 0
    assert out.value == _nblk(20000) * lags * (ncedge + 1) * 4 * 8
    assert _lib.lib().st_dispersion_scratch_bytes(20000, lags, ncedge, nedge + 1, C.byref(out)) == -1
    rows, masks, pairs, r_edges, bins = _limit_case(lags, ncedge)
    assert len(rows) == lags + 1 and r_edges.size == ncedge and bins.size == nedge


# ---- GPU: shapes -----------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TRACK_CASES))
def test_sums_bits_golden(torch, sit, gold_track, name):
    """The inputs of test_pairs_vs_oracle_golden: every ordered pair of the 94 golden buoys on five row pairs."""
    T, _ = gold_track
    posC, mask = T[name + "_posC"], T[name + "_mask"]
    a, b = np.triu_indices(posC.shape[1], 1)
    pairs = np.concatenate([np.stack([a, b], 1), np.stack([b, a], 1)]).astype(np.int32)
    n = 0
    for k0, k1 in GOLD_ROWS:
        dt = (k1 - k0) * RDT / 86400.0
        rows, masks = [posC[k0], posC[k1]], [mask[k0], mask[k1]]
        got = _launch(torch, rows, masks, pairs, 1, dt, r_edges=GOLD_EDGES)
        _check(got, rows, masks, pairs, dt)
        n += int(got["hist"].sum())
    assert n > 5000


@pytest.mark.gpu
def test_sums_bits_lattice(torch, sit):
    """~200 k buoys, 797 k mesh and sampled pairs: every block runs two or three tiles."""
    yx0, yx1, m0, m1, pairs = _lattice_pairs()
    assert pairs.shape[0] > GRID * TILE
    got = _launch(torch, [yx0, yx1], [m0, m1], pairs, 1, 0.25)
    _check(got, [yx0, yx1], [m0, m1], pairs, 0.25)
    assert (got["hist"][0, :-1].sum(1) > 10000).all()


@pytest.mark.gpu
@pytest.mark.parametrize("nQ", NQ)
def test_sums_bits_pair_counts(torch, sit, nQ):
    """One pair, a warp and one pair either side, a block and one either side, and the grid's saturation: 1184 tiles
    less one pair, exactly, and plus one pair (block 0 runs a second tile)."""
    yx0, yx1, m0, m1, pairs = _count_case(nQ)
    got = _launch(torch, [yx0, yx1], [m0, m1], pairs, 1, 0.5)
    assert got["part"].shape[0] == _nblk(nQ)
    _check(got, [yx0, yx1], [m0, m1], pairs, 0.5)


@pytest.mark.gpu
def test_class_dense_warps(torch, sit):
    """63 class edges: a warp of 32 classes, one of the odd classes, one of a single class and one with no valid lane;
    the classes with no pair have sums whose bits are all zero."""
    yx0, yx1, m0, m1, pairs = _dense_case()
    rows, masks = [yx0, yx1], [m0, m1]
    got = _launch(torch, rows, masks, pairs, 1, 0.25, r_edges=DENSE_EDGES)
    _check(got, rows, masks, pairs, 0.25)
    empty = np.arange(32, 64, 2)
    assert not got["sums"][0, empty].view(np.uint64).any() and not got["part"][:, 0, empty].view(np.uint64).any()
    assert not got["hist"][0, empty].any() and (got["hist"][0].sum(1) > 0).sum() == 48


@pytest.mark.gpu
def test_fused_origins_bits(torch, sit):
    """64 origins in one call: each lag's sums (fused and single calls alike) and the per-origin block partials of the
    fused call equal order_sums for that origin."""
    rng = np.random.default_rng(64)
    nP = 3000
    rows = [rng.uniform(0, 1500.0, (nP, 2))]
    masks = [np.ones(nP, np.int8)]
    for _ in range(64):
        rows.append(rows[-1] + rng.normal(0.2, 2.0, (nP, 2)))
        masks.append(masks[-1] * (rng.random(nP) > 0.01).astype(np.int8))
    pairs = sit.SeparationPairs(rows[0], 5.0, 1000.0, 40000, seed=64)
    dt = 0.125
    fused, single, _ = _fused_and_single(torch, rows, masks, pairs, 64, dt)
    got = _launch(torch, rows, masks, pairs, 64, dt)
    assert got["part"].shape[:2] == (_nblk(pairs.shape[0]), 64)
    ref = _check(got, rows, masks, pairs, dt)
    for l, (s, _) in enumerate(ref):
        assert _same_bits(fused[1][l], s).all() and _same_bits(single[1][l], s).all(), l + 1
    assert np.array_equal(fused[0], got["hist"]) and np.array_equal(single[0], got["hist"])


# ---- GPU: masked and non-finite values ------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("poison", [np.nan, np.inf, -np.inf, 1e200])
def test_masked_buoys_poisoned(torch, sit, poison):
    """NaN, +-inf or 1e200 at the positions of masked buoys reach neither the counts nor the sums nor the block
    partials (the same bits as with their finite positions); their pairs' per-pair values are FillValue."""
    (p0, p1), (yx0, yx1), (m0, m1), pairs = _poisoned_case(poison)
    got = _launch(torch, [p0, p1], [m0, m1], pairs, 1, 0.25, per_pair=True)
    fin = _launch(torch, [yx0, yx1], [m0, m1], pairs, 1, 0.25, per_pair=True)
    _check(got, [p0, p1], [m0, m1], pairs, 0.25)
    assert np.array_equal(got["hist"], fin["hist"])
    for k in ("sums", "part", "pp"):
        assert _same_bits(got[k], fin[k]).all(), k
    from oracle import dispersion_ref as O
    valid = O.per_pair(p0, p1, m0, m1, pairs)["valid"]
    assert (got["pp"][:, ~valid] == FILL).all() and np.isfinite(got["sums"]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(NF_CASES))
def test_valid_pairs_nonfinite(torch, sit, name):
    """A valid pair with a NaN coordinate, r0 = inf (s NaN), r1 = inf (s inf) or r0 = 0 (s inf and NaN): its per-pair
    values bit for bit, its count in the class DESIGN section 13 gives and the overflow stretch bin, the sums of that
    class non-finite exactly where the reference's are (NaN with NaN, inf with the same inf), every other class
    finite; all bit for bit against order_sums."""
    from oracle import dispersion_ref as O
    yx0, yx1, m0, m1, pairs, special, cls = _nonfinite_case(name)
    rows, masks = [yx0, yx1], [m0, m1]
    got = _launch(torch, rows, masks, pairs, 1, 0.25, r_edges=NF_EDGES, per_pair=True)
    _check(got, rows, masks, pairs, 0.25)
    assert _same_bits(got["pp"], O.per_pair_filled(yx0, yx1, m0, m1, pairs)).all()
    h, s = got["hist"][0], got["sums"][0]
    assert h[cls, -1] == len(special) and h[:, -1].sum() == len(special)
    assert np.isfinite(s[cls]).tolist() == NF_CASES[name][3]
    assert np.isfinite(np.delete(s, cls, 0)).all()
    if name == "r0_inf":
        assert s[cls, 0] == np.inf
    if name == "r1_inf":
        assert (s[cls, 1:] == np.inf).all()


# ---- GPU: the shared-memory limits --------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("lags,ncedge,nedge,smem", LIMITS)
def test_shared_memory_limits(torch, sit, lags, ncedge, nedge, smem):
    """The largest bins at 64 lags with 9, 63 and 1 class edges and at 1 lag with 63, `lags` origins active: every
    lag bit for bit; a plan one bin larger is refused."""
    from sitrack_b200 import dispersion as P
    rows, masks, pairs, r_edges, bins = _limit_case(lags, ncedge)
    dt = 0.125
    got = _launch(torch, rows, masks, pairs, lags, dt, r_edges=r_edges, bins=bins)
    assert got["hist"].shape == (lags, ncedge + 1, nedge + 1)
    _check(got, rows, masks, pairs, dt)
    assert (got["hist"].sum((1, 2)) > 1000).all()
    with pytest.raises(sit.SitrackCudaError):
        P._Plan(torch, torch.device("cuda", 0), pairs, lags, r_edges, np.r_[bins, bins[-1] * 2])


# ---- GPU: the engine's windows -----------------------------------------------------------------------

_WINDOW_REFS = {}


def _window_refs(T, name, every, lags, pairs, r_edges):
    """Per window: (hist (lags, C, NB), sums (lags, C, 4)) from lag_hist and order_sums on the golden f8 rows in the
    caller's order of _engine."""
    from oracle import dispersion_ref as O
    key = (name, every, lags)
    if key not in _WINDOW_REFS:
        sh = np.random.default_rng(7).permutation(T["pos0"].shape[0])
        posC, mask = T[name + "_posC"][:, sh], T[name + "_mask"][:, sh]
        dt = every * RDT / 86400.0
        Cn, NB = len(r_edges) + 1, O.DEFAULT_BINS.size + 1
        out = []
        for w in range((posC.shape[0] - 1) // every):
            k1 = (w + 1) * every
            hist, sums = np.zeros((lags, Cn, NB), np.int64), np.zeros((lags, Cn, 4))
            for l in range(1, min(lags, w + 1) + 1):
                k0 = (w + 1 - l) * every
                args = (posC[k0], posC[k1], mask[k0], mask[k1], pairs)
                hist[l - 1] = O.lag_hist(O.per_pair(*args), l * dt, r_edges)
                sums[l - 1] = O.order_sums(*args, r_edges=r_edges)[0]
            out.append((hist, sums))
        _WINDOW_REFS[key] = out
    return _WINDOW_REFS[key]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["keep", "sink"])
@pytest.mark.parametrize("rows", ["f8", "f4"])
@pytest.mark.parametrize("every,lags", [(1, 1), (1, 64), (7, 3), (48, 4), (49, 2)])
@pytest.mark.parametrize("name", ["uv1", "win"])
def test_track_windows_bits(torch, sit, gold_track, name, every, lags, rows, mode):
    """track(dispersion=...) on the 48 records of a golden case with the buoys sorted on the host: lags = 1 (one ring
    slot, reused at every window), every = 1 with 64 lags (48 slots; lags past the window count stay zero), every = 7
    (a trailing partial window dropped), 48 (one window) and 49 (no window: an empty list, and the sink is never
    called); every window's sums bit for bit against order_sums, its counts against lag_hist."""
    T, g = gold_track
    assert T["U"].shape[0] == 48
    n = T["pos0"].shape[0]
    a, b = np.triu_indices(n, 1)
    pairs = np.stack([a, b], 1).astype(np.int32)[::3]
    r_edges = [1.0, 3.0, 10.0]
    ref = _window_refs(T, name, every, lags, pairs, r_edges)
    assert len(ref) == 48 // every
    seen = []
    spec = dict(pairs=pairs, every=every, lags=lags, r_edges=r_edges)
    if mode == "sink":
        spec["sink"] = lambda w, st: seen.append((w, st))
    res, _ = _engine(T, g, name, "host", rows, spec)
    if mode == "keep":
        got = res["dispersion"]
        assert seen == [] and isinstance(got, list)
    else:
        assert "dispersion" not in res and [w for w, _ in seen] == list(range(len(ref)))
        got = [st for _, st in seen]
    assert len(got) == len(ref)
    for w, (st, (hist, sums)) in enumerate(zip(got, ref)):
        assert np.array_equal(st["hist_stretch"], hist) and np.array_equal(st["n"], hist.sum(-1)), w
        for q, k in enumerate(("sum_r0", "sum_dr", "sum_dr2", "sum_dD2")):
            assert _same_bits(st[k], sums[..., q]).all(), (w, k)
        assert not st["hist_stretch"][w + 1:].any() and not st["sum_r0"][w + 1:].view(np.uint64).any()
    n = sum(int(st["n"].sum()) for st in got)
    if (name, every) == ("win", 48):
        assert n == 0                                 # no buoy of the win case is alive at both row 0 and row 48
    elif ref:
        assert n > 100
