"""The deformation kernels (csrc/st_deform.cu, csrc/st_deform_scale.cu) pinned to their references
(oracle/deform_ref.py, oracle/deform_scale_ref.py) where a kernel could be subtly wrong and still round to the same f4.

The fixed summation order of the box sums is the contract that keeps the statistics identical run to run, on every
device and in every buoy storage order, so the f8 box records are compared bit for bit at every level (read from the
front of the pass's scratch).  Then the edges: values equal to a histogram edge, box areas equal to the cover
threshold, each validity clause alone, triangles with infinite area and NaN rates, 1 and 4096 edges, 20 levels on a
mesh large enough that every grid-strided loop runs more than once, one box holding 717 k triangles, k_deform around
its block size, and track()'s windows at every = 1, nrec and nrec + 1.

CPU: the sliced level-1 reference against the full call, the premises of the validity cases, and the argument checks
of st_deform_scales_scratch_bytes.  GPU: everything else."""
import ctypes as C

import numpy as np
import pytest

from conftest import engine_for
from test_deformation_scales import FILL, RDT, _check_stats, _lattice


def _same_bits(a, b):
    """Element-wise: the same bit pattern, or both NaN.  -0.0 and +0.0 differ."""
    a, b = np.asarray(a), np.asarray(b)
    assert a.dtype == b.dtype and a.shape == b.shape, (a.dtype, b.dtype, a.shape, b.shape)
    u = {4: np.uint32, 8: np.uint64}[a.dtype.itemsize]
    return (a.view(u) == b.view(u)) | (np.isnan(a) & np.isnan(b))


def _sliced_level1(chunk):
    """deform_scale_ref.level1_sums taken `chunk` boxes at a time: the full call holds nbox x 32 x 7 doubles at once
    (640 MB for the 600 x 600 lattice)."""
    from oracle import deform_scale_ref as O
    full = O.level1_sums

    def level1_sums(Ts, off, boxes=None):
        b = np.arange(off.size - 1) if boxes is None else np.asarray(boxes)
        return np.concatenate([full(Ts, off, boxes=b[a:a + chunk]) for a in range(0, b.size, chunk)])
    return level1_sums


def _oracle(yx0, yx1, m0, m1, dt, H, monkeypatch=None, chunk=None):
    """deform_scale_ref.coarse_grain on the mesh, levels, cover and edges of the BoxHierarchy H (whose hierarchy the
    oracle rebuilds and must agree with); with `chunk`, its level-1 sums are taken in slices."""
    from oracle import deform_scale_ref as O
    G = O.hierarchy(yx0, H.tri, H.L0_km, H.levels)
    assert np.array_equal(G["order"], H.order)
    for s in range(H.levels):
        assert np.array_equal(G["levels"][s]["off"], H.box_tri_off[s])
    if chunk is not None:
        monkeypatch.setattr(O, "level1_sums", _sliced_level1(chunk))
    try:
        return O.coarse_grain(yx0, yx1, m0, m1, H.tri, dt, G, cover=H.cover, edges=H.bin_edges, L0=H.L0_km)
    finally:
        if chunk is not None:
            monkeypatch.undo()


def _device_pass(torch, H, yx0, yx1, m0, m1, dt):
    """The pass as CoarseGrainedRates launches it, plus the f8 box records from the front of its scratch
    (8 x nbox_all doubles, level 1 first: a2, Nux, Nuy, Nvx, Nvy, NY, NX and a pad word that is never written).
    -> (per level (nbox,7) f8 sums, per level dict of f4 BOX_NAMES planes, moments (S,4), hist (S,3,nedge+1))."""
    from sitrack_b200 import deform_scales as DS
    dev = torch.device("cuda", 0)
    with torch.cuda.device(dev):
        t = lambda a, d: torch.from_numpy(np.ascontiguousarray(a, d)).to(dev)
        plan = DS._DevicePlan(torch, dev, H, H.tri)
        mom, hist = plan.outputs()
        nall = int(H.nbox.sum())
        out = torch.empty((7, nall), dtype=torch.float32, device=dev)
        plan.launch(None, t(yx0, np.float64), t(m0, np.int8), t(yx1, np.float64), t(m1, np.int8), dt, mom, hist, out,
                    torch.cuda.current_stream(dev))
        torch.cuda.synchronize(dev)
        rec = plan.scratch[:8 * nall].cpu().numpy().reshape(nall, 8)[:, :7]
        out, mom, hist = out.cpu().numpy(), mom.cpu().numpy(), hist.cpu().numpy()
    b0 = np.r_[0, np.cumsum(H.nbox)]
    S = [rec[b0[s]:b0[s + 1]] for s in range(H.levels)]
    planes = [{k: out[j, b0[s]:b0[s + 1]] for j, k in enumerate(DS.BOX_NAMES)} for s in range(H.levels)]
    return S, planes, mom, hist


def _check_pass(torch, H, yx0, yx1, m0, m1, dt, monkeypatch=None, chunk=None):
    """The pass against the oracle: f8 box sums bit for bit at every level, f4 box planes bit for bit, histograms and
    n exactly, moment sums within 1e-11 where the oracle's are finite and non-finite alike (NaN with NaN, inf with
    the same inf) where they are not.  -> (oracle boxes, oracle stats, device planes, device hist)."""
    from oracle import deform_scale_ref as O
    rb, rs = _oracle(yx0, yx1, m0, m1, dt, H, monkeypatch, chunk)
    S, planes, mom, hist = _device_pass(torch, H, yx0, yx1, m0, m1, dt)
    for s in range(H.levels):
        same = _same_bits(S[s], rb[s]["S"])
        assert same.all(), "level %d: %d of %d box sums differ" % (s + 1, (~same).any(1).sum(), same.shape[0])
        for k in O.BOX_NAMES:
            assert _same_bits(planes[s][k], rb[s][k]).all(), (s + 1, k)
    assert np.array_equal(hist, rs["hist"])
    assert np.array_equal(hist[:, 0].sum(1), rs["n"])
    ref = rs["sums"]
    fin = np.isfinite(ref)
    assert (np.abs(mom[fin] - ref[fin]) <= 1e-11 * np.abs(ref[fin])).all()
    assert ((np.isnan(mom) & np.isnan(ref)) | (mom == ref))[~fin].all(), (mom[~fin], ref[~fin])
    return rb, rs, planes, hist


def _drift(yx0, seed, jumps=0, masked=0.0):
    """Smooth drift plus `jumps` vertices moved across their neighbours (flipped triangles), and masks with about
    `masked` of the buoys set to 0 in each row."""
    rng = np.random.default_rng(seed)
    nP = yx0.shape[0]
    yx1 = yx0 + 1.2 + np.stack([np.sin(yx0[:, 1] / 40.0), np.cos(yx0[:, 0] / 55.0)], 1) * 0.7
    if jumps:
        j = rng.choice(nP, jumps, replace=False)
        yx1[j] += rng.choice([-1.0, 1.0], (jumps, 2)) * 7.0
    return yx1, (rng.random(nP) >= masked).astype(np.int8), (rng.random(nP) >= masked).astype(np.int8)


# ---- the validity cases -------------------------------------------------------------------------

def _tri_at(c, r=1.0, rot=0.3):
    """[y,x] of an anticlockwise triangle (nearly equilateral) of radius r around c."""
    ang = rot + np.array([0.0, 2.1, 4.2])
    return np.stack([c[0] + r * np.sin(ang), c[1] + r * np.cos(ang)], 1)


def _validity_case():
    """One triangle per special case, each on its own three buoys, in its own 10 km box with an ordinary companion:
    -> (yx0, yx1, m0, m1, tri, dt, {name: triangle index})."""
    dt = 0.25
    rng = np.random.default_rng(21)
    P0, P1, K0, K1, idx = [], [], [], [], {}

    def add(name, p0, p1, k0=(1, 1, 1), k1=(1, 1, 1)):
        idx[name] = len(P0)
        P0.append(p0); P1.append(p1); K0.append(k0); K1.append(k1)

    good = lambda p: p + rng.normal(0.0, 0.05, p.shape)
    specials = ["rot180", "collinear_k0", "collinear_k1"] + ["mask%d_v%d" % (r, v) for r in (0, 1) for v in range(3)] + \
               ["huge"]
    for i, name in enumerate(specials):
        xc = 5.0 + 10.0 * i
        p = _tri_at((4.0, xc))
        if name == "rot180":                      # 180 degrees about the origin: anticlockwise at both ends, mid 0
            add(name, p, -p)
        elif name in ("collinear_k0", "collinear_k1"):
            line = np.array([[3.0, xc - 1], [4.0, xc], [5.0, xc + 1]])     # integers on a line: twice_area exactly 0
            bent = line + np.array([[0.0, 0.0], [0.0, 0.0], [1.0, -1.0]])  # the last vertex moved to its left
            add(name, *((line, bent) if name == "collinear_k0" else (bent, line)))
        elif name.startswith("mask"):
            k = [[1, 1, 1], [1, 1, 1]]
            k[int(name[4])][int(name[-1])] = 0
            add(name, p, good(p), tuple(k[0]), tuple(k[1]))
        else:                                     # f8 area +inf at k1 and mid-time, rates NaN, mask 1
            add(name, p, np.array([[0.0, 0.0], [0.0, 1e200], [1e200, 0.0]]))
        q = _tri_at((7.5, xc), rot=1.0)
        add(name + "_companion", q, good(q))
    yx0, yx1 = np.concatenate(P0), np.concatenate(P1)
    m0, m1 = np.array(K0, np.int8).ravel(), np.array(K1, np.int8).ravel()
    tri = np.arange(yx0.shape[0], dtype=np.int32).reshape(-1, 3)
    return yx0, yx1, m0, m1, tri, dt, idx


def _assert_validity_premises(yx0, yx1, m0, m1, tri, dt, idx):
    """Each special triangle is invalid by exactly the clause it is built for (or, 'huge', valid with an infinite
    area and non-finite rates), by the oracle's own arithmetic."""
    from oracle import deform_ref as R
    with np.errstate(all="ignore"):
        r, valid = R.rates_f8(yx0, yx1, m0, m1, tri, dt)
        a0 = R.twice_area(yx0[tri, 1], yx0[tri, 0])
        a1 = R.twice_area(yx1[tri, 1], yx1[tri, 0])
    masks = (m0[tri] != 0).all(1) & (m1[tri] != 0).all(1)
    for name, i in idx.items():
        if name.endswith("_companion"):
            assert valid[i] and np.isfinite(r["area"][i]), name
        elif name == "rot180":
            assert masks[i] and a0[i] > 0 and a1[i] > 0 and r["area"][i] == 0.0 and not valid[i]
        elif name == "collinear_k0":
            assert masks[i] and a0[i] == 0.0 and a1[i] > 0 and r["area"][i] > 0 and not valid[i]
        elif name == "collinear_k1":
            assert masks[i] and a0[i] > 0 and a1[i] == 0.0 and r["area"][i] > 0 and not valid[i]
        elif name.startswith("mask"):
            assert (m0[tri[i]] == 0).sum() + (m1[tri[i]] == 0).sum() == 1
            assert a0[i] > 0 and a1[i] > 0 and r["area"][i] > 0 and not masks[i] and not valid[i]
        else:
            assert valid[i] and r["area"][i] == np.inf and a1[i] == np.inf
            assert not np.isfinite([r[k][i] for k in ("ux", "uy", "vx", "vy", "divergence", "shear")]).any()


# ---- CPU ----------------------------------------------------------------------------------------

@pytest.mark.parametrize("chunk", [1, 5, 64, 10 ** 6])
def test_oracle_sliced_level1_sums_equal_full_call(monkeypatch, chunk):
    """The sliced level-1 reference used on the large meshes gives the full call's bits, alone and inside
    coarse_grain, on boxes of varied sizes with masks and flips."""
    from oracle import deform_scale_ref as O
    yx0, tri = _lattice(40, hole=(60.0, 60.0, 12.0))
    yx1, m0, m1 = _drift(yx0, 3, jumps=40, masked=0.03)
    G = O.hierarchy(yx0, tri, 13.0, 4)
    T, _, _ = O.triangle_terms(yx0, yx1, m0, m1, tri, 0.25)
    Ts = T[G["order"]]
    off = G["levels"][0]["off"]
    assert np.diff(off).max() > 32                                    # boxes span more than one lane round
    full = O.level1_sums(Ts, off)
    assert _same_bits(_sliced_level1(chunk)(Ts, off), full).all()
    assert _same_bits(_sliced_level1(chunk)(Ts, off, boxes=np.arange(3, off.size - 1, 2)), full[3::2]).all()
    ref = O.coarse_grain(yx0, yx1, m0, m1, tri, 0.25, G, L0=13.0)
    monkeypatch.setattr(O, "level1_sums", _sliced_level1(chunk))
    got = O.coarse_grain(yx0, yx1, m0, m1, tri, 0.25, G, L0=13.0)
    for a, b in zip(got[0], ref[0]):
        assert _same_bits(a["S"], b["S"]).all()
    for k in ("n", "sums", "hist"):
        assert np.array_equal(got[1][k], ref[1][k])


def test_oracle_validity_case_premises():
    _assert_validity_premises(*_validity_case())


def _scratch_bytes(nT, levels, nbox, min_area, nedge):
    from sitrack_b200 import _lib
    nb = np.zeros(21, np.int64); nb[:len(nbox)] = nbox
    ma = np.ones(21, np.float64); ma[:len(min_area)] = min_area
    out = C.c_int64(-1)
    rc = _lib.lib().st_deform_scales_scratch_bytes(nT, levels, nb.ctypes.data, ma.ctypes.data, nedge, C.byref(out))
    return rc, out.value


def test_scratch_bytes_accepts_a_valid_plan():
    rc, b = _scratch_bytes(5000, 3, [1000, 300, 80], [0.5, 2.0, 8.0], 61)
    assert rc == 0 and b >= 8 * (8 * 1380 + 4 * 4)               # box records in front, moment partials per scale
    rc, b = _scratch_bytes(2 ** 31 - 1, 20, [1] * 20, [1.0] * 20, 4096)
    assert rc == 0 and b >= 8 * (8 * 20 + 4 * 21)


@pytest.mark.parametrize("case", [
    dict(levels=0), dict(levels=21), dict(nedge=0), dict(nedge=4097), dict(nT=0), dict(nT=2 ** 31),
    dict(nbox=[300, 1000, 80]), dict(nbox=[1000, 300, 301]), dict(nbox=[6000, 300, 80]),
    dict(min_area=[0.5, 0.0, 8.0]), dict(min_area=[0.5, 2.0, -1.0]), dict(min_area=[np.nan, 2.0, 8.0])],
    ids=lambda c: "-".join("%s=%s" % kv for kv in c.items()))
def test_scratch_bytes_rejects(case):
    """st_deform_scales_scratch_bytes returns ST_EINVAL (-1) and leaves the output alone for each bad argument."""
    a = dict(nT=5000, levels=3, nbox=[1000, 300, 80], min_area=[0.5, 2.0, 8.0], nedge=61)
    a.update(case)
    rc, b = _scratch_bytes(a["nT"], a["levels"], a["nbox"], a["min_area"], a["nedge"])
    assert rc == -1 and b == -1


# ---- GPU: f8 box sums, bit for bit ----------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("name", ["uv1", "uv0", "fast", "win"])
def test_box_sums_bits_golden(torch, sit, gold_track, name):
    """The inputs of test_coarse_grained_vs_oracle_golden: golden rows, Delaunay mesh, L0 = 20 km, 5 levels."""
    T, _ = gold_track
    posC, mask = T[name + "_posC"], T[name + "_mask"]
    tri = sit.TriangulateCloud(T["pos0"])
    for k0, k1 in [(0, 6), (5, 29), (12, 48)]:
        H = sit.BoxHierarchy(posC[k0], tri, 20.0, 5)
        _check_pass(torch, H, posC[k0], posC[k1], mask[k0], mask[k1], (k1 - k0) * RDT / 86400.0)


@pytest.mark.gpu
def test_box_sums_bits_lattice(torch, sit):
    """The inputs of test_coarse_grained_vs_oracle_lattice: ~200 k buoys, 2 % masked, 300 flipping vertices, a hole;
    L0 = 12 km, 6 levels."""
    rng = np.random.default_rng(11)
    yx0, tri = _lattice(450, hole=(600.0, 700.0, 90.0), seed=3)
    nP = yx0.shape[0]
    yx1 = yx0 + 1.2 + np.stack([np.sin(yx0[:, 1] / 40.0), np.cos(yx0[:, 0] / 55.0)], 1) * 0.7
    jump = rng.choice(nP, 300, replace=False)
    yx1[jump] += rng.choice([-1.0, 1.0], (300, 2)) * 7.0
    m0 = (rng.random(nP) >= 0.02).astype(np.int8)
    m1 = (rng.random(nP) >= 0.02).astype(np.int8)
    H = sit.BoxHierarchy(yx0, tri, 12.0, 6)
    rb, _, _, _ = _check_pass(torch, H, yx0, yx1, m0, m1, 0.25)
    assert np.diff(H.tri_off).max() == 32 and (~rb[0]["valid"]).any() and rb[0]["valid"].sum() > 1000


@pytest.mark.gpu
@pytest.mark.parametrize("cover", [0.5, 1e-4])
def test_box_sums_bits_box_sizes(torch, sit, cover):
    """The inputs of test_coarse_grained_vs_oracle_box_sizes: level-1 boxes of 1, 31, 32, 33, 64, 65 and 417
    triangles, 4 levels up to a single box."""
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
    tri = tri[rng.permutation(tri.shape[0])]
    yx1 = yx0 + rng.normal(0, 0.01, yx0.shape)
    one = np.ones(yx0.shape[0], np.int8)
    H = sit.BoxHierarchy(yx0, tri, 10.0, 4, cover=cover)
    assert sorted(np.diff(H.tri_off).tolist()) == sorted(sizes) and H.nbox[-1] == 1
    _check_pass(torch, H, yx0, yx1, one, one, 0.25)


# ---- GPU: exact ties ------------------------------------------------------------------------------

def _counted_values(yx0, yx1, m0, m1, tri, dt, H):
    """The f8 eps_tot, |D| and shear of every cell that counts, per scale (the oracle's values)."""
    from oracle import deform_scale_ref as O
    from oracle import deform_ref as R
    r, valid = R.rates_f8(yx0, yx1, m0, m1, tri, dt)
    with np.errstate(all="ignore"):
        o0 = O.rates_of(r["ux"], r["uy"], r["vx"], r["vy"])
    vals = [np.concatenate([o0["total"][valid], np.abs(o0["divergence"][valid]), o0["shear"][valid]])]
    rb, _ = _oracle(yx0, yx1, m0, m1, dt, H)
    for b in rb:
        o, _ = O.box_outputs(b["S"], 0.0)
        ok = b["valid"]
        vals.append(np.concatenate([o["total"][ok], np.abs(o["divergence"][ok]), o["shear"][ok]]))
    return vals


@pytest.mark.gpu
@pytest.mark.parametrize("nedge", [4096, 1])
def test_bin_edge_ties(torch, sit, nedge):
    """Edges that are values the oracle counts, at scale 0 and at every level, including the smallest and the largest
    (4096 edges: 81 932 B of shared memory, above the 48 KB default), and a single edge: every count equals the
    oracle's searchsorted(side="right"), so a value equal to an edge goes to the bin above it."""
    yx0, tri = _lattice(120, hole=(180.0, 200.0, 30.0), seed=4)
    yx1, m0, m1 = _drift(yx0, 5, jumps=60, masked=0.02)
    dt = 0.25
    H0 = sit.BoxHierarchy(yx0, tri, 12.0, 5)
    vals = _counted_values(yx0, yx1, m0, m1, tri, dt, H0)
    rng = np.random.default_rng(6)
    if nedge == 1:
        e = np.array([np.median(vals[1])])
    else:
        allv = np.unique(np.concatenate(vals))
        lo, hi = allv[0], allv[-1]                                  # both extremes
        box = np.unique(np.concatenate(vals[2:]))                   # every value of levels 2..5, some of level 1
        box = np.union1d(box, rng.choice(np.unique(vals[1]), 600, replace=False))
        box = np.setdiff1d(box, [lo, hi])
        rest = np.setdiff1d(allv, np.r_[box, lo, hi])
        e = np.unique(np.concatenate([[lo, hi], box, rng.choice(rest, nedge - 2 - box.size, replace=False)]))
    assert e.size == nedge and np.isfinite(e).all()
    H = sit.BoxHierarchy(yx0, tri, 12.0, 5, bins=e)
    ties = [int(np.isin(v, e).sum()) for v in vals]
    if nedge > 1:                                                   # premise: ties at scale 0 and at every level
        assert all(t > 0 for t in ties) and sum(ties) > 4000 and ties[1] > 500, ties
    else:
        assert ties[1] > 0, ties
    _, rs, _, hist = _check_pass(torch, H, yx0, yx1, m0, m1, dt)
    assert hist[:, :, -1].sum() > 0
    assert rs["n"][0] > 20000 and (rs["n"] > 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("level", [1, 3])
def test_cover_ties(torch, sit, level):
    """L0 = 1 km, so cover * L * L is exact: with cover * L^2 equal to the oracle's f8 area of a chosen box, that box
    counts; with the next f8 cover up, it does not."""
    yx0, tri = _lattice(41, d=0.25, jitter=0.05, seed=7)
    yx1, m0, m1 = _drift(yx0, 8)
    dt = 0.25
    H = sit.BoxHierarchy(yx0, tri, 1.0, 4)
    rb, _ = _oracle(yx0, yx1, m0, m1, dt, H)
    s = level - 1
    area = 0.5 * rb[s]["S"][:, 0]
    k = int(np.argsort(area)[area.size // 2])                       # a box of median area
    scale = 4.0 ** s                                                # L_s^2 with L0 = 1 km
    for cover, counts in ((area[k] / scale, True), (np.nextafter(area[k] / scale, np.inf), False)):
        Hc = sit.BoxHierarchy(yx0, tri, 1.0, 4, cover=cover)
        assert Hc.min_area[s] == (area[k] if counts else np.nextafter(area[k], np.inf))
        rbc, _, planes, _ = _check_pass(torch, Hc, yx0, yx1, m0, m1, dt)
        assert rbc[s]["valid"][k] == counts
        assert (planes[s]["total"][k] != FILL) == counts
        assert 0 < rbc[s]["valid"].sum() < rbc[s]["valid"].size


# ---- GPU: validity and non-finite values ----------------------------------------------------------

@pytest.mark.gpu
def test_validity_clauses_and_nonfinite(torch, sit):
    """A triangle rotated by 180 degrees about the origin (mid-time area exactly 0), triangles exactly collinear at k0
    only and at k1 only, each of the six mask bytes alone, and a triangle whose f8 area is +inf with NaN rates:
    k_deform's fill values and the pass's scale-0 counts and box sums against the oracle; the NaN rates go to the
    overflow bin at every scale, and the moment sums are non-finite on both sides."""
    from oracle import deform_ref as R
    yx0, yx1, m0, m1, tri, dt, idx = _validity_case()
    _assert_validity_premises(yx0, yx1, m0, m1, tri, dt, idx)
    got = sit.DeformationRates(yx0, yx1, m0, m1, tri, dt)
    ref = R.deform(yx0, yx1, m0, m1, tri, dt)
    for k in R.NAMES:
        assert _same_bits(got[k], ref[k]).all(), k
    for name, i in idx.items():
        filled = got["divergence"][i] == FILL
        assert filled == (not name.endswith("_companion") and name != "huge"), name
    h = idx["huge"]
    assert got["area"][h] == np.inf and np.isnan(got["divergence"][h])
    H = sit.BoxHierarchy(yx0, tri, 10.0, 4, cover=1e-3)
    _, rs, planes, hist = _check_pass(torch, H, yx0, yx1, m0, m1, dt)
    assert rs["n"][0] == 11 and hist[0, 0, -1] >= 1                 # the companions and 'huge' (NaN: overflow)
    assert (hist[:, 0, -1] >= 1).all() and np.isnan(planes[0]["total"]).sum() == 1
    assert not np.isfinite(rs["sums"][:, 1]).any()


# ---- GPU: shapes ----------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def big_lattice():
    """A jittered 600 x 600 lattice at 3 km (717 602 triangles) with drift, flips and 1 % masks."""
    yx0, tri = _lattice(600, d=3.0, seed=9)
    yx1, m0, m1 = _drift(yx0, 10, jumps=500, masked=0.01)
    return yx0, yx1, m0, m1, tri


@pytest.mark.gpu
def test_levels20_grid_strided(torch, sit, monkeypatch, big_lattice):
    """20 levels with L0 = the lattice spacing: 358 801 level-1 boxes, more than the 1184 x 256 threads of
    k_scale_stats and the 1184 x 8 warps of k_scale_l1, so both grid-stride; the top levels are single boxes."""
    yx0, yx1, m0, m1, tri = big_lattice
    H = sit.BoxHierarchy(yx0, tri, 3.0, 20)
    assert tri.shape[0] == 717602 and H.nbox[0] == 358801 and H.nbox[0] > 1184 * 256
    assert H.nbox[-1] == 1 and (H.nbox == 1).sum() >= 5
    _, rs, _, _ = _check_pass(torch, H, yx0, yx1, m0, m1, 0.25, monkeypatch, chunk=40000)
    assert (rs["n"][:11] > 0).all() and (rs["n"][11:] == 0).all()     # the single boxes above are below cover


@pytest.mark.gpu
def test_single_box_whole_mesh(torch, sit, monkeypatch, big_lattice):
    """One level-1 box holding all 717 602 triangles (22 426 per lane), levels = 1."""
    yx0, yx1, m0, m1, tri = big_lattice
    H = sit.BoxHierarchy(yx0, tri, 2048.0, 1, cover=0.1)
    assert H.nbox.tolist() == [1]
    rb, rs, _, _ = _check_pass(torch, H, yx0, yx1, m0, m1, 0.25, monkeypatch, chunk=1)
    assert rb[0]["valid"][0] and rs["n"][1] == 1


@pytest.mark.gpu
@pytest.mark.parametrize("nT", [1, 255, 256, 257, 512])
def test_triangle_counts_around_the_block(torch, sit, nT):
    """k_deform with a single partial block, exactly one block, one plus one triangle, and two full blocks; the pass
    on the same triangles."""
    from oracle import deform_ref as R
    yx0, tri = _lattice(20, seed=13)
    yx1, m0, m1 = _drift(yx0, 14, jumps=12, masked=0.03)
    tri = tri[np.random.default_rng(15).permutation(tri.shape[0])[:nT]]
    dt = 0.25
    got = sit.DeformationRates(yx0, yx1, m0, m1, tri, dt)
    ref = R.deform(yx0, yx1, m0, m1, tri, dt)
    for k in R.NAMES:
        assert got[k].shape == (nT,) and _same_bits(got[k], ref[k]).all(), k
    if nT > 1:
        assert (ref["divergence"] == FILL).any() and (ref["divergence"] != FILL).any()
    H = sit.BoxHierarchy(yx0, tri, 6.0, 3, cover=1e-3)
    _check_pass(torch, H, yx0, yx1, m0, m1, dt)


# ---- GPU: engine windows --------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["keep", "sink"])
@pytest.mark.parametrize("every", [1, 48, 49])
def test_track_windows(torch, sit, gold_track, every, mode):
    """track(deform=dict(tri=, every=, scales=H)) on the 48 records of the uv1 case: every = 1 (48 windows, the
    two-deep output ring reused on every record), 48 (one window) and 49 (none: empty lists, no sink call), with
    the rows kept or handed to a sink; each window equals deform_series / coarse_grain_series."""
    from oracle import deform_ref as R
    from oracle import deform_scale_ref as O
    T, g = gold_track
    posC, mask = T["uv1_posC"], T["uv1_mask"]
    nrec = T["U"].shape[0]
    assert nrec == 48
    tri = sit.TriangulateCloud(T["pos0"])
    H = sit.BoxHierarchy(T["pos0"], tri, 20.0, 5)
    ref = R.deform_series(posC, mask, tri, every, RDT)
    refs = O.coarse_grain_series(posC, mask, tri, every, RDT, O.hierarchy(T["pos0"], tri, 20.0, 5), L0=20.0,
                                 edges=H.bin_edges)
    assert len(ref) == len(refs) == nrec // every
    eng = engine_for(g, device=0)
    eng.set_buoys(T["pos0"], T["jiT0"].astype(np.int32))
    spec = dict(tri=tri, every=every, scales=H)
    if mode == "keep":
        res = eng.track((T["U"], T["V"], T["IC"]), nrec, pos0=T["pos0"], deform=spec)
        assert np.array_equal(res["posC"], posC) and np.array_equal(res["mask"], mask)
        dfm, scl = res["deform"], res["deform_scales"]
    else:
        rows, dseen, sseen = [], [], []
        spec.update(sink=lambda w, o: dseen.append((w, {k: v.copy() for k, v in o.items()})),
                    scale_sink=lambda w, st: sseen.append((w, st)))
        res = eng.track((T["U"], T["V"], T["IC"]), nrec, sink=lambda k, *a: rows.append(k), deform=spec)
        assert rows == list(range(nrec)) and "deform" not in res and "deform_scales" not in res
        assert [w for w, _ in dseen] == [w for w, _ in sseen] == list(range(len(ref)))
        dfm, scl = [o for _, o in dseen], [s for _, s in sseen]
    eng.close()
    assert len(dfm) == len(scl) == len(ref)
    for w, (a, b) in enumerate(zip(dfm, ref)):
        for k in R.NAMES:
            assert np.array_equal(a[k], b[k]), (w, k)
    for a, b in zip(scl, refs):
        _check_stats(a, b, H)
    if ref:
        assert sum(int((b["divergence"] != FILL).sum()) for b in ref) > 50


# ---- GPU: entry points refuse bad dt and nT ---------------------------------------------------------

@pytest.mark.gpu
def test_entry_points_refuse_bad_dt_and_nT(torch, sit):
    """st_deform_dev and st_deform_scales_dev, given real, aligned device buffers, return ST_EINVAL for dt_days <= 0
    (and NaN) and nT < 0, and write nothing; the same buffers with dt_days > 0 are accepted."""
    from sitrack_b200 import _lib
    from sitrack_b200 import deform_scales as DS
    L = _lib.lib()
    dev = torch.device("cuda", 0)
    yx0, tri = _lattice(8)
    yx1, m0, m1 = _drift(yx0, 16)
    H = sit.BoxHierarchy(yx0, tri, 6.0, 2)
    t = lambda a, d: torch.from_numpy(np.ascontiguousarray(a, d)).to(dev)
    with torch.cuda.device(dev):
        st = torch.cuda.current_stream(dev)
        tri_t, a_t, b_t = t(tri, np.int32), t(yx0, np.float64), t(yx1, np.float64)
        m0_t, m1_t = t(m0, np.int8), t(m1, np.int8)
        nT = tri.shape[0]
        out = torch.full((6, nT), 7.0, dtype=torch.float32, device=dev)
        plan = DS._DevicePlan(torch, dev, H, H.tri)
        mom, hist = plan.outputs()
        mom.fill_(7.0); hist.fill_(7)
        p = lambda x: C.c_void_p(x.data_ptr())
        for n, dt in [(nT, 0.0), (nT, -0.25), (nT, -0.0), (nT, float("nan")), (-1, 0.25)]:
            assert L.st_deform_dev(None, n, p(tri_t), p(a_t), p(m0_t), p(b_t), p(m1_t), dt, p(out),
                                   C.c_void_p(st.cuda_stream)) == -1, (n, dt)
            assert L.st_deform_scales_dev(
                None, n, p(plan.tri_t), p(a_t), p(m0_t), p(b_t), p(m1_t), dt, H.levels, plan.nbox.ctypes.data,
                plan.min_area.ctypes.data, p(plan.tri_off_t), p(plan.child_t), H.bin_edges.size, p(plan.edges_t),
                p(plan.scratch), plan.scratch_bytes, p(mom), p(hist), None, C.c_void_p(st.cuda_stream)) == -1, (n, dt)
        torch.cuda.synchronize(dev)
        assert (out == 7.0).all().item() and (mom == 7.0).all().item() and (hist == 7).all().item()
        assert L.st_deform_dev(None, nT, p(tri_t), p(a_t), p(m0_t), p(b_t), p(m1_t), 0.25, p(out),
                               C.c_void_p(st.cuda_stream)) == 0
        plan.launch(None, a_t, m0_t, b_t, m1_t, 0.25, mom, hist, None, st)
        torch.cuda.synchronize(dev)
        assert (out != 7.0).any().item() and hist[0, 0].sum().item() > 0 and not (hist == 7).all().item()
