"""Reference of the sampling of SI3 T-cell fields along buoy trajectories (DESIGN.md section 15, csrc/st_sample.cu).

Rows and records.  Row r of the trajectory is the one the reference writes at vTime[r].  Row 0 is sampled with record
kstrt, the record SeedInit uses for Survive; row k+1 (k >= 0) with record kstrt + k, the record whose velocities moved
the buoy there (and whose siconc the reference tests when the buoy enters that cell).  With every = n the sampled rows
are 0, n, 2n, ..., floor(Nt/n) n.

Position and cell.  The buoy's f8 [y, x] and its host cell (jT, iT) at that row: the cell the step leaves in the state,
bit 31 (discontinued) stripped.

Validity.  A buoy whose row mask is 0 gets FillValue (-9999) in every field, and so does a cell outside
1 <= jT <= Nj-2, 1 <= iT <= Ni-2 (only a seed that set_buoys discontinued can carry one; see DESIGN.md section 15 for
why no step leaves a masked-1 row there).

interp = "cell": F[jT, iT], the SI3 T-cell value of the host cell (the host cell is the T-cell: F-point corners), an
exact f4 copy; a non-finite value gives FillValue.

interp = "bilinear", in f8, no FMA, in this order:
  1. The T-quad.  With C = T[jT,iT], S = T[jT-1,iT], N = T[jT+1,iT], W = T[jT,iT-1], E = T[jT,iT+1] and
     orient(A, B, P) = (B.x - A.x)(P.y - A.y) - (B.y - A.y)(P.x - A.x):
       i0 = iT - 1 when orient(S, N, P) > 0 (P west of S->N), else iT;
       j0 = jT - 1 when orient(W, E, P) < 0 (P south of W->E), else jT.
     A point on a line (orient = 0) goes to the quad of the higher index.  The grid is right-handed:
     cross(T[j,i+1] - T[j,i], T[j+1,i] - T[j,i]) > 0 (i eastward, j northward in the projected plane, as the step's
     anticlockwise F-cells are); sitrack_b200.sample.tpoints refuses T-points for which that fails on most quads.  Corners a, b, c, d = T[j0,i0], T[j0,i0+1],
     T[j0+1,i0+1], T[j0+1,i0] (SW, SE, NE, NW).
  2. Inverse bilinear (xi, eta) of P: e = b - a, f = d - a, g = ((a - b) + c) - d, h = P - a, cross(u, v) = u.x v.y -
     u.y v.x, k2 = cross(g, f), k1 = cross(e, f) + cross(h, g), k0 = cross(h, e).
       k2 == 0 (a parallelogram):  eta = -k0 / k1;
       otherwise:  disc = k1 k1 - (4 k0) k2, 0 when negative;  q = -0.5 (k1 + copysign(sqrt(disc), k1));  eta = k0 / q
     (the root of k2 eta^2 + k1 eta + k0 = 0 that tends to the parallelogram's as k2 -> 0, without cancellation).
     dx = e.x + g.x eta, dy = e.y + g.y eta;  xi = (h.x - f.x eta) / dx when |dx| >= |dy|, else (h.y - f.y eta) / dy.
     Each is clamped: v > 0 ? (v < 1 ? v : 1) : 0, so a NaN becomes 0.
  3. Weights (1-xi)(1-eta), xi(1-eta), xi eta, (1-xi) eta of SW, SE, NE, NW.  Per field, in that order from
     num = den = +0: a corner with tmask != 0 and a finite value v (f4 widened exactly) adds w v to num and w to den.
  4. den > 0: num / den; otherwise the cell value.
  5. Rounded once to f4; a non-finite result gives FillValue.

Vectorised over buoys with numpy: every operation is an elementwise IEEE f8 operation in the order above, which numpy
never contracts, so the device matches it bit for bit.
"""
import numpy as np

FillValue = -9999.0
INTERP = {"cell": 0, "bilinear": 1}


def sampled_rows(nrec, every):
    """Rows 0, n, 2n, ..., floor(nrec/n) n."""
    n = int(every)
    return np.arange(0, (nrec // n) * n + 1, n)


def row_record(r, kstrt=0):
    """The record row r is sampled with: kstrt for row 0, kstrt + r - 1 after that."""
    return kstrt + max(int(r) - 1, 0)


def quad(yx, jT, iT, Yt, Xt):
    """-> (j0, i0) of the T-quad of P = yx (n,2) in the cells (jT, iT) (step 1)."""
    Py, Px = yx[:, 0], yx[:, 1]

    def orient(ja, ia, jb, ib):
        Ay, Ax, By, Bx = Yt[ja, ia], Xt[ja, ia], Yt[jb, ib], Xt[jb, ib]
        return (Bx - Ax) * (Py - Ay) - (By - Ay) * (Px - Ax)

    dI = orient(jT - 1, iT, jT + 1, iT)
    dJ = orient(jT, iT - 1, jT, iT + 1)
    return np.where(dJ < 0, jT - 1, jT), np.where(dI > 0, iT - 1, iT)


def _clamp(v):
    return np.where(v > 0, np.where(v < 1, v, 1.0), 0.0)


def inv_bilinear(P, a, b, c, d):
    """(xi, eta) of P (n,2) [y,x] in the quads a, b, c, d (SW, SE, NE, NW; each (n,2)), clamped to [0,1] (step 2)."""
    ex, ey = b[:, 1] - a[:, 1], b[:, 0] - a[:, 0]
    fx, fy = d[:, 1] - a[:, 1], d[:, 0] - a[:, 0]
    gx, gy = ((a[:, 1] - b[:, 1]) + c[:, 1]) - d[:, 1], ((a[:, 0] - b[:, 0]) + c[:, 0]) - d[:, 0]
    hx, hy = P[:, 1] - a[:, 1], P[:, 0] - a[:, 0]
    cross = lambda ux, uy, vx, vy: ux * vy - uy * vx
    k2 = cross(gx, gy, fx, fy)
    k1 = cross(ex, ey, fx, fy) + cross(hx, hy, gx, gy)
    k0 = cross(hx, hy, ex, ey)
    with np.errstate(divide="ignore", invalid="ignore"):
        disc = k1 * k1 - (4.0 * k0) * k2
        disc = np.where(disc < 0, 0.0, disc)
        q = -0.5 * (k1 + np.copysign(np.sqrt(disc), k1))
        eta = np.where(k2 == 0, -k0 / k1, k0 / q)
        dx, dy = ex + gx * eta, ey + gy * eta
        xi = np.where(np.abs(dx) >= np.abs(dy), (hx - fx * eta) / dx, (hy - fy * eta) / dy)
    return _clamp(xi), _clamp(eta)


def sample(fields, tmask, cell, yx, mask, interp="cell", Yt=None, Xt=None):
    """fields (nF,Nj,Ni) f4 of one record, tmask (Nj,Ni), cell (nP,2) host cells (bit 31 is stripped here), yx (nP,2)
    f8 positions, mask (nP,) the row mask -> (nF, nP) f4."""
    F = np.asarray(fields, np.float32)
    if F.ndim == 2:
        F = F[None]
    nF, Nj, Ni = F.shape
    cell = np.asarray(cell, np.int64)
    jT, iT = cell[:, 0] & 0x7fffffff, cell[:, 1]
    ok = (np.asarray(mask) != 0) & (jT >= 1) & (jT <= Nj - 2) & (iT >= 1) & (iT <= Ni - 2)
    out = np.full((nF, cell.shape[0]), FillValue, np.float32)
    idx = np.flatnonzero(ok)
    if idx.size == 0:
        return out
    jT, iT = jT[idx], iT[idx]
    own = F[:, jT, iT].astype(np.float64)
    if INTERP[interp] == 0:
        val = own
    else:
        Yt, Xt = np.asarray(Yt, np.float64), np.asarray(Xt, np.float64)
        P = np.asarray(yx, np.float64)[idx]
        j0, i0 = quad(P, jT, iT, Yt, Xt)
        corners = [(j0, i0), (j0, i0 + 1), (j0 + 1, i0 + 1), (j0 + 1, i0)]
        pts = [np.stack([Yt[j, i], Xt[j, i]], 1) for j, i in corners]
        xi, eta = inv_bilinear(P, *pts)
        w = [(1.0 - xi) * (1.0 - eta), xi * (1.0 - eta), xi * eta, (1.0 - xi) * eta]
        with np.errstate(invalid="ignore", over="ignore"):
            val = _renormalised(F, tmask, corners, w, own, idx.size)
    with np.errstate(over="ignore", invalid="ignore"):
        v4 = val.astype(np.float32)
    out[:, idx] = np.where(np.isfinite(v4), v4, np.float32(FillValue))
    return out


def _renormalised(F, tmask, corners, w, own, n):
    """Step 3 and 4 of every field: the kept corners' weighted sum over their weights, else the cell value."""
    val = np.empty_like(own)
    for f in range(F.shape[0]):
        num = np.zeros(n)
        den = np.zeros(n)
        for (j, i), wk in zip(corners, w):
            v = F[f, j, i].astype(np.float64)
            keep = (tmask[j, i] != 0) & np.isfinite(v)
            num = np.where(keep, num + wk * v, num)
            den = np.where(keep, den + wk, den)
        with np.errstate(divide="ignore", invalid="ignore"):
            val[f] = np.where(den > 0, num / den, own[f])
    return val


def sample_loop(fields, tmask, cell, yx, mask, interp="cell", Yt=None, Xt=None):
    """The same, one buoy and one corner at a time with numpy f8 scalars (IEEE division: x/0 is inf or NaN): the
    per-buoy statement of the definitions that `sample` vectorises."""
    F = np.asarray(fields, np.float32)
    if F.ndim == 2:
        F = F[None]
    nF, Nj, Ni = F.shape
    f8 = np.float64
    out = np.full((nF, len(cell)), FillValue, np.float32)
    with np.errstate(all="ignore"):
        for p in range(len(cell)):
            jT, iT = int(cell[p][0]) & 0x7fffffff, int(cell[p][1])
            if mask[p] == 0 or not (1 <= jT <= Nj - 2 and 1 <= iT <= Ni - 2):
                continue
            if interp == "bilinear":
                T = lambda j, i: (f8(Yt[j, i]), f8(Xt[j, i]))
                py, px = f8(yx[p][0]), f8(yx[p][1])
                orient = lambda A, B: (B[1] - A[1]) * (py - A[0]) - (B[0] - A[0]) * (px - A[1])
                i0 = iT - 1 if orient(T(jT - 1, iT), T(jT + 1, iT)) > 0 else iT
                j0 = jT - 1 if orient(T(jT, iT - 1), T(jT, iT + 1)) < 0 else jT
                cs = [(j0, i0), (j0, i0 + 1), (j0 + 1, i0 + 1), (j0 + 1, i0)]
                a, b, c, d = [T(j, i) for j, i in cs]
                ex, ey, fx, fy = b[1] - a[1], b[0] - a[0], d[1] - a[1], d[0] - a[0]
                gx, gy = ((a[1] - b[1]) + c[1]) - d[1], ((a[0] - b[0]) + c[0]) - d[0]
                hx, hy = px - a[1], py - a[0]
                k2 = gx * fy - gy * fx
                k1 = (ex * fy - ey * fx) + (hx * gy - hy * gx)
                k0 = hx * ey - hy * ex
                if k2 == 0:
                    eta = -k0 / k1
                else:
                    disc = k1 * k1 - (f8(4.0) * k0) * k2
                    if disc < 0:
                        disc = f8(0.0)
                    eta = k0 / (f8(-0.5) * (k1 + np.copysign(np.sqrt(disc), k1)))
                dx, dy = ex + gx * eta, ey + gy * eta
                xi = (hx - fx * eta) / dx if abs(dx) >= abs(dy) else (hy - fy * eta) / dy
                cl = lambda v: (v if v < 1 else f8(1.0)) if v > 0 else f8(0.0)
                xi, eta = cl(xi), cl(eta)
                ws = [(1 - xi) * (1 - eta), xi * (1 - eta), xi * eta, (1 - xi) * eta]
            for f in range(nF):
                v = f8(F[f, jT, iT])
                if interp == "bilinear":
                    num = den = f8(0.0)
                    for (j, i), w in zip(cs, ws):
                        c4 = f8(F[f, j, i])
                        if tmask[j, i] != 0 and np.isfinite(c4):
                            num = num + w * c4
                            den = den + w
                    if den > 0:
                        v = num / den
                v4 = np.float32(v)
                out[f, p] = v4 if np.isfinite(v4) else np.float32(FillValue)
    return out
