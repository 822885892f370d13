"""Reference strain rates of buoy triangles (test infrastructure only; the product never imports it).

Definitions -- the contract of k_deform (sitrack_b200/csrc/st_deform.cu) and DESIGN.md section 10:

Mesh.     tri (nT,3) int indexes the buoys; each triangle is anticlockwise in the (x, y) plane at build time.
          Positions are [y, x] km pairs on the NorthPolarStereo(-45, 70) plane.
Window.   From trajectory row k0 to row k1, dt = (k1 - k0) * rdt / 86400 days.  For each vertex i:
            X_i = 0.5 * (x0_i + x1_i),  Y_i = 0.5 * (y0_i + y1_i)      mid-time positions [km]
            U_i = (x1_i - x0_i) / dt,   V_i = (y1_i - y0_i) / dt       velocities [km/day]
          Line-integral (Green's theorem) estimates of Lindsay & Stern (2003), the RGPS convention, with the sums
          over the three directed edges i -> i+1 (0->1, 1->2, 2->0):
            2A = sum (X_i Y_{i+1} - X_{i+1} Y_i)
            ux = sum (U_{i+1} + U_i)(Y_{i+1} - Y_i) / 2A,   uy = -sum (U_{i+1} + U_i)(X_{i+1} - X_i) / 2A
            vx, vy: the same with V.
Outputs.  Per triangle, f4, each computed in f8 and rounded once:
            divergence = ux + vy                                   [1/day]
            shear      = sqrt((ux - vy)^2 + (uy + vx)^2)          [1/day]
            vorticity  = vx - uy                                   [1/day]
            area       = A = 0.5 * 2A                              [km^2, mid-time, on the projection plane]
            y_ctr, x_ctr = ((Y_0 + Y_1) + Y_2) / 3, same with X    [km, mid-time centroid]
Invalid.  A vertex with mask 0 in row k0 or in row k1; or the signed areas 2A at k0 and at k1 (same formula on the
          end positions) not both positive; or A not positive.  Every output of an invalid triangle is FillValue.
Projection.  The rates are ratios of displacement to length on a conformal plane, so the local map scale cancels
          to first order; `area` is on the projection plane and is not corrected.

Every sum is spelled left to right in the order above (no np.sum, no reordering): numpy's element-wise f8
operations are correctly rounded and never contracted, so the kernel, which uses the same order with
__dadd_rn/__dsub_rn/__dmul_rn/__ddiv_rn/__dsqrt_rn and __double2float_rn, must agree bit for bit.
"""
import numpy as np

FillValue = -9999.0
NAMES = ("divergence", "shear", "vorticity", "area", "y_ctr", "x_ctr")


def twice_area(X, Y):
    """(X0 Y1 - X1 Y0) + (X1 Y2 - X2 Y1) + (X2 Y0 - X0 Y2); X, Y (n,3)."""
    t01 = X[:, 0] * Y[:, 1] - X[:, 1] * Y[:, 0]
    t12 = X[:, 1] * Y[:, 2] - X[:, 2] * Y[:, 1]
    t20 = X[:, 2] * Y[:, 0] - X[:, 0] * Y[:, 2]
    return (t01 + t12) + t20


def edge_sum(F, Z):
    """sum over the edges 0->1, 1->2, 2->0 of (F_{i+1} + F_i)(Z_{i+1} - Z_i)."""
    e01 = (F[:, 1] + F[:, 0]) * (Z[:, 1] - Z[:, 0])
    e12 = (F[:, 2] + F[:, 1]) * (Z[:, 2] - Z[:, 1])
    e20 = (F[:, 0] + F[:, 2]) * (Z[:, 0] - Z[:, 2])
    return (e01 + e12) + e20


def rates_f8(yx0, yx1, mask0, mask1, tri, dt):
    """-> (dict of the f8 values before rounding: ux, uy, vx, vy and the six outputs, valid (nT,) bool)."""
    yx0, yx1 = np.asarray(yx0, np.float64), np.asarray(yx1, np.float64)
    tri = np.asarray(tri, np.int64).reshape(-1, 3)
    dt = np.float64(dt)
    y0, x0 = yx0[tri, 0], yx0[tri, 1]
    y1, x1 = yx1[tri, 0], yx1[tri, 1]
    with np.errstate(all="ignore"):
        X, Y = 0.5 * (x0 + x1), 0.5 * (y0 + y1)
        U, V = (x1 - x0) / dt, (y1 - y0) / dt
        a2 = twice_area(X, Y)
        area = 0.5 * a2
        ux = edge_sum(U, Y) / a2
        uy = -(edge_sum(U, X) / a2)
        vx = edge_sum(V, Y) / a2
        vy = -(edge_sum(V, X) / a2)
        d, e = ux - vy, uy + vx
        r = dict(ux=ux, uy=uy, vx=vx, vy=vy, divergence=ux + vy, shear=np.sqrt(d * d + e * e), vorticity=vx - uy,
                 area=area, y_ctr=((Y[:, 0] + Y[:, 1]) + Y[:, 2]) / 3.0, x_ctr=((X[:, 0] + X[:, 1]) + X[:, 2]) / 3.0)
        valid = (np.asarray(mask0)[tri] != 0).all(1) & (np.asarray(mask1)[tri] != 0).all(1)
        valid &= (twice_area(x0, y0) > 0) & (twice_area(x1, y1) > 0) & (area > 0)
    return r, valid


def deform(yx0, yx1, mask0, mask1, tri, dt):
    """-> dict of (nT,) f4 over NAMES.  yx0, yx1 (nP,2) [y,x] km; mask0, mask1 (nP,); tri (nT,3); dt [days]."""
    r, valid = rates_f8(yx0, yx1, mask0, mask1, tri, dt)
    with np.errstate(all="ignore"):
        return {k: np.where(valid, r[k], FillValue).astype(np.float32) for k in NAMES}


def deform_series(posC, mask, tri, every, rdt):
    """The windows [w*every, (w+1)*every] of a (nrec+1, nP, 2) series; a trailing partial window is dropped."""
    nwin = (posC.shape[0] - 1) // every
    return [deform(posC[w * every], posC[(w + 1) * every], mask[w * every], mask[(w + 1) * every], tri,
                   every * rdt / 86400.0) for w in range(nwin)]
