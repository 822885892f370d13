"""Sea-ice deformation of buoy triangles: the mesh (host, once per run) and the strain rates between two
trajectory rows (k_deform on the device, csrc/st_deform.cu; no CPU fallback).

Definitions (DESIGN.md section 10): for a triangle of buoys followed from row k0 to row k1, dt days apart, the
velocity gradient (ux, uy, vx, vy) is the line integral over its edges of the velocities (x1-x0)/dt at the
mid-time positions (x0+x1)/2 (Lindsay & Stern 2003, the RGPS convention).  Outputs, f4 per triangle:
  divergence ux+vy, shear sqrt((ux-vy)^2+(uy+vx)^2), vorticity vx-uy [1/day];
  area [km^2, mid-time]; y_ctr, x_ctr [km, mid-time centroid].
A triangle with a masked vertex at either end, or whose signed area is not positive at either end or at mid-time,
gets FillValue (-9999) everywhere.  Positions are km on the polar stereographic plane: the rates are ratios of
displacement to length on a conformal plane, so the local map scale cancels to first order; `area` is on the
projection plane and is not corrected.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import as_c, check

__all__ = ["TriangulateCloud", "DeformationRates", "DEFORM_NAMES", "DEFORM_UNITS", "MIN_ANGLE_DEG"]

DEFORM_NAMES = ("divergence", "shear", "vorticity", "area", "y_ctr", "x_ctr")
DEFORM_UNITS = dict(divergence="day-1", shear="day-1", vorticity="day-1", area="km2", y_ctr="km", x_ctr="km")
MIN_ANGLE_DEG = 10.0          # TriangulateCloud drops slivers: rates of a flat triangle are dominated by noise


def _signed2A(yx, tri):
    y, x = yx[tri, 0], yx[tri, 1]
    return (x[:, 1] - x[:, 0]) * (y[:, 2] - y[:, 0]) - (x[:, 2] - x[:, 0]) * (y[:, 1] - y[:, 0])


def TriangulateCloud(pYX, max_edge_km=None):
    """-> tri (nT,3) i4: Delaunay triangles of the buoys pYX (nP,2) [y,x] km, indices in pYX's order.

    Every triangle is anticlockwise in the (x, y) plane.  Triangles with an edge longer than `max_edge_km`
    (default: twice the median edge of the unfiltered mesh; it keeps the mesh off holes and coastlines) or an
    interior angle below MIN_ANGLE_DEG are dropped.  Host-side (scipy.spatial), once per run."""
    try:
        from scipy.spatial import Delaunay
    except ImportError as e:
        raise ImportError("ERROR [TriangulateCloud]: scipy is needed to triangulate the buoys (scipy.spatial.Delaunay)") from e
    yx = as_c(pYX, np.float64).reshape(-1, 2)
    if yx.shape[0] < 3:
        return np.zeros((0, 3), np.int32)
    tri = Delaunay(yx[:, ::-1]).simplices.astype(np.int64)
    tri = tri[_signed2A(yx, tri) != 0]
    flip = _signed2A(yx, tri) < 0
    tri[flip] = tri[flip][:, [0, 2, 1]]
    # edge vectors opposite to vertices 0, 1, 2
    e = np.stack([yx[tri[:, 2]] - yx[tri[:, 1]], yx[tri[:, 0]] - yx[tri[:, 2]], yx[tri[:, 1]] - yx[tri[:, 0]]], 1)
    L = np.sqrt((e * e).sum(-1))
    if max_edge_km is None:
        max_edge_km = 2.0 * float(np.median(L)) if L.size else 0.0
    keep = (L <= max_edge_km).all(1)
    # interior angle at vertex k, between the two edges that meet there (law of cosines)
    cos = np.stack([(L[:, 1] ** 2 + L[:, 2] ** 2 - L[:, 0] ** 2) / (2 * L[:, 1] * L[:, 2]),
                    (L[:, 2] ** 2 + L[:, 0] ** 2 - L[:, 1] ** 2) / (2 * L[:, 2] * L[:, 0]),
                    (L[:, 0] ** 2 + L[:, 1] ** 2 - L[:, 2] ** 2) / (2 * L[:, 0] * L[:, 1])], 1)
    keep &= (cos <= np.cos(np.radians(MIN_ANGLE_DEG))).all(1)
    return as_c(tri[keep], np.int32)


def check_mesh(tri, nP):
    """(nT,3) i4 copy of tri, with every index in [0, nP) (the kernel does not range-check)."""
    tri = as_c(tri, np.int32).reshape(-1, 3)
    if tri.size and (tri.min() < 0 or tri.max() >= nP):
        raise ValueError("triangle vertex index out of range [0, %d)" % nP)
    return tri


def sort_mesh(tri):
    """Triangles sorted (stably) by their smallest vertex, so that a warp's gathers stay close together in a
    cell-major cloud.  -> (sorted (nT,3) i4, inv) with out_in_caller_order = out_sorted[..., inv]."""
    order = np.argsort(tri.min(1), kind="stable")
    inv = np.empty_like(order); inv[order] = np.arange(order.size)
    return as_c(tri[order], np.int32), inv


def launch(L, ctx, nT, tri_t, yx0_t, m0_t, yx1_t, m1_t, dt_days, out_t, stream):
    """st_deform_dev on device tensors (async on `stream`)."""
    check(L.st_deform_dev(ctx, int(nT), tri_t.data_ptr(), yx0_t.data_ptr(), m0_t.data_ptr(), yx1_t.data_ptr(),
                          m1_t.data_ptr(), float(dt_days), out_t.data_ptr(), C.c_void_p(stream.cuda_stream)), ctx)


class _Plan:
    """The triangle pass of TrackEngine.track(deform=...) over a mesh `slots` ((nT,3) buoy indices as stored on the
    device, caller's triangle order), sorted once by sort_mesh."""

    def __init__(self, torch, dev, slots):
        self.torch, self.L = torch, _lib.lib()
        tri, self.inv = sort_mesh(slots)
        self.nT = tri.shape[0]
        self.tri_t = torch.from_numpy(tri).to(dev)

    def outputs(self, pin=False):
        """((6, max(nT,1)) f4,) on the device, or pinned on the host."""
        kw = dict(pin_memory=True) if pin else dict(device=self.tri_t.device)
        return (self.torch.empty((6, max(self.nT, 1)), dtype=self.torch.float32, **kw),)

    def window(self, ctx, origins, yx1_t, m1_t, dt_days, outs, stream):
        (yx0_t, m0_t, _), = origins
        launch(self.L, ctx, self.nT, self.tri_t, yx0_t, m0_t, yx1_t, m1_t, dt_days, outs[0], stream)

    def results(self, outs):
        """(dict of (nT,) f4 DEFORM_NAMES in the caller's triangle order,)"""
        o = outs[0].numpy()[:, :self.nT][:, self.inv]                # a copy
        return ({n: o[j] for j, n in enumerate(DEFORM_NAMES)},)


def _upload_rows(pYX0, pYX1, mask0, mask1, dt_days, device, nP=None):
    """What the host entry points share: positions pYX0, pYX1 ((nP,2) [y,x] km) and masks mask0, mask1 (nP,) of the
    same buoys (nP of them when given), dt_days apart, checked and uploaded to `device` (default config.device).
    -> (torch, dev, nP, (yx0_t, m0_t, yx1_t, m1_t))."""
    from .engine import _torch
    from . import config
    torch = _torch()
    yx0, yx1 = as_c(pYX0, np.float64).reshape(-1, 2), as_c(pYX1, np.float64).reshape(-1, 2)
    nP = yx0.shape[0] if nP is None else nP
    if yx0.shape[0] != nP or yx1.shape[0] != nP or np.shape(mask0) != (nP,) or np.shape(mask1) != (nP,):
        raise ValueError("pYX0, pYX1 (nP,2) and mask0, mask1 (nP,) must describe the same %d buoys" % nP)
    if not dt_days > 0:
        raise ValueError("dt_days must be positive")
    dev = torch.device("cuda", config.device if device is None else int(device))
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt)).to(dev)
    return torch, dev, nP, (t(yx0, np.float64), t(mask0, np.int8), t(yx1, np.float64), t(mask1, np.int8))


def DeformationRates(pYX0, pYX1, mask0, mask1, tri, dt_days, device=None):
    """-> dict of (nT,) f4 over DEFORM_NAMES for the triangles `tri` (nT,3) between positions pYX0 and pYX1
    ((nP,2) [y,x] km) with masks mask0, mask1 (nP,), dt_days apart.  Host arrays in and out; the rates are
    computed on the GPU by k_deform (no CPU fallback)."""
    torch, dev, nP, (yx0_t, m0_t, yx1_t, m1_t) = _upload_rows(pYX0, pYX1, mask0, mask1, dt_days, device)
    with torch.cuda.device(dev):
        plan = _Plan(torch, dev, check_mesh(tri, nP))
        outs = plan.outputs()
        plan.window(None, [(yx0_t, m0_t, 1)], yx1_t, m1_t, dt_days, outs, torch.cuda.current_stream(dev))
        out, = plan.results([o.cpu() for o in outs])
    return {n: as_c(o, np.float32) for n, o in out.items()}
