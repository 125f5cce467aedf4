"""Exact references for the fp32 kernels: the fp32 tables of the flattened world model and rounding bounds of the
kernels' own arithmetic.  A kernel's fp32 decision must equal the exact decision on its fp32 inputs wherever every
deciding margin lies outside the bound.  Used by test_gpu_dubins_edges.py and test_gpu_collide_cost.py."""
import numpy as np

import envelope_worlds as ew

U = 2.0 ** -24          # unit roundoff of fp32
POLY_TOL = 0.01         # m: a point closer than this to the ring has no certain fp32 polygon answer


def f32(a):
    return np.asarray(a, np.float64).astype(np.float32).astype(np.float64)


def bound(d, a):
    """Bound on |q - d^2|, q the fp32 evaluation of the squared distance d^2 between a waypoint p and a circle centre c
    (both fp32), as the kernels compute it: q = fma(dy, dy, dx * dx) with
        culled kernel:                    dx = fl(px - cx)                               (a = 0)
        all-pairs direct formula:         dx = fl(fl(px - ox) - fl(cx - ox)), o = the edge's waypoint 0
                                                                                          (a = |p - o| + |c - o|)
    Each difference carries a relative error <= u, so |dx^ - dx| <= e = u (a + d)(1 + 2u), likewise dy.  Then
        |dx^2 + dy^2 - d^2| <= 2 e (|dx| + |dy|) + 2 e^2 <= 2 sqrt(2) d e + 2 e^2,
    and the rounded square and the fma add a relative (2u + u^2) of dx^2 + dy^2 <= (d + sqrt(2) e)^2.  The all-pairs
    kernel's expansion path decides only outside its guard, where it must agree with this (that is what the guard is
    for); inside, the direct formula decides.  1 % on top for the fp64 evaluation of the bound itself."""
    e = U * (a + d) * (1 + 2 * U)
    return 1.01 * (2 * np.sqrt(2) * d * e + 2 * e * e + (2 * U + U * U) * (d + np.sqrt(2) * e) ** 2)


def sqrt_bound(d):
    """Bound on |sqrtf(q) - d|, q as in `bound(d, 0)` and sqrtf correctly rounded (no fast-math in the build):
        |sqrt(q) - d| = |q - d^2| / (sqrt(q) + d) <= B / d,   B = bound(d, 0),
        |sqrtf(q) - sqrt(q)| <= u sqrt(q) <= u (d + B / d).
    At d = 0 both differences are exact (q = 0).  1 % and 2^-50 d on top for the fp64 evaluation."""
    d = np.asarray(d, np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        bd = np.where(d > 0, bound(d, 0.0) / d, 0.0)
    return 1.01 * (bd + U * (d + bd)) + 2.0 ** -50 * d


def table(world, header=None):
    """the fp32 arrays the kernels read: circles (cx, cy, cr, creff, creff2: the running-minimum radius folded in),
    ring (px, py), habitats (hx, hy, hr, hr2) and time bins (b0, b1).  `header`: the world's fp32 ew.header, if the
    caller has it"""
    h, raw = header or ew.header(dict(dict(habitats=(), bins=(), cells=(), probs=None), **world), "f32")

    def arr(off, n):
        return raw[off:off + 4 * n].view(np.float32).astype(np.float64)
    K, E, H, T = h["K"], h["E"], h["H"], h["T"]
    return dict(cx=arr(h["off_cx"], K), cy=arr(h["off_cy"], K), cr=arr(h["off_cr"], K),
                creff=arr(h["off_creff"], K), creff2=arr(h["off_creff2"], K), px=arr(h["off_px"], E), py=arr(h["off_py"], E),
                hx=arr(h["off_hx"], H), hy=arr(h["off_hy"], H), hr=arr(h["off_hr"], H), hr2=arr(h["off_hr2"], H),
                b0=arr(h["off_b0"], T), b1=arr(h["off_b1"], T))


def ring_distance(t, x, y):
    """crossing-number inside test against the fp32 ring, and the distance to it"""
    px, py = t["px"], t["py"]
    inside, dmin = np.zeros(x.shape, bool), np.full(x.shape, np.inf)
    for i in range(len(px)):
        ax, ay, bx, by = px[i], py[i], px[(i + 1) % len(px)], py[(i + 1) % len(px)]
        cross = (ay > y) != (by > y)
        with np.errstate(divide="ignore", invalid="ignore"):
            xi = ax + (y - ay) * (bx - ax) / (by - ay)
        inside ^= cross & (x < xi)
        ex, ey = bx - ax, by - ay
        s = np.clip(((x - ax) * ex + (y - ay) * ey) / (ex * ex + ey * ey), 0.0, 1.0)
        dmin = np.minimum(dmin, np.hypot(x - ax - s * ex, y - ay - s * ey))
    return inside, dmin


def ring(t, x, y, tol=POLY_TOL):
    """crossing-number inside test against the fp32 ring, and whether the point is farther than `tol` from it"""
    inside, dmin = ring_distance(t, x, y)
    return inside, dmin > tol
