"""CPU-only: the lookup tables of the flattened world model (csrc/env.cuh, built on the host by api.cu) against
the reference's exact predicates.

The kernels decide most waypoint tests with one load from a classification grid and find the shark cell through an
x-bucket table; both are "exact by construction": a code is definitive only if every point of the grid cell grown
by a margin gets the same answer.  These tests walk the tables the way the device code does (geom.cuh: classify,
point_within_c, point_hits_circles_c, point_contrib, find_cell, find_bin) on random and adversarial points and
compare with brute force:
  RRT.check_collision       /root/reference/path_planning/rrt_dubins.py:530-549
  habitat_shark_cost_func   /root/reference/path_planning/cost.py:173-191 (first bin, first cell with the
                            `x <= maxy` typo, first habitat)
"""
import numpy as np
import pytest

import envelope_worlds as ew
from auvrrt import api

HAB_NONE, HAB_AMBIG, HAB_ONE = 128, 192, 64
SLOW = 1 << 31
CIRC_MANY, HAB_MANY, POLY_FULL, CIRC_ONE, POLY_ONE = 1 << 11, 1 << 12, 1 << 13, 1 << 14, 1 << 15


class Blob:
    def __init__(self, world, bins, probs, precision):
        self.h, self.raw = api.env_host_blob(world["circles"], world["boundary"], world["habitats"], bins, world["cells"],
                                             probs, precision)
        self.R = np.float32 if precision == "f32" else np.float64
        h = self.h

        def arr(off, n, dt=None):
            dt = dt or self.R
            return self.raw[off:off + n * np.dtype(dt).itemsize].view(dt)
        # K circles + the "always hit" row K (radius +inf) that cells wholly inside a circle name as their one candidate
        self.cx, self.cy = arr(h["off_cx"], h["K"] + 1).astype(np.float64), arr(h["off_cy"], h["K"] + 1).astype(np.float64)
        self.creff = arr(h["off_creff"], h["K"] + 1).astype(np.float64)
        one = arr(h["off_one"], 4 * (h["K"] + 1 + max(h["E"], 1) + max(h["H"], 1))).astype(np.float64).reshape(-1, 4)
        self.cone, self.pone, self.hone = one[:h["K"] + 1], one[h["K"] + 1:h["K"] + 1 + max(h["E"], 1)], one[h["K"] + 1 + max(h["E"], 1):]
        self.px, self.py = arr(h["off_px"], h["E"]).astype(np.float64), arr(h["off_py"], h["E"]).astype(np.float64)
        self.hx, self.hy = arr(h["off_hx"], h["H"]).astype(np.float64), arr(h["off_hy"], h["H"]).astype(np.float64)
        self.hr = arr(h["off_hr"], h["H"]).astype(np.float64)
        self.b0, self.b1 = arr(h["off_b0"], h["T"]).astype(np.float64), arr(h["off_b1"], h["T"]).astype(np.float64)
        self.b1m1 = float(arr(h["off_b1"] - np.dtype(self.R).itemsize, 1)[0])
        self.brk = arr(h["off_brk"], h["NB"] + 1).astype(np.float64)
        self.piece = arr(h["off_piece"], h["NP"] + 1, np.int32)
        self.c1 = arr(h["off_c1"], h["NCAND"]).astype(np.float64)
        self.cell = arr(h["off_cell"], h["NCAND"], np.int32)
        self.xb = arr(h["off_xb"], h["nxb"], np.uint16)
        pf = self.raw[h["off_pfirst"]:h["off_pfirst"] + h["NP"] * (8 if precision == "f32" else 16)]
        if precision == "f32":
            pf = pf.view(np.dtype([("c1", np.float32), ("v", np.int32)]))
        else:
            pf = pf.view(np.dtype([("c1", np.float64), ("v", np.int32), ("pad", np.int32)]))
        self.pf_c1, self.pf_v = pf["c1"].astype(np.float64), pf["v"]
        ncell = h["gnx"] * h["gny"]
        g = arr(h["off_grid"], 3 * ncell, np.uint32)
        self.w0, self.w1, self.w2 = g[:ncell], g[ncell:2 * ncell], g[2 * ncell:]
        self.cells = np.asarray(world["cells"], dtype=np.float64).astype(self.R).astype(np.float64)   # R-rounded bounds


# the Catalina map keeps its plain ids ("f32", "f64"); the envelope worlds (envelope_worlds.py) are "<world>-<precision>"
_BLOBS = [(w, p) for w in ew.NAMES for p in ("f32", "f64")]


@pytest.fixture(scope="module", params=_BLOBS, ids=[p if w == "catalina" else "%s-%s" % (w, p) for w, p in _BLOBS])
def blob(request):
    from auvrrt import _lib
    _lib.lib()        # needs the built library, not a device
    name, prec = request.param
    world = ew.assert_flags(name, (prec,))
    b = Blob(world, world["bins"], world["probs"], prec)
    b.name = name
    return b


def _inside(b, x, y):
    """inside the boundary ring; for a convex ring also the signed edge terms det[point, edge] of the half-plane test"""
    ax, ay = b.px, b.py
    bx, by = np.roll(ax, -1), np.roll(ay, -1)
    det = (bx - ax)[None] * (y[:, None] - ay[None]) - (by - ay)[None] * (x[:, None] - ax[None])
    if b.h["convex"] != 0:
        return (det > 0).all(1) if b.h["convex"] > 0 else (det < 0).all(1), det
    inside = np.zeros(len(x), bool)          # even-odd crossings, as the host builder's inside_poly
    for xi, yi, xj, yj in zip(ax, ay, np.roll(ax, 1), np.roll(ay, 1)):
        with np.errstate(divide="ignore", invalid="ignore"):
            inside ^= ((yi > y) != (yj > y)) & (x < (xj - xi) * (y - yi) / (yj - yi) + xi)
    return inside, det


def test_catalina_header():
    h, _ = ew.header(ew.build("catalina")[0], "f32")
    assert h["K"] == 27 and h["E"] == 5 and h["H"] == 10 and h["T"] == 10 and h["C"] == 986
    assert h["convex"] != 0 and h["bins_uniform"] == 1 and h["gnx"] > 0 and h["nxb"] > 0
    assert h["hot_bytes"] <= 24 * 1024 - 16          # the planners stage the hot part next to 7 resident CTAs


def test_header_and_layout(blob):
    """the world is on its branch (the blob fixture asserts the builder's flags) and the layout is consistent"""
    h = blob.h
    assert h["hot_bytes"] % 16 == 0 and h["hot_bytes"] <= h["off_probs"] < h["total_bytes"] <= h["off_grid"]
    assert np.isinf(blob.brk[-1]) and np.all(np.diff(blob.brk[:-1]) > 0)


def test_classification_grid_is_exact(blob):
    """every claim a grid code makes holds for random points of its cell (and for points on cell borders)"""
    h = blob.h
    rs = np.random.RandomState(3)
    n = min(400_000, max(20_000, 12_000_000 // (h["K"] + 1)))      # the brute force below is n x K
    x = rs.uniform(h["minx"] - 8, h["maxx"] + 8, n)
    y = rs.uniform(h["miny"] - 8, h["maxy"] + 8, n)
    # points exactly on grid lines, filed under either neighbour
    k = n // 8
    x[:k] = h["gx0"] + h["gs"] * rs.randint(0, h["gnx"], k)
    y[k:2 * k] = h["gy0"] + h["gs"] * rs.randint(0, h["gny"], k)
    if blob.R is np.float32:
        x, y = x.astype(np.float32).astype(np.float64), y.astype(np.float32).astype(np.float64)
    for nudge in (0.0, 1e-4, -1e-4):        # the device's cell index may differ by its rounding error
        fx, fy = (x - h["gx0"]) / h["gs"] + nudge, (y - h["gy0"]) / h["gs"] + nudge
        on = (fx >= 0) & (fy >= 0) & (fx < h["gnx"]) & (fy < h["gny"])
        idx = (np.floor(fy[on]).astype(np.int64) * h["gnx"] + np.floor(fx[on]).astype(np.int64))
        xs, ys = x[on], y[on]
        code, w1, w2 = blob.w0[idx], blob.w1[idx], blob.w2[idx]
        inside, det = _inside(blob, xs, ys)
        # points off the grid are outside the polygon
        assert not _inside(blob, x[~on], y[~on])[0].any()
        pc = code & 3
        assert inside[pc == 1].all() and not inside[pc == 2].any()
        one = (pc == 0) & ((code & POLY_ONE) != 0)
        ei = ((code >> 26) & 0x1F).astype(np.int64)
        d1 = det[np.arange(len(xs)), np.minimum(ei, h["E"] - 1)]
        assert np.array_equal(inside[one], (d1[one] > 0) if h["convex"] > 0 else (d1[one] < 0))
        two = (pc == 0) & ((code & (POLY_ONE | POLY_FULL)) == 0)
        e0, e1 = ((w2 >> 18) & 0x1F).astype(np.int64), ((w2 >> 23) & 0x1F).astype(np.int64)
        ok = np.ones(len(xs), bool)
        for e in (e0, e1):
            de = det[np.arange(len(xs)), np.minimum(e, h["E"] - 1)]
            ok &= (e == 0x1F) | ((de > 0) if h["convex"] > 0 else (de < 0))
        assert np.array_equal(inside[two], ok[two])
        # circles (inflated radii)
        dist = np.hypot(xs[:, None] - blob.cx[None], ys[:, None] - blob.cy[None])
        hitk = dist <= blob.creff[None]                  # column K: the always-hit row
        assert hitk[:, h["K"]].all()
        hit = hitk[:, :h["K"]].any(1)
        assert not hit[(code & 4) != 0].any()
        c1 = ((code & 4) == 0) & ((code & CIRC_ONE) != 0)
        kk = ((code >> 16) & 0x3FF).astype(np.int64)
        assert np.array_equal(hit[c1], hitk[np.arange(len(xs)), np.minimum(kk, h["K"])][c1])
        c3 = ((code & 4) == 0) & ((code & (CIRC_ONE | CIRC_MANY)) == 0)
        h3 = np.zeros(len(xs), bool)
        for s in range(3):
            ks = ((w1 >> (10 * s)) & 0x3FF).astype(np.int64)
            h3 |= (ks != 0x3FF) & hitk[np.arange(len(xs)), np.minimum(ks, h["K"] - 1)]
        assert np.array_equal(hit[c3], h3[c3])
        # habitats: first match in list order
        inh = np.hypot(xs[:, None] - blob.hx[None], ys[:, None] - blob.hy[None]) <= blob.hr[None]
        first = np.where(inh.any(1), inh.argmax(1), -1)
        hc = (code >> 3) & 0xFF
        assert np.array_equal(first[hc < 64], hc[hc < 64].astype(np.int64))
        assert (first[hc == HAB_NONE] == -1).all()
        o = (hc >= HAB_ONE) & (hc < 128)
        hh = np.minimum((hc & 63).astype(np.int64), h["H"] - 1)
        assert np.array_equal(first[o], np.where(inh[np.arange(len(xs)), hh], hh, -1)[o])
        a3 = (hc == HAB_AMBIG) & ((code & HAB_MANY) == 0)
        f3 = np.full(len(xs), -1)
        for s in (2, 1, 0):
            hs = ((w2 >> (6 * s)) & 0x3F).astype(np.int64)
            f3 = np.where((hs != 0x3F) & inh[np.arange(len(xs)), np.minimum(hs, h["H"] - 1)], hs, f3)
        assert np.array_equal(first[a3], f3[a3])
        # the branch-free collision rule of point_unsafe_one (geom.cuh) for every cell not flagged SLOW: both single
        # candidates are always fetched (row 0 when the cell has none) and masked by the code
        ce = blob.cone[((code >> 16) & 0x3FF).astype(np.int64)]
        pe = blob.pone[((code >> 26) & 0x1F).astype(np.int64)]
        q = (xs - ce[:, 0]) ** 2 + (ys - ce[:, 1]) ** 2
        det1 = pe[:, 2] * (ys - pe[:, 1]) - pe[:, 3] * (xs - pe[:, 0])
        hit1 = ((code & CIRC_ONE) != 0) & (np.sqrt(q) <= ce[:, 3])
        in1 = (pc == 1) | (((code & POLY_ONE) != 0) & (det1 > 0))
        fast = (code & SLOW) == 0
        assert np.array_equal((~in1 | hit1)[fast], (~inside | hit)[fast])
        assert np.array_equal(blob.cone[:, 3], blob.creff) and np.array_equal(blob.hone[:h["H"], 3], blob.hr)
        # the straight-line cases must dominate on the Catalina map, or a thread-per-edge warp always takes a slow path
        if blob.name == "catalina":
            inside_free = inside & ~hit
            assert fast[inside_free].mean() > 0.97
            assert (hc != HAB_AMBIG)[inside_free].mean() > 0.97


def _find_cell_tables(b, x, y, nudge):
    """geom.cuh find_cell, step by step"""
    h = b.h
    if h["NB"] == 0:
        return -1

    def walk():
        """find_cell_walk: from any start its two loops end at the last breakpoint <= x"""
        if not (x >= b.brk[0]) or not (x <= b.brk[h["NB"] - 1]):
            return -1
        lo = int(np.searchsorted(b.brk[:h["NB"]], x, "right")) - 1
        p = 2 * lo + (0 if x == b.brk[lo] else 1)
        for k in range(b.piece[p], b.piece[p + 1]):
            if b.c1[k] <= y:
                return int(b.cell[k])
        return -1
    if h["nxb"] == 0:                 # no bucket table: every lookup walks
        return walk()
    bi = int(np.floor((x - h["xb0"]) / h["xbw"] + nudge))
    bi = min(max(bi, 0), h["nxb"] - 1)
    e = int(b.xb[bi])
    lo = (e & 0x7FFF) - 1
    if e & 0x8000:
        return walk()
    nxt = b.brk[lo + 1]
    cur = b.brk[lo] if lo >= 0 else 0.0
    if nxt <= x:
        lo, cur = lo + 1, nxt
    if lo < 0:
        return -1
    p = 2 * lo + (0 if x == cur else 1)
    v = int(b.pf_v[p])
    if v < 0:
        return -1
    if y >= b.pf_c1[p]:
        return v & 0x3FFFFFFF
    if not (v >> 30):
        return -1
    return walk()


def test_shark_cell_index_matches_first_match_scan(blob):
    """cost.py:181-184: first cell in dict order with x>=c0 and x<=c2 and y>=c1 and x<=c3 (sic)"""
    h = blob.h
    rs = np.random.RandomState(4)
    n = 6000
    x = rs.uniform(h["minx"] - 5, h["maxx"] + 5, n)
    y = rs.uniform(h["miny"] - 5, h["maxy"] + 5, n)
    # adversarial: exactly on breakpoints / cell bounds, and one ulp either side
    bk = blob.brk[:-1]
    sel = rs.randint(0, len(bk), 1500)
    x[:500] = bk[sel[:500]]
    x[500:1000] = np.nextafter(bk[sel[500:1000]].astype(blob.R), blob.R(np.inf)).astype(np.float64)
    x[1000:1500] = np.nextafter(bk[sel[1000:1500]].astype(blob.R), blob.R(-np.inf)).astype(np.float64)
    y[1500:2000] = blob.cells[rs.randint(0, len(blob.cells), 500), 1]
    if blob.R is np.float32:
        x, y = x.astype(np.float32).astype(np.float64), y.astype(np.float32).astype(np.float64)
    c = blob.cells
    multi = 0
    for i in range(n):
        m = (x[i] >= c[:, 0]) & (x[i] <= c[:, 2]) & (y[i] >= c[:, 1]) & (x[i] <= c[:, 3])
        want = int(np.argmax(m)) if m.any() else -1
        for nudge in (0.0, 1e-3, -1e-3):
            assert _find_cell_tables(blob, x[i], y[i], nudge) == want, (i, x[i], y[i], nudge)
    multi = int(((blob.xb & 0x8000) != 0).sum())
    assert multi <= 0.02 * h["nxb"]          # buckets that need the walk must stay rare


def test_time_bin_guess_matches_first_match_scan(blob):
    """cost.py:173-177: first bin in dict order with b0 <= t <= b1, found by the arithmetic guess of find_bin"""
    h = blob.h
    if blob.name == "bins":
        # unequal, gapped, overlapping bins: the device scans them in list order (find_bin), never guesses
        assert h["bins_uniform"] == 0
        return
    rs = np.random.RandomState(5)
    t = np.concatenate([rs.uniform(blob.b0[0] - 60, blob.b1[-1] + 60, 20000), blob.b0, blob.b1,
                        np.nextafter(blob.b1.astype(blob.R), blob.R(np.inf)).astype(np.float64),
                        np.nextafter(blob.b0.astype(blob.R), blob.R(-np.inf)).astype(np.float64)])
    if blob.R is np.float32:
        t = t.astype(np.float32).astype(np.float64)
    T = h["T"]
    for ti in t:
        m = (ti >= blob.b0) & (ti <= blob.b1)
        want = int(np.argmax(m)) if m.any() else -1
        for nudge in (0.0, 1e-3, -1e-3):
            k = int(np.floor((ti - h["bin_s0"]) / h["bin_w"] + nudge))
            k = min(max(k, 0), T - 1)
            up, dn = blob.b1[k], (blob.b1[k - 1] if k > 0 else blob.b1m1)     # b1[-1]: the sentinel just below b0[0]
            k += int(ti > up) - int(ti <= dn)
            got = k if ti <= blob.b1[T - 1] else -1
            assert got == want, (ti, nudge, got, want)
