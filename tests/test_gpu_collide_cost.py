"""GPU: the four host entries that carry the reference's collision and cost rules, on every envelope world
(envelope_worlds.py):

    auvrrt_collide         k_collide         RRT.check_collision on explicit paths (running-minimum radius)
    auvrrt_collide_points  k_collide_points  check_collision_obstacle (each circle's own radius)
    auvrrt_cost            k_cost            habitat_shark_cost_func (first bin, first cell, first habitat)
    auvrrt_cost_point      k_cost_point      habitat_shark_cost_point

They are the narrowest copy of the lookups the planners inline (classify, point_unsafe_c, find_bin, find_cell,
point_contrib).  The points sit on every decision surface those lookups have: classification-grid lines, cell bounds
(the breakpoints of the shark-cell index), ring vertices and their y levels, circle and habitat rims, time-bin
edges, each exactly and one ulp either side, and non-finite coordinates.

(0) The staging mode each launcher picks from the world's size: the table below, so that every mode runs.
(1) fp64 build against the oracle, bit for bit, with path lengths around the 32-lane chunks, grid-stride batches,
    bin masks, habitat counts and visited masks above bit 31.
(2) fp32 build against the exact decision on its own fp32 inputs.  Time bin and shark cell are settled by comparing
    fp32 inputs with fp32 bounds, so they must be exact on every point.  Circle, habitat and ring decisions must be
    exact wherever every deciding margin lies outside a rounding bound of the kernel's arithmetic (fp32_exact.py).
"""
import numpy as np
import pytest

import envelope_worlds as ew
import fp32_exact as fx

pytestmark = pytest.mark.gpu

from oracle import orc  # noqa: E402

U = fx.U
W64 = [-3.0, -3.0, -4.0]
PATH_LENGTHS = [0, 1, 31, 32, 33, 64, 65, 200, 257]
COLLIDE_WAVE = 148 * 8 * 4      # k_collide: at most 8 CTAs of 4 warps per SM, one path per warp
COST_WAVE = 148 * 4 * 4         # k_cost: at most 4 CTAs of 4 warps per SM
SCALES = (0.5, 2.0, 10.0, 100.0)


_CACHE = {}


def _cached(key, make):
    if key not in _CACHE:
        _CACHE[key] = make()
    return _CACHE[key]


def _header(name, prec):
    return _cached(("header", name, prec), lambda: ew.header(ew.build(name)[0], prec))


def _table(name):
    return _cached(("table", name), lambda: fx.table(ew.build(name)[0], _header(name, "f32")))


# ------------------------------------------------------------------------------------ (0) staging modes
def _stage_mode(hot, total, budget):
    """env_stage_mode (kernels.cu): 2 = hot part and probability table staged, 1 = hot part only, 0 = nothing"""
    if total + 16 <= budget:
        return 2
    if hot + 16 <= budget:
        return 1
    return 0


COLLIDE_BUDGET, COST_BUDGET = 100 * 1024, 200 * 1024
_UNSTAGED = ("huge", "biggrid")


def _expected_mode(kernel, name, prec):
    if name in _UNSTAGED:
        return 0
    if kernel == "cost" and name == "bins" and prec == "f64":
        return 1
    return 2


@pytest.mark.parametrize("name", ew.NAMES)
def test_staging_modes(name):
    """k_collide stages the hot part only (launch_collide passes it as the total); k_cost stages what fits in 200 KB.
    Modes 0 and 1 of k_cost and mode 0 of k_collide are reached by no other world, so a change that moves a world
    off its mode must fail here rather than quietly test mode 2 again"""
    for prec in ("f32", "f64"):
        h, _ = _header(name, prec)
        assert _stage_mode(h["hot_bytes"], h["hot_bytes"], COLLIDE_BUDGET) == _expected_mode("collide", name, prec)
        assert _stage_mode(h["hot_bytes"], h["total_bytes"], COST_BUDGET) == _expected_mode("cost", name, prec)


# ------------------------------------------------------------------------------------ decision-surface points
def _tri(a, b, dt):
    """(a, its dt neighbours below and above) paired with b: three rows per entry"""
    a = np.asarray(a, np.float64).astype(dt)
    a3 = np.concatenate([a, np.nextafter(a, dt(-np.inf)), np.nextafter(a, dt(np.inf))]).astype(np.float64)
    return a3, np.tile(np.asarray(b, np.float64), 3)


def _rims(c, r, n_ang, rs, dt):
    """points on the rims of circles (centres c[:, :2], radii r): in fp64 the y (a few ulps searched) where the
    oracle's distance sqrt(pow(dx, 2) + pow(dy, 2)) equals r exactly, with its y neighbours; in fp32 the rounded rim
    point and its neighbours.  -> x, y, number of exact rim points found"""
    a = rs.uniform(-np.pi, np.pi, (len(c), n_ang))
    x = (c[:, :1] + r[:, None] * np.cos(a)).ravel().astype(dt).astype(np.float64)
    y0 = (c[:, 1:2] + r[:, None] * np.sin(a)).ravel().astype(dt)
    cx, cy, rr = np.repeat(c[:, 0], n_ang), np.repeat(c[:, 1], n_ang), np.repeat(r, n_ang)
    y = y0.astype(np.float64)
    found = np.zeros(len(x), bool)
    if dt is np.float64:
        lo, hi = y0.copy(), y0.copy()
        steps = [y0]
        for _ in range(6):
            lo, hi = np.nextafter(lo, -np.inf), np.nextafter(hi, np.inf)
            steps += [lo, hi]
        for s in steps:
            hit = ~found & (np.sqrt(np.power(x - cx, 2) + np.power(s - cy, 2)) == rr)
            y[hit], found[hit] = s[hit], True
    y3, x3 = _tri(y, x, dt)
    return x3, y3, int(found.sum())


def _times(world, dt, rs):
    b = np.asarray(world["bins"], np.float64)
    edges = np.concatenate([b[:, 0], b[:, 1]])
    t, _ = _tri(edges, edges, dt)
    order = np.argsort(b[:, 0])
    mids = (b[order[:-1], 1] + b[order[1:], 0]) / 2            # gaps and overlaps between neighbouring bins
    extra = [b.min() - 5.0, b.max() + 5.0, b.min() - 1e-3, b.max() + 1e-3]
    rnd = rs.uniform(b.min() - 10, b.max() + 10, 200)
    t = np.concatenate([t, mids, extra, rnd]).astype(dt).astype(np.float64)
    return np.concatenate([t, [np.nan, np.inf, -np.inf]])


def _points(name, dt, seed=7):
    """[n, 3] (x, y, t) rows, dt-representable, on the world's decision surfaces; and the exact rim counts"""
    world, _ = ew.build(name)
    h = _header(name, "f64")[0]
    rs = np.random.RandomState(seed)
    lo, hi = np.array([h["minx"], h["miny"]]) - 10.0, np.array([h["maxx"], h["maxy"]]) + 10.0
    xs, ys = [], []

    def add(x, y):
        xs.append(np.asarray(x, np.float64).ravel())
        ys.append(np.asarray(y, np.float64).ravel())
    n = 3000
    add(rs.uniform(lo[0], hi[0], n), rs.uniform(lo[1], hi[1], n))
    # classification grid lines x = gx0 + i gs, y = gy0 + j gs
    gi = rs.choice(h["gnx"] + 1, min(200, h["gnx"] + 1), replace=False)
    gj = rs.choice(h["gny"] + 1, min(200, h["gny"] + 1), replace=False)
    add(*_tri(h["gx0"] + gi * h["gs"], rs.uniform(lo[1], hi[1], len(gi)), dt))
    y3, x3 = _tri(h["gy0"] + gj * h["gs"], rs.uniform(lo[0], hi[0], len(gj)), dt)
    add(x3, y3)
    # cell bounds: x == c0, x == min(c2, c3) (cost.py's `x <= c3`), y == c1; on biggrid every breakpoint
    cells = np.asarray(world["cells"], np.float64)
    sel = np.arange(len(cells)) if name == "biggrid" else rs.choice(len(cells), min(len(cells), 700), replace=False)
    c = cells[sel]
    xr = np.minimum(c[:, 2], c[:, 3])
    for xb in (c[:, 0], xr):
        add(*_tri(xb, rs.uniform(c[:, 1], c[:, 1] + 8.0), dt))
    c = c[:2000]
    y3, x3 = _tri(c[:, 1], rs.uniform(c[:, 0], np.maximum(c[:, 0], np.minimum(c[:, 2], c[:, 3]))), dt)
    add(x3, y3)
    # ring vertices, and points at a vertex's y level (the crossing-number tie)
    ring = np.asarray(world["boundary"], np.float64)
    add(*_tri(ring[:, 0], ring[:, 1], dt))
    y3, x3 = _tri(ring[:, 1], ring[:, 0], dt)
    add(x3, y3)
    add(rs.uniform(lo[0], hi[0], (len(ring), 24)), np.repeat(ring[:, 1], 24).reshape(len(ring), 24))
    # circle rims (own radius and running-minimum radius) and habitat rims
    circ = np.asarray(world["circles"], np.float64)
    ci = rs.choice(len(circ), min(len(circ), 300), replace=False)
    creff = np.maximum.accumulate(circ[::-1, 2])[::-1]
    found = {}
    for tag, r in (("circle", circ[ci, 2]), ("creff", creff[ci])):
        x, y, found[tag] = _rims(circ[ci], r, 3, rs, dt)
        add(x, y)
    hab = np.asarray(world["habitats"], np.float64)
    x, y, found["habitat"] = _rims(hab, hab[:, 2], 8, rs, dt)
    add(x, y)
    x, y = np.concatenate(xs).astype(dt).astype(np.float64), np.concatenate(ys).astype(dt).astype(np.float64)
    if name == "huge":                # 6,000 circles make the oracle's loops slow: a random subset of these rows
        keep = np.sort(rs.choice(len(x), 10000, replace=False))
        x, y = x[keep], y[keep]
    # non-finite rows (appended after any subsetting, so every world keeps all of them)
    x0, y0 = (lo + hi) / 2
    bad = np.array([[np.nan, y0], [np.inf, y0], [-np.inf, y0], [x0, np.nan], [x0, np.inf], [x0, -np.inf],
                    [np.nan, np.nan], [np.inf, -np.inf]])
    x, y = np.concatenate([x, bad[:, 0]]), np.concatenate([y, bad[:, 1]])
    t = _times(world, dt, rs)
    tt = np.concatenate([t, t[rs.randint(len(t), size=max(0, len(x) - len(t)))]])[:len(x)]
    perm = rs.permutation(len(x))
    pts = np.stack([x[perm], y[perm], tt], 1)
    return pts, found


def _dyadic_probs(world):
    """probs[b][c] = (b C + c + 1) 2^-20: distinct, exact in fp32, so a one-point path's c2 names its (bin, cell)"""
    T, Cn = len(world["bins"]), len(world["cells"])
    return (np.arange(T * Cn, dtype=np.float64).reshape(T, Cn) + 1.0) * 2.0 ** -20


def _decode(v, Cn):
    """c2 of a one-point path with w3 = 1 and t_total = 0 -> (bin, cell), (-1, -1) for 0"""
    k = np.rint(np.asarray(v) * 2.0 ** 20).astype(np.int64) - 1
    return np.where(k >= 0, k // Cn, -1), np.where(k >= 0, k % Cn, -1)


@pytest.fixture(scope="module")
def api():
    import auvrrt
    assert auvrrt.api.device_count() > 0, "no CUDA device"
    return auvrrt.api


@pytest.fixture(scope="module")
def worlds(api):
    """name -> (Env with the dyadic probability table, OracleWorld on the same data, world dict)"""
    cache = {}

    def get(name):
        if name not in cache:
            w = dict(ew.assert_flags(name))
            w["probs"] = _dyadic_probs(w)
            e = api.Env(**w)
            cache[name] = (e, orc.OracleWorld(**w), w)
        return cache[name]
    yield get
    for e, _, _ in cache.values():
        e.close()


def _oracle_collide(ow, paths):
    return np.array([orc.check_collision(p, ow) for p in paths]).astype(np.int64) % 256


def _random_paths(pts, rs, lengths=PATH_LENGTHS, per=6):
    return [pts[rs.randint(len(pts), size=L)] for L in lengths for _ in range(per)]


# ------------------------------------------------------------------------------------ (1) fp64 against the oracle
@pytest.mark.parametrize("name", ew.NAMES)
def test_f64_collide_vs_oracle(api, worlds, name):
    """collide on one-point paths (more than one grid-stride wave) and on paths of every chunk length, empty
    included (255: min([]) raises in the reference); collide_points at n = 1, 255, 256, 257 and all points"""
    e, ow, w = worlds(name)
    pts, found = _points(name, np.float64)
    # Far from the origin (offset) one ulp of y moves the oracle's distance by more than one ulp of r, so the search
    # finds almost no exact-rim points there and the fp64 `<=` rim decision has no guaranteed witness on that world;
    # every other world must have them
    if name != "offset":
        assert found["circle"] + found["creff"] >= 20 and found["habitat"] >= 30, found
    xy = pts[:, :2]
    assert (~np.isfinite(xy)).any(1).sum() == 8
    singles = [xy[i:i + 1] for i in range(len(xy))]
    assert len(singles) > COLLIDE_WAVE
    want = _oracle_collide(ow, singles)
    assert np.array_equal(api.collide(e, singles, "f64"), want)
    assert 0.05 < (want == 1).mean() < 0.95
    rs = np.random.RandomState(1)
    paths = _random_paths(xy, rs)
    got = api.collide(e, paths, "f64")
    assert np.array_equal(got, _oracle_collide(ow, paths))
    assert (got[:6] == 255).all()
    wp = np.array([orc.check_collision_obstacle(x, y, ow) for x, y in xy])
    for n in (1, 255, 256, 257, len(xy)):
        assert np.array_equal(api.collide_points(e, xy[:n], "f64"), wp[:n]), n
    assert 0.01 < (wp == 0).mean() < 0.98


@pytest.mark.parametrize("name", ew.NAMES)
def test_f64_cost_vs_oracle(api, worlds, name):
    """cost, all four outputs, on one-point paths (more than one grid-stride wave, t_total 0 or not) and on paths of
    every chunk length; cost_point with visited bits set above 31, at the first and the last time bin"""
    e, ow, w = worlds(name)
    pts, _ = _points(name, np.float64)
    rs = np.random.RandomState(2)
    singles = [pts[i:i + 1] for i in range(len(pts))]
    assert len(singles) > COST_WAVE
    tt = rs.choice([0.0, 3.7, 250.0], len(singles))
    got = api.cost(e, singles, tt, W64, precision="f64")
    want = np.array([orc.cost(p, t, ow, W64) for p, t in zip(singles, tt)])
    assert np.array_equal(got, want)
    assert (want[:, 3] != 0).mean() > 0.2 and (want[:, 2] != 0).sum() > 50
    paths = _random_paths(pts, rs)
    tt = rs.choice([0.0, 41.0, 333.3], len(paths))
    want = np.array([orc.cost(p, t, ow, W64) for p, t in zip(paths, tt)])
    assert np.array_equal(api.cost(e, paths, tt, W64, precision="f64"), want)
    H, T = len(w["habitats"]), len(w["bins"])
    xy = pts[:, :2]
    for vis in (np.zeros(H, np.uint8), (rs.uniform(size=H) < 0.5).astype(np.uint8), np.ones(64, np.uint8)):
        if H > 32:
            vis[32::3] = 1
        for tb in (0, T - 1):
            wp = np.array([orc.cost_point(x, y, ow, vis, tb, W64) for x, y in xy])
            for n in (1, 255, 256, 257, len(xy)):
                assert np.array_equal(api.cost_point(e, xy[:n], vis, tb, W64, "f64"), wp[:n]), (n, tb)


@pytest.mark.parametrize("name", ["catalina", "offset"])
def test_bin_mask_vs_oracle(api, worlds, name):
    """partial, all-zero and explicitly full masks at the bin-edge time stamps: with a mask the uniform bins take the
    list loop instead of the guess.  fp64 bit for bit; fp32 (bin, cell) exact"""
    e, ow, w = worlds(name)
    T, Cn = len(w["bins"]), len(w["cells"])
    pts, _ = _points(name, np.float64, seed=9)
    rs = np.random.RandomState(3)
    pts = pts[rs.choice(len(pts), 4000, replace=False)]
    b = np.asarray(w["bins"])
    for dt, prec in ((np.float64, "f64"), (np.float32, "f32")):
        t, _ = _tri(np.concatenate([b[:, 0], b[:, 1]]), 0, dt)
        p = pts.astype(dt).astype(np.float64)
        p[:, 2] = t[rs.randint(len(t), size=len(p))]
        ow_p = ow if prec == "f64" else _oracle_f32(w, _table(name))
        singles = [p[i:i + 1] for i in range(len(p))]
        for mask in ((rs.uniform(size=T) < 0.5).astype(np.uint8), np.zeros(T, np.uint8), np.ones(T, np.uint8)):
            if prec == "f64":
                got = api.cost(e, singles, np.zeros(len(p)), W64, bin_mask=mask, precision="f64")
                want = np.array([orc.cost(s, 0.0, ow_p, W64, bin_mask=mask) for s in singles])
                assert np.array_equal(got, want), mask
                path = p[:300]
                assert np.array_equal(api.cost(e, [path], [50.0], W64, bin_mask=mask, precision="f64")[0],
                                      orc.cost(path, 50.0, ow_p, W64, bin_mask=mask))
            else:
                got = api.cost(e, singles, np.zeros(len(p)), [0.0, 0.0, 1.0], bin_mask=mask, precision="f32")[:, 3]
                want = np.array([orc.cost(s, 0.0, ow_p, [0.0, 0.0, 1.0], bin_mask=mask)[3] for s in singles])
                bad = np.where(got != want)[0]
                assert len(bad) == 0, (mask, _decode(got[bad[:5]], Cn), _decode(want[bad[:5]], Cn), p[bad[:5]])


def test_bin_mask_and_visited_checks(api, worlds):
    """a mask over more than 32 bins is refused (UNSUPPORTED); a mask or visited list shorter than the world's bins or
    habitats is refused on the host (the library reads one byte per bin / habitat)"""
    from auvrrt._lib import AuvrrtError
    e, _, w = worlds("bins")
    p = [np.array([[-200.0, 0.0, 10.0]])]
    for prec in ("f32", "f64"):
        with pytest.raises(AuvrrtError, match=r"\(status 3\)"):
            api.cost(e, p, [1.0], W64, bin_mask=np.ones(40, np.uint8), precision=prec)
    e, _, w = worlds("catalina")
    with pytest.raises(ValueError):
        api.cost(e, p, [1.0], W64, bin_mask=np.ones(9, np.uint8))
    with pytest.raises(ValueError):
        api.cost_point(e, p[0][:, :2], np.zeros(9, np.uint8), 0, W64)
    api.cost_point(e, p[0][:, :2], np.zeros(64, np.uint8), 0, W64)


@pytest.mark.parametrize("name", ["habitats48", "habitats64"])
def test_n_habitats_vs_oracle(api, worlds, name):
    """n_habitats in {0, 1, 32, H-1, H} against an oracle world holding only the first n habitats"""
    e, _, w = worlds(name)
    H = len(w["habitats"])
    pts, _ = _points(name, np.float64, seed=11)
    rs = np.random.RandomState(4)
    singles = [pts[i:i + 1] for i in rs.choice(len(pts), 3000, replace=False)]
    paths = singles + _random_paths(pts, rs)
    tt = rs.choice([0.0, 41.0], len(paths))
    for nh in (0, 1, 32, H - 1, H):
        ow = orc.OracleWorld(**dict(w, habitats=w["habitats"][:nh]))
        want = np.array([orc.cost(p, t, ow, W64) for p, t in zip(paths, tt)])
        assert np.array_equal(api.cost(e, paths, tt, W64, n_habitats=nh, precision="f64"), want), nh


# ------------------------------------------------------------------------------------ (2) fp32, exact decisions
def _oracle_f32(w, t):
    """an oracle world whose bins and cell bounds are the fp32 tables `t`: on fp32 inputs its first-match bin and
    cell are the exact answers to the fp32 kernels' comparisons"""
    cells = fx.f32(w["cells"])
    return orc.OracleWorld(**dict(w, bins=np.stack([t["b0"], t["b1"]], 1), cells=cells))


def _pairs(x, y, cx, cy):
    """exact squared distances [n, k] from fp32 points to fp32 centres (fp64 differences of fp32 values are exact),
    in row chunks"""
    chunk = max(64, 4_000_000 // max(len(cx), 1))
    for s in range(0, len(x), chunk):
        dx = x[s:s + chunk, None] - cx[None, :]
        dy = y[s:s + chunk, None] - cy[None, :]
        yield slice(s, s + chunk), dx * dx + dy * dy


def _sq_decide(x, y, cx, cy, r2, first=False):
    """q = fma(dy, dy, dx * dx) <= r2 for every centre: exact answer (any hit, or the first hit) and certainty (every
    margin d^2 - r2 outside bound(d, 0) plus the fp64 evaluation's 2^-51 (d^2 + r2))"""
    n = len(x)
    hit = np.zeros(n, bool) if not first else np.full(n, -1)
    sure = np.ones(n, bool)
    if len(cx) == 0:
        return hit, sure
    for sl, d2 in _pairs(x, y, cx, cy):
        with np.errstate(invalid="ignore"):
            m = d2 - r2
            b = fx.bound(np.sqrt(d2), 0.0) + 2.0 ** -51 * (d2 + r2)
            h = m <= 0
            ok = np.abs(m) > b
        if first:
            hit[sl] = np.where(h.any(1), h.argmax(1), -1)
            sure[sl] = ok.all(1)
        else:
            hit[sl] = h.any(1)
            sure[sl] = (h & ok).any(1) | ok.all(1)
    return hit, sure


def _sqrt_decide(x, y, cx, cy, r):
    """sqrtf(q) <= r for every centre: [n, k] exact hits and per-point certainty (fx.sqrt_bound)"""
    hits = np.zeros((len(x), len(cx)), bool)
    sure = np.ones(len(x), bool)
    for sl, d2 in _pairs(x, y, cx, cy):
        with np.errstate(invalid="ignore"):
            d = np.sqrt(d2)
            m = d - r
            b = fx.sqrt_bound(d) + 2.0 ** -50 * (d + r)
            hits[sl] = m <= 0
            sure[sl] = (np.abs(m) > b).all(1)
    return hits, sure


def _ring_margin(t, x, y):
    """signed distance to the fp32 ring: > 0 inside"""
    inside, dmin = fx.ring_distance(t, x, y)
    return np.where(inside, dmin, -dmin)


def _lattice(x0, y0, k=30):
    """fp32 points within k ulps of (x0, y0) in each coordinate"""
    def around(v):
        v = np.float32(v)
        lo, hi, out = v, v, [v]
        for _ in range(k):
            lo, hi = np.nextafter(lo, np.float32(-np.inf)), np.nextafter(hi, np.float32(np.inf))
            out += [lo, hi]
        return np.array(out, np.float64)
    X, Y = np.meshgrid(around(x0), around(y0))
    return X.ravel(), Y.ravel()


def _plant_rim(cx, cy, rim, kind, sign, s, rs):
    """an fp32 point near the rim of the circle (cx, cy) whose margin is sign * (0.3 .. 3) * s times the kernel's
    bound: kind "sq" (q <= rim^2 as an fp32 r^2 table value, bound(d, 0)) or "sqrt" (sqrtf(q) <= rim, sqrt_bound).
    -> (x, y, margin / bound) or None"""
    for _ in range(8):
        a = rs.uniform(-np.pi, np.pi)
        R = np.sqrt(rim) if kind == "sq" else rim
        b = fx.bound(R, 0.0) / (2 * R) if kind == "sq" else fx.sqrt_bound(R)
        d = R + sign * s * b
        X, Y = _lattice(cx + d * np.cos(a), cy + d * np.sin(a))
        d2 = (X - cx) ** 2 + (Y - cy) ** 2
        if kind == "sq":
            ratio = (d2 - rim) / (fx.bound(np.sqrt(d2), 0.0) + 2.0 ** -51 * (d2 + rim))
        else:
            dd = np.sqrt(d2)
            ratio = (dd - rim) / (fx.sqrt_bound(dd) + 2.0 ** -50 * (dd + rim))
        ok = (np.sign(ratio) == sign) & (np.abs(ratio) > 0.3 * s) & (np.abs(ratio) < 3 * s)
        if ok.any():
            i = np.where(ok)[0][np.argmin(np.abs(np.log(np.abs(ratio[ok]) / s)))]
            return X[i], Y[i], ratio[i]
    return None


def _plant_ring(t, sign, s, rs):
    """an fp32 point at signed distance sign * (0.3 .. 3) * s * POLY_TOL from the ring (> 0 inside)"""
    E = len(t["px"])
    for _ in range(8):
        i = rs.randint(E)
        ax, ay, bx, by = t["px"][i], t["py"][i], t["px"][(i + 1) % E], t["py"][(i + 1) % E]
        u = rs.uniform(0.2, 0.8)
        L = np.hypot(bx - ax, by - ay)
        nx, ny = -(by - ay) / L, (bx - ax) / L
        for side in (1.0, -1.0):
            p = np.array([ax + u * (bx - ax) + side * nx * s * fx.POLY_TOL, ay + u * (by - ay) + side * ny * s * fx.POLY_TOL])
            p = fx.f32(p)
            ratio = _ring_margin(t, p[:1], p[1:])[0] / fx.POLY_TOL
            if np.sign(ratio) == sign and 0.3 * s < abs(ratio) < 3 * s:
                return p[0], p[1], ratio
    return None


def _planted(t, rs, n_obj=8):
    """planted fp32 points: kind -> list of (x, y, ratio)"""
    out = {k: [] for k in ("creff2", "cr", "hr2", "hr", "ring")}
    inside = fx.ring(t, t["cx"], t["cy"], 5.0)
    circ = np.where(inside[0] & inside[1])[0]
    circ = circ[np.argsort(-t["cr"][circ], kind="stable")][:n_obj]
    hab = rs.choice(len(t["hx"]), min(n_obj, len(t["hx"])), replace=False)
    for sign in (-1, 1):
        for s in SCALES:
            for k in circ:
                for kind, tab, rim in (("creff2", "sq", t["creff2"][k]), ("cr", "sqrt", t["cr"][k])):
                    p = _plant_rim(t["cx"][k], t["cy"][k], rim, tab, sign, s, rs)
                    if p:
                        out[kind].append(p)
            for h in hab:
                for kind, tab, rim in (("hr2", "sq", t["hr2"][h]), ("hr", "sqrt", t["hr"][h])):
                    p = _plant_rim(t["hx"][h], t["hy"][h], rim, tab, sign, s, rs)
                    if p:
                        out[kind].append(p)
            for _ in range(n_obj):
                p = _plant_ring(t, sign, s, rs)
                if p:
                    out["ring"].append(p)
    return {k: np.array(v).reshape(-1, 3) for k, v in out.items()}


def _f32_reference(w, t, pts, vis, tb):
    """exact fp32 decisions on `pts` (fp32 tables `t`) and whether each is certain"""
    x, y = pts[:, 0], pts[:, 1]
    ref = {}
    hit, hsure = _sq_decide(x, y, t["cx"], t["cy"], t["creff2"])
    with np.errstate(invalid="ignore"):
        inside, far = fx.ring(t, x, y)
    ref["unsafe"] = hit | ~inside
    ref["unsafe_sure"] = (hit & hsure) | (~inside & far) | (hsure & inside & far)
    hits, ref["cp_sure"] = _sqrt_decide(x, y, t["cx"], t["cy"], t["cr"])
    ref["cp_hit"] = hits.any(1)
    ref["hab"], ref["hab_sure"] = _sq_decide(x, y, t["hx"], t["hy"], t["hr2"], first=True)
    hh, ref["pt_sure"] = _sqrt_decide(x, y, t["hx"], t["hy"], t["hr"])
    ref["pt_new"] = (hh & ~vis[None, :len(t["hx"])].astype(bool)).sum(1)
    ref["pt_hits"] = hh.sum(1)
    ow32 = _oracle_f32(w, t)
    ref["id"] = np.array([orc.cost(p[None], 0.0, ow32, [0.0, 0.0, 1.0])[3] for p in pts])
    ref["cell_id"] = np.array([orc.cost_point(p[0], p[1], ow32, vis, tb, [0.0, 0.0, 1.0]) for p in pts])
    return ref


@pytest.mark.parametrize("name", ew.NAMES)
def test_f32_match_exact_decision(api, worlds, capsys, name):
    """fp32 collide, collide_points, cost and cost_point against the exact decision on their own fp32 inputs.

    Bin and cell: one-point paths with w3 = 1 and t_total = 0 report probs[bin][cell], a distinct dyadic id, in c2;
    it must equal the exact first match on every point, non-finite rows included.  Habitats (c1 = 1 per point in a
    bin and a habitat, c0 = the distinct count through rcp.approx, rounded), circles, ring and cost_point's counts
    must be exact wherever every deciding margin is outside the bound.  Planted points sit at +-(0.5, 2, 10, 100)
    times the bound around circle rims, habitat rims and ring edges; a minimum number of them must be certain"""
    e, _, w = worlds(name)
    t = _table(name)
    H, T, Cn = len(w["habitats"]), len(w["bins"]), len(w["cells"])
    rs = np.random.RandomState(5)
    pts, _ = _points(name, np.float32)
    plants = _planted(t, rs)
    tmid = fx.f32((t["b0"][0] + t["b1"][0]) / 2)
    kinds = []
    for k, v in plants.items():
        pts = np.concatenate([pts, np.stack([v[:, 0], v[:, 1], np.full(len(v), tmid)], 1)])
        kinds += [(k, r) for r in v[:, 2]]
    n_pl = len(kinds)
    pl = slice(len(pts) - n_pl, len(pts))
    vis = np.zeros(64, np.uint8)
    vis[1::3] = 1
    tb = T - 1
    ref = _f32_reference(w, t, pts, vis, tb)
    xy = pts[:, :2]
    stats = {}

    # bin and cell, exact on every point; habitat first match where certain
    singles = [pts[i:i + 1] for i in range(len(pts))]
    out = api.cost(e, singles, np.zeros(len(pts)), [float(H), 1.0, 1.0], precision="f32")
    bad = np.where(out[:, 3] != ref["id"])[0]
    assert len(bad) == 0, (len(bad), pts[bad[:5]], _decode(out[bad[:5], 3], Cn), _decode(ref["id"][bad[:5]], Cn))
    binned = np.isfinite(pts[:, 2]) & ((pts[:, 2][:, None] >= t["b0"]) & (pts[:, 2][:, None] <= t["b1"])).any(1)
    want_c1 = (binned & (ref["hab"] >= 0)).astype(float)
    sure = ref["hab_sure"] | ~binned
    assert np.array_equal(out[sure, 2], want_c1[sure])
    assert np.array_equal(np.rint(out[sure, 1]), want_c1[sure])
    stats["cost_uncertain"] = int((~sure).sum())
    stats["cost_uncertain_disagree"] = int((~sure & (out[:, 2] != want_c1)).sum())

    # collide (one-point paths) and collide_points
    got = api.collide(e, [p[None] for p in xy], "f32")
    s = ref["unsafe_sure"]
    bad = np.where(s & (got != (~ref["unsafe"]).astype(np.uint8)))[0]
    assert len(bad) == 0, ("collide", pts[bad[:5]])
    stats["collide_uncertain"] = int((~s).sum())
    stats["collide_uncertain_disagree"] = int((~s & (got != (~ref["unsafe"]).astype(np.uint8))).sum())
    gp = api.collide_points(e, xy, "f32")
    s = ref["cp_sure"]
    bad = np.where(s & (gp != (~ref["cp_hit"]).astype(np.uint8)))[0]
    assert len(bad) == 0, ("collide_points", pts[bad[:5]])
    stats["collide_points_uncertain"] = int((~s).sum())
    stats["collide_points_uncertain_disagree"] = int((~s & (gp != (~ref["cp_hit"]).astype(np.uint8))).sum())

    # cost_point: cell id exact; new-habitat and habitat counts where certain
    assert np.array_equal(api.cost_point(e, xy, vis, tb, [0.0, 0.0, 1.0], "f32"), ref["cell_id"])
    s = ref["pt_sure"]
    c0 = np.rint(api.cost_point(e, xy, vis, tb, [float(H), 0.0, 0.0], "f32"))
    c1 = np.rint(api.cost_point(e, xy, vis, tb, [0.0, float(H), 0.0], "f32"))
    assert np.array_equal(c0[s], ref["pt_new"][s]) and np.array_equal(c1[s], ref["pt_hits"][s])
    assert (ref["pt_new"][s] > 0).sum() > 20 and ((ref["pt_new"] < ref["pt_hits"])[s]).sum() > 5
    stats["cost_point_uncertain"] = int((~s).sum())
    stats["cost_point_uncertain_disagree"] = int((~s & ((c0 != ref["pt_new"]) | (c1 != ref["pt_hits"]))).sum())

    # planted points: the certain ones decided right (asserted above); count them per kind
    sure_of = {"creff2": ref["unsafe_sure"], "ring": ref["unsafe_sure"], "cr": ref["cp_sure"],
               "hr2": ref["hab_sure"], "hr": ref["pt_sure"]}
    certain = {k: 0 for k in plants}
    for i, (k, r) in enumerate(kinds):
        certain[k] += int(sure_of[k][pl][i] and abs(r) > 1)
    stats["planted_certain"] = certain
    for k, n in certain.items():
        assert n >= 12, (k, certain)

    # sums over multi-point paths of points whose habitat answer is certain: c2, c1 within the bound, c0 (the
    # distinct-habitat count through rcp.approx) exact once rounded
    pool = np.where(sure)[0]
    paths_i = [pool[rs.randint(len(pool), size=L)] for L in PATH_LENGTHS[1:] for _ in range(12)]
    T_tot = 37.0
    out = api.cost(e, [pts[i] for i in paths_i], np.full(len(paths_i), T_tot), [float(H), 1.0, 1.0], precision="f32")
    n_multi = 0
    for j, i in enumerate(paths_i):
        n = len(i)
        rel = 1.01 * ((n - 1) * U / (1 - n * U) + 8 * U)          # any-order sum of n terms, then c * rcp.approx(T)
        v2, v1 = ref["id"][i], want_c1[i]
        assert abs(out[j, 3] - v2.sum() / T_tot) <= rel * v2.sum() / T_tot, (j, n)
        assert abs(out[j, 2] - v1.sum() / T_tot) <= 1.01 * 8 * U * v1.sum() / T_tot, (j, n)
        habs = set(ref["hab"][i][binned[i] & (ref["hab"][i] >= 0)])
        assert np.rint(out[j, 1]) == len(habs), (j, n)
        n_multi += len(habs) > 1
    assert n_multi > len(paths_i) // 2
    with capsys.disabled():
        print("\n", name, "points", len(pts), "planted", n_pl, stats)
