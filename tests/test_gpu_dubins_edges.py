"""GPU: the Dubins edge kernels behind auvrrt_edges_dubins / auvrrt_edges_dubins_cost (csrc/kernels.cu).

`k_edges_dubins` is the all-pairs kernel (AUVRRT_EDGES_BRUTE=1): every waypoint against every circle.  Its fp32 build
keeps a 512-circle tile in shared memory, reads the SoA arrays for the rest, evaluates |p - c|^2 as the packed
expansion |p|^2 - 2 p.c + |c|^2 relative to the edge's first waypoint, and re-evaluates a result within a rounding
guard of the decision with the direct formula.  `k_edges_dubins_culled` (the default for a world with a boundary)
tests every waypoint against the circles its classification-grid cell names.

(1) The all-pairs kernel, fp64 build, against the oracle at every waypoint tier, around the shared-memory tile, with the
    circle order reversed (the running-minimum radius `creff`), and with nothing staged.
(2) Both kernels, fp32 build, against the exact decision on the kernels' own inputs, with circles planted at chosen
    margins around the decision; padding slots of the all-pairs tiers after a launch that filled them.
(3) The culled kernels, with and without cost, on every envelope world (envelope_worlds.py) against the oracle.
(4) Planner mode 3 (Dubins-RRT, best parent) against the oracle on three envelope worlds.
"""
import numpy as np
import pytest

import envelope_worlds as ew
from fp32_exact import bound as _bound, f32 as _f32, ring as _ring, table as _table

pytestmark = pytest.mark.gpu

from oracle import orc  # noqa: E402

TOL64 = 1e-9
RHO = 1.0
ED_MAX_CTAS = 148 * 12  # the all-pairs launch's grid: at most 12 CTAs of 256 threads per SM


@pytest.fixture(scope="module")
def api():
    import auvrrt
    assert auvrrt.api.device_count() > 0, "no CUDA device"
    return auvrrt.api


@pytest.fixture
def brute(monkeypatch):
    monkeypatch.setenv("AUVRRT_EDGES_BRUTE", "1")
    monkeypatch.delenv("AUVRRT_ED_MINB", raising=False)


@pytest.fixture
def culled(monkeypatch):
    monkeypatch.delenv("AUVRRT_EDGES_BRUTE", raising=False)


def _edges(n, seed, origin=(0.0, 0.0), dist=(2.0, 40.0), circles=None):
    """n Dubins edges in the planning region; with `circles`, half of them start near a circle's rim"""
    rs = np.random.RandomState(seed)
    q0 = np.stack([rs.uniform(-400, 50, n) + origin[0], rs.uniform(-100, 120, n) + origin[1],
                   rs.uniform(-np.pi, np.pi, n)], 1)
    if circles is not None and len(circles):
        h = n // 2
        c = np.asarray(circles, float)[rs.randint(len(circles), size=h)]
        a, r = rs.uniform(-np.pi, np.pi, h), c[:, 2] + rs.uniform(-1.0, 4.0, h)
        q0[:h, 0], q0[:h, 1] = c[:, 0] + r * np.cos(a), c[:, 1] + r * np.sin(a)
    ang, d = rs.uniform(-np.pi, np.pi, n), rs.uniform(dist[0], dist[1], n)
    q1 = np.stack([q0[:, 0] + d * np.cos(ang), q0[:, 1] + d * np.sin(ang), rs.uniform(-np.pi, np.pi, n)], 1)
    return q0, q1


def _near_tie(q0, q1, rho):
    """two words of equal length within rounding (the rule of test_dubins_f64_vs_oracle_and_closure)"""
    _, _, _, al = orc.dubins_shortest(q0, q1, rho)
    alt = np.sort(al[al >= 0])
    return len(alt) > 1 and alt[1] - alt[0] < 1e-9 * max(1.0, alt[0])


def _check_f64(got, want, q0, q1, rho):
    """fp64 build against the oracle: words equal except at near-ties, booleans equal where the words are, lengths
    within 1e-9.  -> mask of the edges whose words agree"""
    safe, word, length = got[:3]
    ws, ww, wl = want
    diff = np.where(word != ww)[0]
    assert all(_near_tie(q0[i], q1[i], rho) for i in diff), diff
    same = word == ww
    assert np.array_equal(safe[same], ws[same])
    fin = np.isfinite(wl)
    assert np.array_equal(np.isfinite(length), fin)
    assert np.all(np.abs(length[fin] - wl[fin]) <= TOL64 * np.maximum(np.abs(wl[fin]), 1.0))
    return same


# ------------------------------------------------------------------------------------ (1) all-pairs, fp64
def _catalina(reverse=False):
    w, _ = ew.build("catalina")
    c = w["circles"][::-1] if reverse else w["circles"]
    return dict(circles=np.ascontiguousarray(c), boundary=w["boundary"])


def _random_circles(K, seed, rmin, rmax):
    rs = np.random.RandomState(seed)
    return np.stack([rs.uniform(-467, 82, K), rs.uniform(-153, 191, K), rs.uniform(rmin, rmax, K)], 1)


def _world_k(K):
    """a world with the Catalina boundary and K circles"""
    b = _catalina()["boundary"]
    if K == 27:
        return _catalina()
    if K == 1100:
        return dict(circles=ew.assert_flags("dense")["circles"], boundary=b)
    if K == 1:
        return dict(circles=_catalina()["circles"][10:11], boundary=b)       # r = 26.6
    return dict(circles=_random_circles(K, K, 0.5, 4.0), boundary=b)


def _oracle_waypoints(ow, q0, q1, W, rho=RHO):
    wp = np.zeros((len(q0), W, 3))
    for i in range(len(q0)):
        wp[i] = orc.edge_dubins(ow, q0[i], q1[i], rho, W)[4]
    return wp


def _creff_sensitive(world, q0, q1, W):
    """edges whose oracle decision depends on the running-minimum radius: inside the ring, and within `creff` but not
    within the own radius of some circle"""
    c = np.asarray(world["circles"], float)
    creff = np.maximum.accumulate(c[::-1, 2])[::-1]
    wp = _oracle_waypoints(orc.OracleWorld(**world), q0, q1, W)
    d = np.hypot(wp[:, :, None, 0] - c[:, 0], wp[:, :, None, 1] - c[:, 1])
    ring = orc.OracleWorld(boundary=world["boundary"])
    inside = np.array([orc.check_collision(p[:, :2], ring) == 1 for p in wp])
    return int((inside & (d <= creff).any((1, 2)) & ~(d <= c[:, 2]).any((1, 2))).sum())


ALLPAIRS_W = [2, 3, 8, 9, 12, 13, 16, 17, 20, 21, 24, 25, 32]


@pytest.mark.parametrize("order", ["forward", "reversed"])
@pytest.mark.parametrize("W", ALLPAIRS_W)
def test_allpairs_f64_waypoint_tiers(api, brute, W, order):
    """every waypoint tier (8, 12, 16, 20, 24, 32) at its upper edge and one past the tier below, on the Catalina map in
    both circle orders.  Reversed, more circles have an effective radius above their own; some edges are decided by
    that difference, so a kernel testing the own radius fails"""
    world = _catalina(order == "reversed")
    e, ow = api.Env(**world), orc.OracleWorld(**world)
    q0, q1 = _edges(2000, 100 + W, circles=world["circles"])
    got = api.edges_dubins(e, q0, q1, RHO, W, "f64")
    same = _check_f64(got, orc.edges_dubins_batch(ow, q0, q1, RHO, W), q0, q1, RHO)
    assert 0.05 < got[0][same].mean() < 0.95
    if order == "reversed":
        assert _creff_sensitive(world, q0, q1, W) >= 5
    e.close()


@pytest.mark.parametrize("W", [9, 32])
@pytest.mark.parametrize("K", [0, 1, 27, 511, 512, 513, 1100])
def test_allpairs_f64_circle_counts(api, brute, K, W):
    """no circle, one, an odd count, the 512-circle tile's edge and past it"""
    world = _world_k(K)
    assert len(world["circles"]) == K
    e, ow = api.Env(**world), orc.OracleWorld(**world)
    q0, q1 = _edges(3000, 200 + K + W, circles=world["circles"] if K else None)
    got = api.edges_dubins(e, q0, q1, RHO, W, "f64")
    same = _check_f64(got, orc.edges_dubins_batch(ow, q0, q1, RHO, W), q0, q1, RHO)
    assert 0.02 < got[0][same].mean() < 0.98
    e.close()


def test_allpairs_f64_unstaged(api, brute):
    """6,000 circles: the world model is not staged in shared memory"""
    world = ew.assert_flags("huge")
    e, ow = api.Env(**world), orc.OracleWorld(**world)
    q0, q1 = _edges(1000, 300)
    got = api.edges_dubins(e, q0, q1, RHO, 13, "f64")
    same = _check_f64(got, orc.edges_dubins_batch(ow, q0, q1, RHO, 13), q0, q1, RHO)
    assert 0.05 < got[0][same].mean() < 0.95
    e.close()


def test_allpairs_rejects_waypoint_counts(api, brute):
    from auvrrt._lib import AuvrrtError
    e = api.Env(**_catalina())
    q0, q1 = _edges(8, 1)
    for prec in ("f32", "f64"):
        with pytest.raises(AuvrrtError):
            api.edges_dubins(e, q0, q1, RHO, 1, prec)
        with pytest.raises(AuvrrtError, match=r"\(status 3\)"):       # AUVRRT_ERR_UNSUPPORTED
            api.edges_dubins(e, q0, q1, RHO, 33, prec)
    e.close()


# ------------------------------------------------------------------------------------ (2) fp32, exact decisions
def _margins(t, wp, o):
    """m = d^2 - creff2 for every (waypoint, circle) pair of the fp32 inputs (differences of fp32 values are exact in
    fp64; the fp64 squares and sum add at most 2^-51 (d^2 + creff2), added to both bounds), and the two bounds"""
    dx, dy = wp[:, :, None, 0] - t["cx"], wp[:, :, None, 1] - t["cy"]
    d2 = dx * dx + dy * dy
    m = d2 - t["creff2"]
    d = np.sqrt(d2)
    pa = np.hypot(wp[:, :, 0] - o[:, None, 0], wp[:, :, 1] - o[:, None, 1])[:, :, None]
    ca = np.hypot(t["cx"] - o[:, 0, None], t["cy"] - o[:, 1, None])[:, None, :]
    f64 = 2.0 ** -51 * (d2 + t["creff2"])
    return m, _bound(d, 0.0) + f64, _bound(d, pa + ca) + f64


def _exact(t, wp, word, chunk=96):
    """per edge: the exact decision on the fp32 inputs, and whether each kernel's fp32 decision is certain (some pair
    hits or a waypoint is outside by more than the bound, or every pair misses and every waypoint is inside by more)"""
    n = len(wp)
    ok = word != 255
    safe = np.zeros(n, bool)
    sure = {"culled": ~ok, "allpairs": ~ok}
    for s in range(0, n, chunk):
        sl = slice(s, min(n, s + chunk))
        w = wp[sl, :, :2]
        inside, psure = _ring(t, w[:, :, 0], w[:, :, 1])
        safe[sl] = ok[sl] & inside.all(1)
        out_sure = (~inside & psure).any(1)
        in_sure = (inside & psure).all(1)
        if len(t["cx"]):
            m, bc, ba = _margins(t, w, w[:, 0])
            safe[sl] &= ~(m <= 0).any((1, 2))
            for name, b in (("culled", bc), ("allpairs", ba)):
                sure[name][sl] |= ok[sl] & ((m < -b).any((1, 2)) | out_sure | ((m > b).all((1, 2)) & in_sure))
        else:
            for name in sure:
                sure[name][sl] |= ok[sl] & (out_sure | in_sure)
    return safe, sure


def _base_world(base):
    if base == "tile513":
        return dict(circles=_random_circles(511, 513, 0.2, 1.2), boundary=_catalina()["boundary"]), np.zeros(2)
    w = ew.assert_flags(base)
    return dict(circles=w["circles"], boundary=w["boundary"]), ew.origin(base)


def _select(t, wp, word, n_want, clear=0.6):
    """edges that are safe with room: every waypoint more than `clear` from every rim and from the ring; their boxes
    grown by 1 m do not overlap, so a circle planted next to one edge is far from every other selected edge"""
    ok = word != 255
    rim = np.full(len(wp), np.inf)
    for s in range(0, len(wp), 96):
        w = wp[s:s + 96, :, :2]
        d = np.hypot(w[:, :, None, 0] - t["cx"], w[:, :, None, 1] - t["cy"]) - np.sqrt(t["creff2"])
        rim[s:s + 96] = d.min((1, 2))
    inside, far = _ring(t, wp[:, :, 0], wp[:, :, 1], clear)
    cand = np.where(ok & (rim > clear) & (inside & far).all(1))[0]
    chosen, lo, hi = [], np.zeros((0, 2)), np.zeros((0, 2))
    for i in cand:
        a, b = wp[i, :, :2].min(0) - 1.0, wp[i, :, :2].max(0) + 1.0
        if not ((a < hi).all(1) & (lo < b).all(1)).any():
            chosen.append(i)
            lo, hi = np.vstack([lo, a]), np.vstack([hi, b])
            if len(chosen) == n_want:
                return chosen
    raise AssertionError("only %d separated clear edges" % len(chosen))


SCALES = (0.5, 2.0, 10.0, 100.0, 1000.0)
CASES = [(k, sign, s) for k in ("near", "last") for sign in (-1, 1) for s in SCALES]


def _plant(wpe, k, sign, scale, d0):
    """a circle (fp32 centre and radius) off waypoint k of one edge, at distance ~d0 on the side away from the other
    waypoints, with a radius that puts the exact margin d^2 - r^2 at sign * scale * (the all-pairs bound)"""
    P = wpe[k, :2]
    nrm = np.array([-np.sin(wpe[k, 2]), np.cos(wpe[k, 2])])
    others = np.delete(wpe[:, :2], k, 0)
    best = None
    for side in (1.0, -1.0):
        C = _f32(P + side * d0 * nrm)
        clear = np.hypot(*(others - C).T).min() if len(others) else np.inf
        if best is None or clear > best[0]:
            best = (clear, C)
    C = best[1]
    d2 = float(((P - C) ** 2).sum())
    b = float(_bound(np.sqrt(d2), np.hypot(*(P - wpe[0, :2])) + np.hypot(*(C - wpe[0, :2]))))
    target = sign * scale * b
    r = up = dn = np.float32(np.sqrt(d2 - target))
    cands = [r]
    for _ in range(4):                                   # the fp32 radius whose creff2 = fl(r * r) is nearest the target
        up, dn = np.nextafter(up, np.float32(np.inf)), np.nextafter(dn, np.float32(0))
        cands += [up, dn]
    r = float(min(cands, key=lambda x: abs((d2 - float(x * x)) - target)))
    return [C[0], C[1], r]


def _f32_kernels(api, monkeypatch, e, q0, q1, W):
    """(culled, all-pairs) outputs; the all-pairs kernel at its three register targets, which must agree bit for bit"""
    monkeypatch.delenv("AUVRRT_EDGES_BRUTE", raising=False)
    cul = api.edges_dubins(e, q0, q1, RHO, W, "f32")
    monkeypatch.setenv("AUVRRT_EDGES_BRUTE", "1")
    outs = []
    for mb in ("1", "2", "3"):
        monkeypatch.setenv("AUVRRT_ED_MINB", mb)
        outs.append(api.edges_dubins(e, q0, q1, RHO, W, "f32"))
    monkeypatch.delenv("AUVRRT_ED_MINB")
    monkeypatch.delenv("AUVRRT_EDGES_BRUTE")
    for o in outs[1:]:
        for a, b in zip(outs[0], o):
            assert np.array_equal(a, b), "AUVRRT_ED_MINB changes the all-pairs kernel's output"
    return cul, outs[0]


def _compare_exact(tag, t, wp, word, length, cul, allp, stats):
    """both kernels against the exact decision wherever it is certain.  The all-pairs kernel's six-word solve equals
    steer_dubins' bit for bit.  The culled kernel's solve is compiled into a different kernel and may contract its
    multiply-adds differently: on a B200 its length differed from steer_dubins' in the last bits (at most 2.0e-7
    relative) on 2-3 % of the edges, words never.  Its waypoints may then differ as well, so those edges are left out
    of its exact comparison.  -> mask of the edges the culled kernel is compared on"""
    assert np.array_equal(allp[1], word) and np.array_equal(allp[2], length), tag
    assert np.array_equal(cul[1], word), tag
    assert np.all(np.abs(cul[2] - length) <= 4e-7 * np.maximum(length, 1.0)), tag
    same = cul[2] == length
    safe, sure = _exact(t, wp, word)
    sure["culled"] &= same
    for name, out in (("culled", cul), ("allpairs", allp)):
        got = out[0].astype(bool)
        bad = np.where(sure[name] & (got != safe))[0]
        assert len(bad) == 0, (tag, name, bad[:10])
        stats[name + "_in_bound"] += int((~sure[name]).sum())
        stats[name + "_in_bound_disagree"] += int((~sure[name] & (got != safe)).sum())
    stats["culled_other_rounding"] += int((~same).sum())
    both = sure["culled"] & sure["allpairs"]
    assert np.array_equal(cul[0][both], allp[0][both]), tag
    return same


def _planted_status(t, wpe, k, cp):
    """(margin / all-pairs bound of the planted pair, whether every other pair and waypoint is certain to be safe)"""
    m, _, ba = _margins(t, wpe[None, :, :2], wpe[None, 0, :2])
    m, ba = m[0], ba[0]
    ratio = m[k, cp] / ba[k, cp]
    m[k, cp], ba[k, cp] = 1.0, 0.0
    inside, psure = _ring(t, wpe[:, 0], wpe[:, 1])
    return ratio, bool((m > ba).all() and (inside & psure).all())


@pytest.mark.parametrize("W", [9, 20, 32])
@pytest.mark.parametrize("base", ["catalina", "offset", "dense", "tile513"])
def test_f32_kernels_match_exact_decision(api, monkeypatch, capsys, base, W):
    """fp32 culled and all-pairs kernels against the exact decision d^2 <= creff2 on their own inputs: waypoints from
    steer_dubins "f32" (the same solve and sampler; see `_compare_exact` for how far each kernel's solve equals it), circle
    table from the fp32 world model.  Wherever every deciding margin lies outside the kernel's rounding bound (`_bound`)
    the kernel must give the exact decision.

    Planted circles put the margin of one (waypoint, circle) pair of an otherwise clear edge at (0.5, 2, 10, 100, 1000)
    times the all-pairs bound, both signs, at waypoint 1 and at the last waypoint (the largest |p - o|).  For the
    all-pairs kernel these sit inside its guard (4e-6 (|p - o|^2 + |c - o|^2)), so its direct formula decides them.  On
    catalina and offset the planted circles share the tile with the map's and pair with each other (the count is odd
    for W = 9, 32 and even for W = 20, where a small far circle is added last); on dense they are all in the SoA tail;
    tile513 plants at indices 511 (the tile's last slot) and 512 (the first tail circle)."""
    world, origin = _base_world(base)
    q0, q1 = _edges(2000, 400 + W, origin=origin, dist=(3.0, 12.0))
    q0, q1 = _f32(q0), _f32(q1)
    word, _, length, wp = api.steer_dubins(q0, q1, RHO, W, "f32")
    t0 = _table(world)
    base_c = np.asarray(world["circles"], float)
    if base == "tile513":
        sel = _select(t0, wp, word, 8)
        specs = [[(sel[2 * i], "last", sign, s, 0.17), (sel[2 * i + 1], "near", sign, s, 0.15)]
                 for i, (sign, s) in enumerate([(-1, 2.0), (-1, 100.0), (1, 2.0), (1, 100.0)])]
    else:
        sel = _select(t0, wp, word, 6 * len(CASES))
        specs = [[(j, *CASES[i % len(CASES)], 0.15) for i, j in enumerate(sel)]]
    stats = dict(culled_in_bound=0, culled_in_bound_disagree=0, culled_other_rounding=0, allpairs_in_bound=0,
                 allpairs_in_bound_disagree=0)
    exercised = {}
    for spec in specs:
        planted = np.array([_plant(wp[j], 1 if k == "near" else W - 1, sign, s, d0) for j, k, sign, s, d0 in spec])
        order = np.argsort(-planted[:, 2], kind="stable")            # radii descending: each planted creff is its own r
        planted = planted[order]
        spec = [spec[i] for i in order]
        extra = [[-460.0 + origin[0], 180.0 + origin[1], 0.1]] if (W == 20 and base != "tile513") else []
        circles = np.concatenate([base_c, planted, np.reshape(extra, (-1, 3))])
        w = dict(circles=circles, boundary=world["boundary"])
        t = _table(w)
        K0 = len(base_c)
        assert np.array_equal(t["creff"][K0:K0 + len(planted)], t["cr"][K0:K0 + len(planted)])
        if base == "tile513":
            assert len(circles) == 513
        e = api.Env(**w)
        cul, allp = _f32_kernels(api, monkeypatch, e, q0, q1, W)
        e.close()
        same = _compare_exact((base, W), t, wp, word, length, cul, allp, stats)
        for i, (j, k, sign, s, d0) in enumerate(spec):
            kk = 1 if k == "near" else W - 1
            ratio, clear = _planted_status(t, wp[j], kk, K0 + i)
            assert np.sign(ratio) == sign and 0.3 * s < abs(ratio) < 3 * s, (j, k, sign, s, ratio)
            if clear and abs(ratio) > 1:
                exercised[(k, sign, s)] = exercised.get((k, sign, s), 0) + 1
                assert allp[0][j] == (sign > 0) and (cul[0][j] == (sign > 0) or not same[j]), (base, W, j, k, sign, s, ratio)
    with capsys.disabled():
        print("\n", base, "W=%d" % W, stats, "planted and certain:", dict(sorted(exercised.items())))
    if base == "tile513":
        for sign in (-1, 1):
            assert exercised.get(("last", sign, 100.0), 0) == 1 and exercised.get(("near", sign, 100.0), 0) == 1
    else:
        for k, sign, s in CASES:
            if s > 1:
                assert exercised.get((k, sign, s), 0) >= 3, (k, sign, s, exercised)


@pytest.mark.parametrize("W,tier", [(3, 8), (9, 12), (17, 20), (25, 32)])
def test_allpairs_f32_padding_slots_hold_to(api, brute, W, tier):
    """waypoint slots W .. tier-1 of an all-pairs tier repeat `to`.  A launch of the same kernel at the tier's full
    width first fills every slot of every CTA with points inside one large circle; a W-waypoint launch that read any
    of those slots instead of writing it would report hits the exact decision does not have"""
    world = _catalina()
    e = api.Env(**world)
    t = _table(world)
    big = world["circles"][10]
    n = ED_MAX_CTAS * 256
    rs = np.random.RandomState(tier)
    a, r = rs.uniform(-np.pi, np.pi, n), rs.uniform(0.0, 8.0, n)
    p0 = np.stack([big[0] + r * np.cos(a), big[1] + r * np.sin(a), rs.uniform(-np.pi, np.pi, n)], 1)
    p1 = p0 + np.stack([rs.uniform(-3, 3, n), rs.uniform(-3, 3, n), np.zeros(n)], 1)
    assert not api.edges_dubins(e, p0, p1, RHO, tier, "f32")[0].any()
    q0, q1 = _edges(3000, 500 + W)
    q0, q1 = _f32(q0), _f32(q1)
    word, _, length, wp = api.steer_dubins(q0, q1, RHO, W, "f32")
    safe, sure = _exact(t, wp, word)
    got = api.edges_dubins(e, q0, q1, RHO, W, "f32")
    assert np.array_equal(got[1], word) and np.array_equal(got[2], length)
    ok = sure["allpairs"]
    assert (ok & safe).sum() >= 200
    assert np.array_equal(got[0][ok].astype(bool), safe[ok])
    e.close()


# ------------------------------------------------------------------------------------ (3) culled, envelope worlds
@pytest.fixture(scope="module")
def envworlds(api):
    cache = {}

    def get(name):
        if name not in cache:
            w = ew.assert_flags(name)
            cache[name] = (api.Env(**w), orc.OracleWorld(**w), w, ew.origin(name))
        return cache[name]
    yield get
    for e, _, _, _ in cache.values():
        e.close()


@pytest.mark.parametrize("world", ew.NAMES)
def test_culled_vs_oracle_envelope(api, culled, envworlds, world):
    """test_edges_dubins_vs_oracle on every envelope world: fp64 exact (words but for near-ties, booleans, lengths
    1e-9), fp32 within test_edges_dubins_vs_oracle's bars.  Measured on a B200 (1000 W): no fp32 word or boolean differed
    from the oracle's on any world"""
    e, ow, _, origin = envworlds(world)
    n = 1500 if world == "huge" else 6000
    q0, q1 = _edges(n, 600, origin=origin)
    got = api.edges_dubins(e, q0, q1, RHO, 20, "f64")
    want = orc.edges_dubins_batch(ow, q0, q1, RHO, 20)
    _check_f64(got, want, q0, q1, RHO)
    assert 0.05 < want[0].mean() < 0.95
    q0f, q1f = _f32(q0), _f32(q1)
    ws, ww, _ = orc.edges_dubins_batch(ow, q0f, q1f, RHO, 20)
    s32, w32, _ = api.edges_dubins(e, q0f, q1f, RHO, 20, "f32")
    print(world, "fp32 word mismatch %.4f, safe mismatch %.4f" % ((w32 != ww).mean(), (s32 != ws).mean()))
    assert np.mean(w32 != ww) < 0.01
    assert np.mean(s32 != ws) < 0.01


def _first_habitat(hab, x, y):
    """orc.cost's habitat of a point: the first one (in order) within its radius, -1 if none"""
    d = np.hypot(hab[:, 0] - x[:, None], hab[:, 1] - y[:, None]) <= hab[:, 2]
    return np.where(d.any(1), d.argmax(1), -1)


@pytest.mark.parametrize("world", ew.NAMES)
def test_culled_cost_vs_oracle_envelope(api, culled, envworlds, world):
    """test_edges_dubins_cost_vs_oracle on every envelope world: cost terms exact against orc.cost on the oracle's own
    waypoints 1..W-1 (time stamp = arclength / velocity), fp32 within that test's bars.  The velocity spreads the time
    stamps over 0 .. ~450 s, so that on `bins` waypoints fall in the gap between two bins and in overlapping bins;
    on `habitats64` edges visit habitats 32..63.  Measured on a B200 (1000 W): fp32 and fp64 booleans, words and integer
    cost terms were identical on every world"""
    e, ow, w, origin = envworlds(world)
    rs = np.random.RandomState(12)
    n, W, rho, vel, w3 = (400 if world == "huge" else 1200), 12, 1.5, 0.15, -4.0
    q0 = np.stack([rs.uniform(-300, -100, n) + origin[0], rs.uniform(-60, 100, n) + origin[1], rs.uniform(-np.pi, np.pi, n)], 1)
    ang, dist = rs.uniform(-np.pi, np.pi, n), rs.uniform(2, 60, n)
    q1 = np.stack([q0[:, 0] + dist * np.cos(ang), q0[:, 1] + dist * np.sin(ang), rs.uniform(-np.pi, np.pi, n)], 1)
    s0, w0, l0 = api.edges_dubins(e, q0, q1, rho, W, "f64")
    safe, word, length, cost = api.edges_dubins_cost(e, q0, q1, rho, W, vel, w3, "f64")
    assert np.array_equal(safe, s0) and np.array_equal(word, w0) and np.array_equal(length, l0)
    nh = ow.c.H
    hab, bins = np.asarray(w["habitats"], float), np.asarray(w["bins"], float)
    n_pos = n_cell = n_high = n_gap = n_overlap = n_cmp = 0
    for i in range(n):
        osafe, oword, _prm, olen, wp = orc.edge_dubins(ow, q0[i], q1[i], rho, W)
        if oword != word[i]:
            assert _near_tie(q0[i], q1[i], rho), i
            continue
        n_cmp += 1
        assert osafe == safe[i], i
        assert abs(length[i] - olen) <= TOL64 * max(1.0, olen), i
        s = np.concatenate([np.arange(W - 1) * (olen / (W - 1)), [olen]])
        pts = np.stack([wp[1:, 0], wp[1:, 1], s[1:] / vel], 1)
        want = orc.cost(pts, 1.0, ow, [float(nh), 1.0, w3])
        assert cost[i, 2] == want[1] and cost[i, 1] == want[2], i
        assert abs(cost[i, 0] - want[3]) <= 1e-12 * max(1.0, abs(want[3])), i
        n_pos += cost[i, 1] > 0
        n_cell += cost[i, 0] != 0
        tt = pts[:, 2]
        inbin = ((tt[:, None] >= bins[:, 0]) & (tt[:, None] <= bins[:, 1])).sum(1)
        n_gap += int(((inbin == 0) & (tt < bins[:, 1].max())).any())
        n_overlap += int((inbin >= 2).any())
        n_high += int((_first_habitat(hab, pts[:, 0], pts[:, 1])[inbin > 0] >= 32).any())
    assert n_cmp >= 0.99 * n and n_pos > 20 and n_cell > 100
    if world == "habitats64":
        assert n_high > 0
    if world == "bins":
        assert n_gap > 0 and n_overlap > 0
    q0f, q1f = _f32(q0), _f32(q1)
    s64 = api.edges_dubins_cost(e, q0f, q1f, rho, W, vel, w3, "f64")
    s32 = api.edges_dubins_cost(e, q0f, q1f, rho, W, vel, w3, "f32")
    same = (s32[0] == s64[0]) & (s32[1] == s64[1])
    ints = (s32[3][same][:, 1:] == s64[3][same][:, 1:]).all(1)
    print(world, "fp32 same %.4f, integer cost terms %.4f" % (same.mean(), ints.mean()))
    assert same.mean() > 0.98
    assert ints.mean() > 0.98
    assert np.all(np.abs(s32[3][same][ints][:, 0] - s64[3][same][ints][:, 0])
                  <= 1e-4 * np.maximum(np.abs(s64[3][same][ints][:, 0]), 1.0))


# ------------------------------------------------------------------------------------ (4) mode 3, envelope worlds
def _mode3_params(api_or_orc, iters, **kw):
    return api_or_orc.plan_params(iters, mode=3, v=1.0, max_traj_time=200.0, dubins_rho=1.0, dubins_eta=20.0,
                                  near_radius=15.0, dubins_w=12, **kw)


@pytest.mark.parametrize("world", ["coast", "dense", "offset"])
def test_mode3_f64_matches_oracle_envelope(api, envworlds, world):
    """test_mode3_dubins_best_parent_f64_matches_oracle on a non-convex ring, on 1,100 circles and far from the origin:
    fp64 build against the oracle, decision by decision"""
    e, ow, _, _ = envworlds(world)
    Q, I = 3, 256
    starts = ew.free_starts(world, Q, 7)
    seeds = np.arange(Q) + 4200
    r = api.plan_batch(e, starts, seeds, _mode3_params(api, I, trace=True, path_cap=2048, chain_cap=255), "f64")
    n_found = 0
    for q in range(Q):
        o = orc.exploring(ow, starts[q], _mode3_params(orc, I), seed=int(seeds[q]))
        assert np.array_equal(r["trace"]["parent"][q], o["parent"]), q
        assert np.array_equal(r["trace"]["safe"][q], o["safe"]) and np.array_equal(r["trace"]["upos"][q], o["upos"])
        assert np.allclose(r["trace"]["leaf"][q], o["leaf"], rtol=1e-9, atol=1e-9)
        rec = r["records"][q]
        assert rec["status"] == o["status"] and rec["n_nodes"] == o["n_nodes"] and rec["n_cost_evals"] == len(o["cost_evals"])
        assert rec["n_waypoints"] == o["n_waypoints_total"]
        if o["status"] == 0:
            n_found += 1
            assert rec["best_iter"] == o["best_iter"] and rec["best_node"] == o["best_node"]
            assert np.allclose(rec["cost"], o["result"][1:], rtol=1e-9, atol=1e-12)
            assert np.isclose(rec["path_length"], o["result"][0], rtol=1e-9)
            assert rec["n_path"] == o["n_path"]
            assert np.allclose(r["path"][q][:o["n_path"]], o["path"], rtol=1e-9, atol=1e-9)
    assert (r["trace"]["safe"] == 0).any() and (r["trace"]["safe"] == 1).any()
    assert n_found >= 2
