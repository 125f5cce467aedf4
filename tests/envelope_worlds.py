"""Deterministic worlds that move the kernels off the Catalina map's fast paths, one branch each.

Every launcher picks a template instantiation from the shape of the world: lookup tables present or not, how many
habitats, time bins, circles and polygon edges, how large the hot part of the world model is.  The Catalina map
(27 circles, a convex 5-edge ring, 10 habitats, 10 equal contiguous time bins, 986 cells) reaches only the fastest
of them.  Each builder here returns ``(world, flags)``: ``world`` holds the keyword arguments of ``api.Env`` and
``orc.OracleWorld``; ``flags`` the header values of the flattened world model (``api.env_host_blob``) that put it on
its branch.  ``assert_flags`` checks them on the host, so a change that moves a world off its branch fails loudly
instead of quietly testing the fast path again.

Flag values: an int is compared exactly; ``(op, v)`` with op in ``<``, ``<=``, ``>``, ``>=``, ``!=``.  Besides
the header fields, ``circ_many``, ``hab_many`` and ``poly_full`` count classification-grid cells with that code.
"""
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

CIRC_MANY, HAB_MANY, POLY_FULL = 1 << 11, 1 << 12, 1 << 13
OFFSET = (2500.0, -1500.0)


def catalina_parts():
    with open(os.path.join(GOLDEN, "catalina_map.json")) as f:
        m = json.load(f)
    z = np.load(os.path.join(GOLDEN, "shark_grid.npz"))
    return dict(circles=np.asarray(m["circles"], float), boundary=np.asarray(m["boundary"], float),
                habitats=np.asarray(m["habitats"], float), bins=np.asarray(z["bins"], float),
                cells=np.asarray(m["cells"], float), probs=np.asarray(z["probs"], float))


def catalina():
    return catalina_parts(), {"K": 27, "E": 5, "H": 10, "T": 10, "C": 986, "convex": ("!=", 0), "bins_uniform": 1,
                              "gnx": (">", 0), "nxb": (">", 0), "hot_bytes": ("<=", 24 * 1024 - 16)}


def bins():
    """40 time bins of unequal widths with a gap, an overlap and a listed-out-of-order overlapping pair: the first
    bin in list order that holds a time stamp is not the earliest one"""
    w = catalina_parts()
    rs = np.random.RandomState(40)
    edges = np.concatenate([[0.0], np.cumsum(rs.uniform(6.0, 22.0, 40))])
    b = np.stack([edges[:-1], edges[1:]], 1)
    b[13:, :] += 3.0                               # a 3 s gap between bins 12 and 13: time stamps there have no bin
    b[20, 0] -= 4.0                                # bin 20 overlaps bin 19: the first match is 19
    b[31, 0] -= 5.0                                # bin 31 overlaps bin 30 ...
    b[[30, 31]] = b[[31, 30]]                      # ... and is listed first: the first match is the later bin
    w["bins"] = b * (520.0 / b[:, 1].max())
    w["probs"] = rs.uniform(0.0, 0.6, (40, len(w["cells"])))
    return w, {"T": 40, "bins_uniform": 0, "gnx": (">", 0), "nxb": (">", 0), "H": 10}


def _habitats(n, seed):
    w = catalina_parts()
    rs = np.random.RandomState(seed)
    extra = np.stack([rs.uniform(-320, -80, n - 10), rs.uniform(-80, 120, n - 10), rs.uniform(6.0, 26.0, n - 10)], 1)
    w["habitats"] = np.concatenate([w["habitats"], extra])
    return w


def habitats48():
    """48 overlapping habitats over the region the planners explore: habitat indices 32..47 are visited"""
    return _habitats(48, 48), {"H": 48, "gnx": (">", 0)}


def habitats64():
    """64 habitats: the grid cannot name three candidates by 6-bit index (HAB_MANY)"""
    return _habitats(64, 64), {"H": 64, "gnx": (">", 0), "hab_many": (">", 0)}


def coast():
    """a non-convex ring of 40 vertices around the planning region, circles close to its edges"""
    w = catalina_parts()
    rs = np.random.RandomState(41)
    a = np.linspace(0, 2 * np.pi, 40, endpoint=False)
    r = 230.0 + 55.0 * np.sin(5 * a) + rs.uniform(-12, 12, 40)
    ring = np.stack([-190.0 + r * np.cos(a), 20.0 + 0.8 * r * np.sin(a)], 1)
    near = ring[::2] + (np.array([-190.0, 20.0]) - ring[::2]) * rs.uniform(0.02, 0.06, (20, 1))
    w["boundary"] = ring
    w["circles"] = np.concatenate([w["circles"], np.concatenate([near, rs.uniform(2.0, 6.0, (20, 1))], 1)])
    return w, {"E": 40, "convex": 0, "gnx": (">", 0), "poly_full": (">", 0)}


def _many_circles(K, seed, rmax):
    w = catalina_parts()
    rs = np.random.RandomState(seed)
    c = np.stack([rs.uniform(-467, 82, K), rs.uniform(-153, 191, K), rs.uniform(0.2, rmax, K)], 1)
    w["circles"] = np.concatenate([w["circles"][:0], c])
    return w


def dense():
    """1,100 small circles: K > 1022 (no 10-bit circle index in the grid), K > 512 (no all-pairs circle table), and a
    hot part over 24 KB, so the planners stage less and the thread-per-tree planner leaves its fast form"""
    return _many_circles(1100, 1100, 1.2), {"K": 1100, "circ_many": (">", 0), "hot_bytes": (">", 24 * 1024)}


def huge():
    """6,000 circles: a hot part over 200 KB in both precisions, so the arc-edge launcher takes the warp-per-edge
    kernel"""
    return _many_circles(6000, 6000, 0.6), {"K": 6000, "hot_bytes": (">", 200 * 1024)}


def biggrid():
    """16,400 shark cells with distinct x bounds: 32,800 breakpoints, past the 15-bit entries of the x-bucket table
    (nxb == 0: every lookup walks the breakpoints), and a probability table no kernel can stage"""
    w = catalina_parts()
    rs = np.random.RandomState(16400)
    n = 16400
    x0, y0 = rs.uniform(-467, 70, 2 * n), rs.uniform(-153, 180, 2 * n)
    c = np.stack([x0, y0, x0 + rs.uniform(3.0, 14.0, 2 * n), y0 + rs.uniform(3.0, 14.0, 2 * n)], 1)
    # cost.py's `x <= maxy` makes a cell's x range [c0, min(c2, c3)]: keep cells whose x range ends at c2
    w["cells"] = c[c[:, 3] >= c[:, 2]][:n]
    w["probs"] = rs.uniform(0.0, 0.5, (len(w["bins"]), n))
    return w, {"C": n, "NB": (">=", 32760), "nxb": 0, "total_bytes": (">", 227 * 1024)}


def offset():
    """Catalina translated by (+2500, -1500) m: the fp32 grid margins far from the origin.  The fourth cell bound moves
    with x because cost.py compares it with x (`x <= maxy`); moved with y no cell would ever match"""
    w = catalina_parts()
    dx, dy = OFFSET
    w["circles"] = w["circles"] + [dx, dy, 0.0]
    w["boundary"] = w["boundary"] + [dx, dy]
    w["habitats"] = w["habitats"] + [dx, dy, 0.0]
    w["cells"] = w["cells"] + [dx, dy, dx, dx]
    return w, {"K": 27, "E": 5, "convex": ("!=", 0), "bins_uniform": 1, "nxb": (">", 0), "minx": (">", 2000.0)}


BUILDERS = {f.__name__: f for f in (catalina, bins, habitats48, habitats64, coast, dense, huge, biggrid, offset)}
NAMES = sorted(BUILDERS)

_cache = {}


def build(name):
    if name not in _cache:
        _cache[name] = BUILDERS[name]()
    return _cache[name]


def origin(name):
    """where the world's planning region sits relative to Catalina's"""
    return np.array(OFFSET) if name == "offset" else np.zeros(2)


def header(world, precision):
    """the header of the flattened world model plus the counts of grid codes named in the module docstring"""
    from auvrrt import api
    h, raw = api.env_host_blob(world["circles"], world["boundary"], world["habitats"], world["bins"], world["cells"],
                               world["probs"], precision)
    h = dict(h)
    n = h["gnx"] * h["gny"]
    code = raw[h["off_grid"]:h["off_grid"] + 4 * n].view(np.uint32)
    h["circ_many"] = int(((code & CIRC_MANY) != 0).sum())
    h["hab_many"] = int(((code & HAB_MANY) != 0).sum())
    h["poly_full"] = int(((code & POLY_FULL) != 0).sum())
    return h, raw


_OPS = {"<": np.less, "<=": np.less_equal, ">": np.greater, ">=": np.greater_equal, "!=": np.not_equal}


def assert_flags(name, precisions=("f32", "f64")):
    """the world is on the branch it was built for, in both precisions"""
    world, flags = build(name)
    for prec in precisions:
        h, _ = header(world, prec)
        for k, want in flags.items():
            if isinstance(want, tuple):
                assert _OPS[want[0]](h[k], want[1]), (name, prec, k, h[k], want)
            else:
                assert h[k] == want, (name, prec, k, h[k], want)
    return world


def free_starts(name, n, seed, box=(-260, -140, -20, 60)):
    """collision-free start states [n, 5] in the world's planning region (the oracle's check_collision)"""
    from oracle import orc
    world, _ = build(name)
    ow = orc.OracleWorld(**world)
    ox, oy = origin(name)
    rs = np.random.RandomState(seed)
    out = []
    while len(out) < n:
        x, y = rs.uniform(box[0], box[1]) + ox, rs.uniform(box[2], box[3]) + oy
        if orc.check_collision([[x, y]], ow) == 1:
            out.append([x, y, 0.0, 0.0, 0.0])
    return np.array(out)
