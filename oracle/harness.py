"""TEST INFRASTRUCTURE ONLY -- deterministic replay harness for the UNMODIFIED reference.

Nothing under `oracle/` is product code.  Only `tests/`, `__graft_entry__.smoke()` and
`bench.py`'s cpu_baseline / `--impl reference` leg may import it, and only as the checker.

What it does (SURVEY.md section 8c):
  * puts `oracle/shims` (shapely/geopy/matplotlib/descartes stand-ins) and the reference's own
    directories on sys.path in the order the reference needs
    ([shims, /root/reference/path_planning, /root/reference]) and imports the unmodified
    `rrt_dubins`, `cost`, `catalina`, `motion_plan_state` modules;
  * replaces `rrt_dubins.random` by a player of a PRE-GENERATED uniform stream
    (`random.uniform(a, b)` is `a + (b - a) * random()` in CPython, Lib/random.py) and
    `rrt_dubins.time` by a fake clock that turns the wall-clock budget of
    `RRT.exploring` (/root/reference/path_planning/rrt_dubins.py:107-118) into an exact budget of
    I steer calls;
  * records, per loop iteration, the parent index, the accept flag and the new node.

`/root/reference` only exists in the build container; on the GPU box the committed fixtures under
tests/golden/ (written by oracle/make_golden.py from this harness) are used instead.
"""
from __future__ import annotations

import math
import os
import sys
import types

import numpy as np

REFERENCE_ROOT = os.environ.get("AUVRRT_REFERENCE", "/root/reference")
_HERE = os.path.dirname(os.path.abspath(__file__))
SHIMS = os.path.join(_HERE, "shims")

_REF_MODULE_NAMES = [
    "rrt_dubins", "cost", "catalina", "motion_plan_state", "sharkOccupancyGrid", "sharkEstimate",
    "path_planning", "path_planning.sharkOccupancyGrid", "shapely", "shapely.geometry",
    "shapely.ops", "shapely.wkt", "geopy", "geopy.distance", "matplotlib", "matplotlib.pyplot",
    "matplotlib.cm", "matplotlib.patches", "matplotlib.collections", "matplotlib.path",
    "descartes",
]


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "path_planning", "rrt_dubins.py"))


_ref_cache = None


def load_reference():
    """Import the unmodified reference modules; return a namespace holding them.

    The modules are removed from sys.modules again (and whatever was there before is put back) so
    that the product's drop-in modules of the same names (`rrt_dubins`, `cost`, ...) can live in
    the same process.
    """
    global _ref_cache
    if _ref_cache is not None:
        return _ref_cache
    if not reference_available():
        raise RuntimeError("reference tree not present at %s" % REFERENCE_ROOT)
    saved_mods = {n: sys.modules.pop(n) for n in _REF_MODULE_NAMES if n in sys.modules}
    saved_path = list(sys.path)
    sys.path[:0] = [SHIMS, os.path.join(REFERENCE_ROOT, "path_planning"), REFERENCE_ROOT]
    try:
        import rrt_dubins  # noqa
        import cost  # noqa
        import catalina  # noqa
        import motion_plan_state  # noqa
        import shapely.geometry as shp  # noqa
        ns = types.SimpleNamespace(
            rrt_dubins=rrt_dubins, cost=cost, catalina=catalina,
            motion_plan_state=motion_plan_state, shapely_geometry=shp,
            RRT=rrt_dubins.RRT, MPS=motion_plan_state.Motion_plan_state,
            Polygon=shp.Polygon, Point=shp.Point)
    finally:
        sys.path[:] = saved_path
        for n in _REF_MODULE_NAMES:
            sys.modules.pop(n, None)
        sys.modules.update(saved_mods)
    _ref_cache = ns
    return ns


# ---------------------------------------------------------------------------------------------
# The pre-generated sample sequence: a counter hash with 32-bit multiplies (DESIGN.md section 3).
# Position k of seed's stream is the 64-bit word hi:lo,
#   hi = M32a(c * 0x9E3779B9 + key_lo),  lo = M32b(c * 0x85EBCA77 + key_hi),  c = k + 1 mod 2^32,
# key = SplitMix64 finaliser of (seed + 1) * golden.  u_k(seed) is a pure function of (seed, k), so
# the GPU can evaluate any position without state and numpy can pre-generate the same doubles for
# the reference.  (Restated independently of the product's csrc/common.cuh; tests check both agree.)
# ---------------------------------------------------------------------------------------------
_M64 = (1 << 64) - 1
_M32 = (1 << 32) - 1
_GOLDEN = 0x9E3779B97F4A7C15


def _mix64(z: int) -> int:
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _M64
    return z ^ (z >> 31)


def stream_key(seed: int) -> int:
    return _mix64(((seed + 1) * _GOLDEN) & _M64)


def stream_bits(seed: int, k: int) -> int:
    key = stream_key(seed)
    c = (k + 1) & _M32
    a = (c * 0x9E3779B9 + (key & _M32)) & _M32
    a ^= a >> 16; a = (a * 0x21F0AAAD) & _M32; a ^= a >> 15; a = (a * 0x735A2D97) & _M32
    b = (c * 0x85EBCA77 + (key >> 32)) & _M32
    b ^= b >> 15; b = (b * 0xD168AAAD) & _M32; b ^= b >> 15; b = (b * 0xAF723597) & _M32
    return (a << 32) | b


def stream_u53(seed: int, k: int) -> float:
    return (stream_bits(seed, k) >> 11) * (2.0 ** -53)


def stream_u23(seed: int, k: int) -> float:
    """The fp32 build's uniform: the top 23 bits, exactly representable in fp32, in [0, 1)."""
    return (stream_bits(seed, k) >> 41) * (2.0 ** -23)


def stream_block(seed: int, start: int, n: int, f32u: bool = False) -> np.ndarray:
    """Vectorised u_k for k in [start, start+n) as float64 (f32u: the fp32 build's 23-bit u)."""
    key = stream_key(seed)
    with np.errstate(over="ignore"):
        c = np.arange(start + 1, start + n + 1, dtype=np.uint64).astype(np.uint32)
        a = c * np.uint32(0x9E3779B9) + np.uint32(key & _M32)
        a ^= a >> np.uint32(16); a *= np.uint32(0x21F0AAAD); a ^= a >> np.uint32(15); a *= np.uint32(0x735A2D97)
        b = c * np.uint32(0x85EBCA77) + np.uint32(key >> 32)
        b ^= b >> np.uint32(15); b *= np.uint32(0xD168AAAD); b ^= b >> np.uint32(15); b *= np.uint32(0xAF723597)
    z = (a.astype(np.uint64) << np.uint64(32)) | b.astype(np.uint64)
    if f32u:
        return (z >> np.uint64(41)).astype(np.float64) * (2.0 ** -23)
    return (z >> np.uint64(11)).astype(np.float64) * (2.0 ** -53)


def steer_arc_uniforms(i: int, n: int) -> np.ndarray:
    """The n uniforms RRT.steer drew in case i of tests/golden/steer_arc.npz (oracle/make_golden.py): Python's own
    Mersenne Twister seeded with i for i % 5 == 4, else stream 1000 + i from position 0.  Both are exact functions
    of (i, n), so the golden file stores only the counts."""
    i = int(i)          # numpy integers overflow in stream_key's arithmetic
    if i % 5 == 4:
        r = RecordingRandom(i)
        return np.array([r.random() for _ in range(n)], dtype=np.float64)
    return stream_block(1000 + i, 0, n)


class StreamPlayer:
    """Stands in for the `random` module inside the reference: plays u_0, u_1, ...

    Slot addressing of RRT.steer (DESIGN.md section 3).  In the stream of a planning query a steer call
    owns 1 + 3 * n_expand consecutive positions: its n_expand draw, then THREE slots per arc primitive
    (dist, diff, velocity_temp).  The reference only draws velocity_temp when abs(dist) > abs(diff)
    (/root/reference/path_planning/rrt_dubins.py:266,279); otherwise the primitive's third slot is left
    unread and the reference's next draw is served from the next primitive's first slot.  The harness
    brackets every steer call with begin_steer() / end_steer() so that the player can do that skipping;
    the reference itself is unmodified and sees a plain flat sequence of uniforms (`served` records it).
    Outside steer calls (parent picks) and without the bracket the player is plain flat.
    """

    def __init__(self, seed=None, values=None, f32u=False, record=False):
        self.seed = seed
        self.values = None if values is None else np.asarray(values, dtype=np.float64)
        self.f32u = f32u
        self.pos = 0
        self._block = None
        self._block_start = 0
        self._steer = None          # inside a steer call: [draws served, dist, edge base position, n_expand]
        self.served = [] if record else None

    def begin_steer(self):
        self._steer = {"n": 0, "dist": None, "base": self.pos, "n_expand": None}

    def end_steer(self):
        st, self._steer = self._steer, None
        if st is not None and st["n_expand"] is not None:
            self.pos = st["base"] + 1 + 3 * st["n_expand"]      # past the edge's slots, read or not

    def uniform(self, a, b):
        st = self._steer
        if st is None:
            return a + (b - a) * self.random()
        # inside steer: draw 0 is n_expand; then per primitive slot 0 = dist, slot 1 = diff, slot 2 =
        # velocity_temp, which the reference asks for only when abs(dist) > abs(diff)
        if st["n_expand"] is None:
            v = a + (b - a) * self.random()
            st["n_expand"] = int(math.floor(v / 1))
            st["slot"] = 0
            return v
        if st["slot"] == 0:
            v = a + (b - a) * self.random()
            st["dist"] = v
            st["slot"] = 1
            return v
        if st["slot"] == 1:
            v = a + (b - a) * self.random()
            if abs(st["dist"]) > abs(v):
                st["slot"] = 2
            else:
                self.pos += 1       # the unread velocity slot
                st["slot"] = 0
            return v
        v = a + (b - a) * self.random()
        st["slot"] = 0
        return v

    def random(self) -> float:
        k = self.pos
        self.pos += 1
        if self.values is not None:
            u = float(self.values[k])
        else:
            if self._block is None or not (self._block_start <= k < self._block_start + len(self._block)):
                self._block_start = k
                self._block = stream_block(self.seed, k, 4096, self.f32u)
            u = float(self._block[k - self._block_start])
        if self.served is not None:
            self.served.append(u)
        return u

    def choice(self, seq):
        """random.choice on the pre-generated sequence: element int(u * len)."""
        return seq[int(self.random() * len(seq))]


class RecordingRandom:
    """Wraps Python's own Mersenne Twister and records every u it hands out."""

    def __init__(self, seed):
        import random as _r
        self._r = _r.Random(seed)
        self.log = []

    def random(self):
        u = self._r.random()
        self.log.append(u)
        return u

    def uniform(self, a, b):
        return a + (b - a) * self.random()

    def choice(self, seq):
        return seq[int(self.random() * len(seq))]


class BudgetClock:
    """`time` stand-in: time() is `done * dt` (0.0 when dt == 0) until `budget` steer calls have
    completed, then +inf.  dt > 0 simulates a planner that spends max_plan_time evenly over its steer
    calls: the clock the wall-clock parent pick (get_closest_mps_time) is replayed on."""

    def __init__(self, budget, dt=0.0):
        self.budget = budget
        self.done = 0
        self.dt = dt

    def time(self):
        return self.done * self.dt if self.done < self.budget else float("inf")

    def sleep(self, _):
        pass


# ---------------------------------------------------------------------------------------------
# World model
# ---------------------------------------------------------------------------------------------
def clip_polygon_to_rect(pts, x0, y0, x1, y1):
    """Sutherland-Hodgman clip of polygon `pts` against the axis-aligned rectangle."""
    def clip(poly, inside, intersect):
        out = []
        n = len(poly)
        for i in range(n):
            cur, prv = poly[i], poly[i - 1]
            ci, pi = inside(cur), inside(prv)
            if ci:
                if not pi:
                    out.append(intersect(prv, cur))
                out.append(cur)
            elif pi:
                out.append(intersect(prv, cur))
        return out

    def ix(xc):
        return lambda p, q: (xc, p[1] + (q[1] - p[1]) * (xc - p[0]) / (q[0] - p[0]))

    def iy(yc):
        return lambda p, q: (p[0] + (q[0] - p[0]) * (yc - p[1]) / (q[1] - p[1]), yc)

    poly = list(pts)
    for inside, inter in ((lambda p: p[0] >= x0, ix(x0)), (lambda p: p[0] <= x1, ix(x1)),
                          (lambda p: p[1] >= y0, iy(y0)), (lambda p: p[1] <= y1, iy(y1))):
        if not poly:
            break
        poly = clip(poly, inside, inter)
    return poly


def polygon_area(pts):
    a = 0.0
    for i in range(len(pts)):
        x0, y0 = pts[i - 1]
        x1, y1 = pts[i]
        a += x0 * y1 - x1 * y0
    return 0.5 * a


def lattice_cell_polygons(boundary_pts, cell_size=10.0, min_area=1e-9):
    """same lattice as lattice_cells(), returning each clipped piece's vertex list (column-major)"""
    xs = [p[0] for p in boundary_pts]
    ys = [p[1] for p in boundary_pts]
    minx, miny, maxx, maxy = min(xs), min(ys), max(xs), max(ys)
    polys = []
    nx = int(math.ceil((maxx - minx) / cell_size))
    ny = int(math.ceil((maxy - miny) / cell_size))
    for i in range(nx):
        for j in range(ny):
            x0, y0 = minx + i * cell_size, miny + j * cell_size
            piece = clip_polygon_to_rect(boundary_pts, x0, y0, x0 + cell_size, y0 + cell_size)
            if len(piece) >= 3 and abs(polygon_area(piece)) > min_area:
                # drop consecutive duplicates the clipper can emit
                out = []
                for p in piece:
                    if not out or (p[0], p[1]) != out[-1]:
                        out.append((float(p[0]), float(p[1])))
                if len(out) > 1 and out[0] == out[-1]:
                    out.pop()
                polys.append(out)
    return polys


def lattice_cells(boundary_pts, cell_size=10.0, min_area=1e-9):
    """Cell bounds of the 10 m lattice clipped to the boundary polygon, COLUMN-MAJOR order.

    Stand-in for `splitCell` (/root/reference/path_planning/sharkOccupancyGrid.py:376-393), which
    needs shapely.ops.split.  Same lattice (anchored at the polygon's minx/miny); each cell's
    `.bounds` is the bounding box of the clipped piece, as shapely would report.  The ORDER in which
    GEOS emits the pieces cannot be known here (parity unpinned, SURVEY.md section 8c), so the
    order is defined as: columns by increasing x, then rows by increasing y.
    """
    xs = [p[0] for p in boundary_pts]
    ys = [p[1] for p in boundary_pts]
    minx, miny, maxx, maxy = min(xs), min(ys), max(xs), max(ys)
    cells = []
    nx = int(math.ceil((maxx - minx) / cell_size))
    ny = int(math.ceil((maxy - miny) / cell_size))
    for i in range(nx):
        for j in range(ny):
            x0, y0 = minx + i * cell_size, miny + j * cell_size
            piece = clip_polygon_to_rect(boundary_pts, x0, y0, x0 + cell_size, y0 + cell_size)
            if len(piece) >= 3 and abs(polygon_area(piece)) > min_area:
                px = [p[0] for p in piece]
                py = [p[1] for p in piece]
                cells.append((min(px), min(py), max(px), max(py)))
    return cells


class Cell:
    """Object with `.bounds`, the only attribute the hot path reads from `cell_list` entries."""

    def __init__(self, bounds):
        self.bounds = tuple(float(b) for b in bounds)


def catalina_world(ref=None):
    """Cartesian Catalina map computed by the reference's own catalina.create_environs
    (/root/reference/path_planning/catalina.py:32-65) on top of the Vincenty shim."""
    ref = ref or load_reference()
    cat = ref.catalina
    env = cat.create_environs(cat.OBSTACLES, cat.BOUNDARIES, cat.BOATS, cat.HABITATS)
    obstacles = env[0] + env[2]
    boundary_pts = [(float(m.x), float(m.y)) for m in env[1]]
    habitats = env[3]
    return {
        "circles": [[float(o.x), float(o.y), float(o.size)] for o in obstacles],
        "boundary": [list(p) for p in boundary_pts],
        "habitats": [[float(h.x), float(h.y), float(h.size)] for h in habitats],
        "cells": [list(c) for c in lattice_cells(boundary_pts, 10.0)],
    }


def world_objects(ref, world, grid_csv=None, grid=None):
    """Turn a world dict into the reference's own argument objects."""
    MPS = ref.MPS
    obstacles = [MPS(c[0], c[1], size=c[2]) for c in world["circles"]]
    habitats = [MPS(h[0], h[1], size=h[2]) for h in world["habitats"]]
    poly = ref.Polygon([tuple(p) for p in world["boundary"]])
    cells = [Cell(c) for c in world["cells"]]
    if grid_csv is not None:
        shark = ref.rrt_dubins.createSharkGrid(grid_csv, cells)
    elif grid is not None:
        shark = {}
        for (t0, t1), probs in grid:
            shark[(t0, t1)] = {cells[i].bounds: float(p) for i, p in enumerate(probs)}
    else:
        shark = {}
    return obstacles, poly, habitats, cells, shark


def shark_arrays(shark, cells):
    """{(t0,t1): {bounds: p}} -> (bins [T,2], probs [T,C]) in dict order."""
    bins = np.array([[k[0], k[1]] for k in shark.keys()], dtype=np.float64).reshape(-1, 2)
    probs = np.zeros((len(shark), len(cells)), dtype=np.float64)
    for ti, grid in enumerate(shark.values()):
        for ci, c in enumerate(cells):
            if c.bounds in grid:
                probs[ti, ci] = grid[c.bounds]
    return bins, probs


# ---------------------------------------------------------------------------------------------
# Traced runs of the unmodified planner
# ---------------------------------------------------------------------------------------------
def traced_exploring(ref, rrt, initial, habitats, *, iterations, rng, bin_interval=5, v=2,
                     shark_interval=50, traj_time_stamp=True, max_plan_time=10.0,
                     max_traj_time=500.0, plan_time=True, weights=(-3, -3, -4),
                     plot_interval=0.5):
    """Run RRT.exploring (/root/reference/path_planning/rrt_dubins.py:92-176) for exactly
    `iterations` steer calls on the injected uniform stream `rng`; return (result, trace).

    trace: dict of arrays, one row per steer call:
      parent  index into mps_list of the node steer started from
      safe    check_collision result (True = safe, i.e. node accepted)
      nwp     len(new.path) (waypoints incl. path[0] = parent)
      leaf    (x, y, theta, traj_time_stamp, length) of the new node
      upos    stream position before the iteration's first draw
    plus  cost_evals: list of (iteration, cost_total) for every cost evaluation, and
          best_iter: iteration whose node became the final optimum.
    """
    mod = ref.rrt_dubins
    clock = BudgetClock(iterations, (max_plan_time / iterations) if (plan_time and not traj_time_stamp) else 0.0)
    saved = (mod.random, mod.time, mod.habitat_shark_cost_func)
    tr = {"parent": [], "safe": [], "nwp": [], "leaf": [], "upos": []}
    cost_evals = []
    index_of = {}

    orig_steer = rrt.steer
    orig_cc = rrt.check_collision
    state = {"upos": 0}

    def steer(mps, *a, **k):
        if not index_of:
            pass
        for i in range(len(index_of), len(rrt.mps_list)):
            index_of[id(rrt.mps_list[i])] = i
        tr["parent"].append(index_of[id(mps)])
        if hasattr(rng, "begin_steer"):
            rng.begin_steer()
        try:
            new = orig_steer(mps, *a, **k)
        finally:
            if hasattr(rng, "end_steer"):
                rng.end_steer()
        tr["nwp"].append(len(new.path))
        tr["leaf"].append((new.x, new.y, new.theta, new.traj_time_stamp, new.length))
        return new

    def check_collision(mps, obstacles):
        r = orig_cc(mps, obstacles)
        tr["safe"].append(bool(r))
        tr["upos"].append(state["upos"])
        state["upos"] = getattr(rng, "pos", len(getattr(rng, "log", ())))
        clock.done += 1
        return r

    def cost_spy(path, t, habitats_, grid, w):
        c = saved[2](path, t, habitats_, grid, w)
        cost_evals.append((len(tr["parent"]) - 1, c[0], c[1][0], c[1][1], c[1][2], len(path)))
        return c

    rrt.steer = steer
    rrt.check_collision = check_collision
    mod.random, mod.time, mod.habitat_shark_cost_func = rng, clock, cost_spy
    try:
        try:
            res = rrt.exploring(initial, habitats, plot_interval, bin_interval, v, shark_interval,
                                traj_time_stamp=traj_time_stamp, max_plan_time=max_plan_time,
                                max_traj_time=max_traj_time, plan_time=plan_time,
                                weights=list(weights))
        except TypeError:
            res = None  # no node reached the horizon: opt_path is None (rrt_dubins.py:174)
    finally:
        mod.random, mod.time, mod.habitat_shark_cost_func = saved
        del rrt.steer, rrt.check_collision
    trace = {
        "parent": np.array(tr["parent"], dtype=np.int32),
        "safe": np.array(tr["safe"], dtype=np.uint8),
        "nwp": np.array(tr["nwp"], dtype=np.int32),
        "leaf": np.array(tr["leaf"], dtype=np.float64).reshape(-1, 5),
        "upos": np.array(tr["upos"], dtype=np.int64),
        "cost_evals": np.array(cost_evals, dtype=np.float64).reshape(-1, 6),
        "n_uniforms": getattr(rng, "pos", len(getattr(rng, "log", ()))),
    }
    return res, trace


def path_to_array(path):
    """list[Motion_plan_state] -> [n, 6] (x, y, theta, v, traj_time_stamp, length)."""
    return np.array([[p.x, p.y, p.theta, p.v, p.traj_time_stamp, p.length] for p in path],
                    dtype=np.float64).reshape(-1, 6)


# ---------------------------------------------------------------------------------------------
# gym_rrt.envs.rrt_dubins.Planner_RRT (the goal-directed planner the RL environment drives).
# ---------------------------------------------------------------------------------------------
_gym_cache = None


def load_gym_reference():
    """Import the unmodified gym_rrt/envs/{rrt_dubins,motion_plan_state_rrt,grid_cell_rrt}.py.

    The package __init__ files pull in `gym` (absent here), so empty package stubs whose __path__
    points at the reference directories stand in for them; the three modules themselves are the
    reference's own files, executed unmodified."""
    global _gym_cache
    if _gym_cache is not None:
        return _gym_cache
    if not reference_available():
        raise RuntimeError("reference tree not present at %s" % REFERENCE_ROOT)
    import importlib
    names = ["gym_rrt", "gym_rrt.envs", "gym_rrt.envs.rrt_dubins", "gym_rrt.envs.motion_plan_state_rrt",
             "gym_rrt.envs.grid_cell_rrt", "matplotlib", "matplotlib.pyplot", "matplotlib.path",
             "matplotlib.patches"]
    saved_mods = {n: sys.modules.pop(n) for n in names if n in sys.modules}
    saved_path = list(sys.path)
    sys.path[:0] = [SHIMS]
    try:
        pkg = types.ModuleType("gym_rrt")
        pkg.__path__ = [os.path.join(REFERENCE_ROOT, "gym_rrt")]
        sub = types.ModuleType("gym_rrt.envs")
        sub.__path__ = [os.path.join(REFERENCE_ROOT, "gym_rrt", "envs")]
        sys.modules["gym_rrt"], sys.modules["gym_rrt.envs"] = pkg, sub
        mod = importlib.import_module("gym_rrt.envs.rrt_dubins")
        mps = importlib.import_module("gym_rrt.envs.motion_plan_state_rrt")
        ns = types.SimpleNamespace(rrt_dubins=mod, Planner_RRT=mod.Planner_RRT, MPS=mps.Motion_plan_state)
    finally:
        sys.path[:] = saved_path
        for n in names:
            sys.modules.pop(n, None)
        sys.modules.update(saved_mods)
    _gym_cache = ns
    return ns


GYM_MAIN_OBSTACLES = [(12.0, 38.0, 4.0), (17.0, 34.0, 5.0), (20.0, 29.0, 4.0), (25.0, 25.0, 3.0),
                      (29.0, 20.0, 4.0), (34.0, 17.0, 3.0), (37.0, 8.0, 5.0)]   # gym_rrt/envs/rrt_dubins.py:509-517


def traced_gym_planning(gref, start, goal, boundary, obstacles, *, rng, max_step=200, exp_rate=1,
                        dist_to_end=2, diff_max=0.5, freq=50, cell_side_length=2, subsections_in_cell=8,
                        actions=None):
    """Run the unmodified Planner_RRT on the sequence `rng`; record what each step decided.

    start = (x, y, theta), goal = (x, y), boundary = (x0, y0, x1, y1), obstacles = [(x, y, size)].
    actions=None drives Planner_RRT.planning (cells drawn with random.choice); otherwise `actions`
    is a list of (row, col, subsection), or a callable(planner) -> (row, col, subsection) asked
    max_step times, fed to generate_one_node the way RRTEnv.step does
    (gym_rrt/envs/rrt_env.py:213-224), an empty cell being skipped by the caller.
    Returns a dict of arrays (one row per step) plus the final path (goal -> start order)."""
    M = gref.MPS
    mod = gref.rrt_dubins
    s = M(x=start[0], y=start[1], theta=start[2])
    g = M(x=goal[0], y=goal[1])
    b = [M(x=boundary[0], y=boundary[1]), M(x=boundary[2], y=boundary[3])]
    obs = [M(x=o[0], y=o[1], size=o[2]) for o in obstacles]
    saved_random = mod.random
    mod.random = rng
    try:
        pl = gref.Planner_RRT(s, g, b, obs, [], exp_rate=exp_rate, dist_to_end=dist_to_end, diff_max=diff_max,
                              freq=freq, cell_side_length=cell_side_length,
                              subsections_in_cell=subsections_in_cell)
        index_of = {id(s): 0}
        rows = []
        cur = {}
        orig_steer, orig_gen = pl.steer, pl.generate_one_node

        def steer(mps, *a, **k):
            cur["parent"] = index_of[id(mps)]
            out = orig_steer(mps, *a, **k)
            cur["nwp"] = len(out.path) - 1
            cur["cand"] = (out.x, out.y, out.theta, out.traj_time_stamp)
            return out

        def gen(cell, *a, **k):
            cur.clear()
            n_before = len(pl.mps_list)
            pos0 = rng.pos
            done, path = orig_gen(cell, *a, **k)
            accepted = len(pl.mps_list) > n_before
            if accepted:
                index_of[id(pl.mps_list[-1])] = len(pl.mps_list) - 1
            rows.append((cur["parent"], cur["nwp"], int(accepted), int(done), len(pl.mps_list),
                         len(pl.occupied_grid_cells_array), rng.pos - pos0) + cur["cand"])
            return done, path

        pl.steer, pl.generate_one_node = steer, gen
        if actions is None:
            path, step, _ = pl.planning(max_step=max_step)
            done = bool(rows and rows[-1][3])
        else:
            path, step, done = None, 0, False
            fed = []
            it = (actions(pl) for _ in range(max_step)) if callable(actions) else iter(actions)
            for (r, c, k) in it:
                fed.append((r, c, k))
                cell = pl.env_grid[r][c].subsection_cells[k]
                if cell.node_array == []:
                    continue
                done, path = pl.generate_one_node(cell)
                step += 1
                if done:
                    break
    finally:
        mod.random = saved_random
    rows = np.array(rows, dtype=np.float64).reshape(-1, 11)
    out = {
        "parent": rows[:, 0].astype(np.int32), "nwp": rows[:, 1].astype(np.int32),
        "accepted": rows[:, 2].astype(np.uint8), "done": rows[:, 3].astype(np.uint8),
        "n_nodes": rows[:, 4].astype(np.int32), "n_occupied": rows[:, 5].astype(np.int32),
        "n_uniforms": rows[:, 6].astype(np.int32), "cand": rows[:, 7:11].copy(),
        "steps": step, "found": bool(done),
        "occupied": np.array(pl.occupied_grid_cells_array, dtype=np.int32).reshape(-1, 3),
        "nodes": np.array([[m.x, m.y, m.theta, m.traj_time_stamp] for m in pl.mps_list]),
        "counts": np.array([[len(sc.node_array) for sc in cell.subsection_cells]
                            for row in pl.env_grid for cell in row], dtype=np.int32),
        "grid_shape": np.array([len(pl.env_grid), len(pl.env_grid[0])], dtype=np.int32),
    }
    if actions is not None:
        out["actions"] = np.array(fed, dtype=np.int32).reshape(-1, 3)
    if done:
        out["path"] = np.array([[m.x, m.y, m.theta] for m in path])
        out["goal_arc_length"] = float(path[0].length)
    else:
        out["path"] = np.zeros((0, 3))
        out["goal_arc_length"] = 0.0
    return out


# ---------------------------------------------------------------------------------------------
# path_planning/astar_fixLenSOG.py: the fixed-length lattice A* with the shark-occupancy cost.
# ---------------------------------------------------------------------------------------------
_astar_cache = None


def load_astar_reference():
    """Import the unmodified path_planning/astar_fixLenSOG.py the way the reference's own driver does
    (astarAnalysis.py:10-14: repository root on sys.path, so `catalina`, `motion_plan_state`,
    `sharkOccupancyGrid` and `cost` resolve to the root-level modules).  `splitCell` -- shapely.ops.split,
    whose cell order is unpinned -- is only used to label a CSV shark grid when none is passed in, so the
    harness always passes the grid and stubs splitCell out."""
    global _astar_cache
    if _astar_cache is not None:
        return _astar_cache
    if not reference_available():
        raise RuntimeError("reference tree not present at %s" % REFERENCE_ROOT)
    import importlib
    names = ["path_planning", "path_planning.astar_fixLenSOG", "catalina", "motion_plan_state", "sharkOccupancyGrid",
             "cost", "shapely", "shapely.geometry", "shapely.wkt", "shapely.ops", "geopy", "geopy.distance",
             "matplotlib", "matplotlib.pyplot", "matplotlib.cm", "matplotlib.patches", "matplotlib.collections",
             "matplotlib.path", "descartes"]
    saved_mods = {n: sys.modules.pop(n) for n in names if n in sys.modules}
    saved_path = list(sys.path)
    sys.path[:0] = [SHIMS, REFERENCE_ROOT]
    try:
        mod = importlib.import_module("path_planning.astar_fixLenSOG")
        mod.splitCell = lambda poly, size: []
        mps = importlib.import_module("motion_plan_state")
        shp = importlib.import_module("shapely.geometry")
        ns = types.SimpleNamespace(mod=mod, astar=mod.astar, Node=mod.Node, MPS=mps.Motion_plan_state, Polygon=shp.Polygon)
    finally:
        sys.path[:] = saved_path
        for n in names:
            sys.modules.pop(n, None)
        sys.modules.update(saved_mods)
    _astar_cache = ns
    return ns


def round_cells(cells):
    """cell bounds as get_cell_prob compares them: every coordinate through Python's round(v, 2)
    (astar_fixLenSOG.py:494-495)"""
    return np.array([[round(float(v), 2) for v in c] for c in cells], dtype=np.float64).reshape(-1, 4)


def traced_astar(aref, start, circles, boundary, habitats, bins, cells, probs, *, velocity=1, path_len_limit=300,
                 weights=(0, 10, 10, 100)):
    """Run the unmodified astar.astar (prints swallowed); -> dict with the expansion order, the node path,
    the cost list and which trajectory points smoothPath kept, or {"raised": ExceptionName}."""
    import contextlib
    import io
    M = aref.MPS
    grid = {}
    for t, (b0, b1) in enumerate(bins):
        key = (int(b0), int(b1)) if float(b0).is_integer() and float(b1).is_integer() else (float(b0), float(b1))
        grid[key] = {tuple(float(v) for v in c): float(probs[t][i]) for i, c in enumerate(cells)}
    obst = [M(c[0], c[1], size=c[2]) for c in circles]
    bnd = [M(p[0], p[1]) for p in boundary]
    hab = [M(h[0], h[1], size=h[2]) for h in habitats]
    expanded = []
    out = {}
    with contextlib.redirect_stdout(io.StringIO()):
        a = aref.astar((start[0], start[1]), obst, bnd, hab, grid, {}, velocity)
        orig = a.curr_neighbors

        def curr_neighbors(node, bl):
            expanded.append((node.position[0], node.position[1], float(node.pathLen), float(node.f), float(node.cost),
                             float(node.time_stamp)))
            return orig(node, bl)
        a.curr_neighbors = curr_neighbors
        try:
            r = a.astar(path_len_limit, list(weights), {})
        except Exception as ex:       # AttributeError (no time bin), TypeError (no cell), IndexError (top-n)
            out["raised"] = type(ex).__name__
            r = None
    out["expanded"] = np.array(expanded, dtype=np.float64).reshape(-1, 6)
    out["n_visited"] = int(a.visited_nodes.sum())
    c = aref.Polygon([(p[0], p[1]) for p in boundary]).centroid.coords[0]
    out["centroid"] = np.array(c, dtype=np.float64)
    if r is not None:
        nodes = r["node"]
        out["nodes"] = np.array([[n.position[0], n.position[1], float(n.pathLen), float(n.time_stamp), float(n.cost),
                                  float(n.f)] for n in nodes], dtype=np.float64)
        out["cost"] = float(r["cost"])
        out["cost_list"] = np.array(r["cost list"], dtype=np.float64)
        kept = {(p.x, p.y) for p in r["path"]}
        out["smooth_keep"] = np.array([(n.position[0], n.position[1]) in kept for n in nodes], dtype=np.uint8)
        assert out["smooth_keep"].sum() == len(r["path"]) == r["path length"]
        out["smooth_path"] = np.array([[p.x, p.y, p.traj_time_stamp] for p in r["path"]], dtype=np.float64)
    elif "raised" not in out:
        out["exhausted"] = True      # open list ran empty: astar() returns None
    return out


# ---------------------------------------------------------------------------------------------
# Timing the unmodified planner (bench.py --impl reference): no tracing, Python's own Mersenne Twister
# ---------------------------------------------------------------------------------------------
def timed_exploring(ref, rrt, initial, habitats, *, iterations, seed, bin_interval=5, v=2, shark_interval=50,
                    max_plan_time=10.0, max_traj_time=500.0, weights=(-3, -3, -4), plot_interval=0.5):
    """RRT.exploring (/root/reference/path_planning/rrt_dubins.py:92-176) in its default mode for exactly `iterations`
    steer calls (the wall-clock budget is replaced by BudgetClock, nothing else is touched) on `random.Random(seed)`.
    Returns (result dict or None, steer calls, seconds spent inside exploring)."""
    import random as _random
    import time as _time
    mod = ref.rrt_dubins
    clock = BudgetClock(iterations)
    saved = (mod.random, mod.time)
    orig_cc = rrt.check_collision

    def check_collision(mps, obstacles):          # exactly one call per steer call (:141-143): the iteration counter
        clock.done += 1
        return orig_cc(mps, obstacles)

    rrt.check_collision = check_collision
    mod.random, mod.time = _random.Random(seed), clock
    t0 = _time.perf_counter()
    try:
        try:
            res = rrt.exploring(initial, habitats, plot_interval, bin_interval, v, shark_interval, traj_time_stamp=True,
                                max_plan_time=max_plan_time, max_traj_time=max_traj_time, plan_time=True,
                                weights=list(weights))
        except TypeError:
            res = None                            # no node reached the horizon (rrt_dubins.py:174)
    finally:
        dt = _time.perf_counter() - t0
        mod.random, mod.time = saved
        del rrt.check_collision
    return res, clock.done, dt


# ---------------------------------------------------------------------------------------------
# RRT.replanning (/root/reference/path_planning/rrt_dubins.py:51-90) under the harness
# ---------------------------------------------------------------------------------------------
class _RandomProxy:
    """`random` stand-in whose player is swapped for every exploring call of a replanning run"""

    def __init__(self):
        self.player = None

    def uniform(self, a, b):
        return self.player.uniform(a, b)

    def random(self):
        return self.player.random()


def traced_replanning(ref, rrt, start, habitats, plan_time_budget, traj_time_length, replan_time_interval, weight, *,
                      iterations, seed):
    """Run the unmodified RRT.replanning with every inner exploring call k = 0, 1, ... limited to `iterations` steer
    calls on the slot-addressed stream of seed + k.  Returns (traj, time_dict, cost, segments) where segments[k] holds
    the initial state of call k, whether that object had a live .parent (a node of the previous tree: the reference
    then walks on into the old tree, SURVEY.md section 8a), the call's result cost and its first-interval points."""
    mod = ref.rrt_dubins
    proxy = _RandomProxy()
    clock = BudgetClock(iterations)
    saved = (mod.random, mod.time)
    segs = []
    orig_steer, orig_cc, orig_expl = rrt.steer, rrt.check_collision, rrt.exploring

    def steer(mps, *a, **k):
        proxy.player.begin_steer()
        try:
            return orig_steer(mps, *a, **k)
        finally:
            proxy.player.end_steer()

    def check_collision(mps, obstacles):
        clock.done += 1
        return orig_cc(mps, obstacles)

    def exploring(initial, *a, **k):
        clock.done = 0
        proxy.player = StreamPlayer(seed=seed + len(segs))
        seg = {"initial": (initial.x, initial.y, initial.theta, initial.traj_time_stamp, initial.length),
               "has_parent": initial.parent is not None, "max_traj_time": k.get("max_traj_time")}
        segs.append(seg)
        res = orig_expl(initial, *a, **k)
        seg["cost"] = [res["cost"][0]] + list(res["cost"][1])
        seg["path_length"] = res["path length"]
        first = res["path"][1][list(res["path"][1].keys())[0]]
        seg["first_interval"] = path_to_array(first)
        seg["n_path"] = len(res["path"][0])
        return res

    rrt.steer, rrt.check_collision, rrt.exploring = steer, check_collision, exploring
    mod.random, mod.time = proxy, clock
    try:
        traj, time_dict, cost = rrt.replanning(start, habitats, plan_time_budget, traj_time_length, replan_time_interval, weight)
    finally:
        mod.random, mod.time = saved
        del rrt.steer, rrt.check_collision, rrt.exploring
    return traj, time_dict, cost, segs
