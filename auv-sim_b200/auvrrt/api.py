"""numpy-level wrappers over the host-buffer C ABI (include/auvrrt.h).

Each function marshals flat arrays into libauvrrt.so and returns numpy arrays; the arithmetic all
happens in the CUDA kernels.  Names follow the reference functions they replace
(/root/reference/path_planning/rrt_dubins.py, cost.py).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import F32, F64, PlanParams, PlanRecord, PlanTrace, check, lib

_dp = C.POINTER(C.c_double)


def _f64(a, shape=None):
    a = np.ascontiguousarray(np.asarray(a, dtype=np.float64))
    if shape is not None:
        a = a.reshape(shape)
    return a


def _p(a, ty=C.c_double):
    return a.ctypes.data_as(C.POINTER(ty))


def _prec(precision):
    if precision in ("f32", "fp32", "fast", F32, np.float32):
        return F32
    if precision in ("f64", "fp64", "verify", F64, np.float64):
        return F64
    raise ValueError("precision must be 'f32' or 'f64'")


def device_count():
    return lib().auvrrt_device_count()


def launch_count():
    return int(lib().auvrrt_launch_count())


def stream_u(seed, k, f32u=False):
    return lib().auvrrt_stream_u(int(seed), int(k), int(f32u))


class Env:
    """World model resident in HBM: obstacle circles (obstacle_list order), boundary ring, habitats,
    shark grid {bins, cells, probs} (RRT.__init__, rrt_dubins.py:26-49; createSharkGrid :612-630)."""

    def __init__(self, circles=(), boundary=(), habitats=(), bins=(), cells=(), probs=None, device=0):
        self.circles = _f64(circles, (-1, 3))
        self.boundary = _f64(boundary, (-1, 2))
        self.habitats = _f64(habitats, (-1, 3))
        self.bins = _f64(bins, (-1, 2))
        self.cells = _f64(cells, (-1, 4))
        T, Cn = len(self.bins), len(self.cells)
        probs = _f64(probs if probs is not None else np.zeros((T, Cn)), (T, Cn))
        self.device = int(device)
        self._h = C.c_void_p()
        check(lib().auvrrt_env_create(_p(self.circles), len(self.circles), _p(self.boundary),
                                      len(self.boundary), _p(self.habitats), len(self.habitats),
                                      _p(self.bins), T, _p(self.cells), Cn, _p(probs), self.device,
                                      C.byref(self._h)))

    @classmethod
    def from_map(cls, world: dict, bins=(), probs=None, device=0, with_cells=True):
        return cls(world["circles"], world["boundary"], world["habitats"], bins,
                   world["cells"] if with_cells else (), probs, device)

    @property
    def handle(self):
        return self._h

    @property
    def shape(self):
        """(T, C) of the shark-occupancy table probs[T][C]"""
        return len(self.bins), len(self.cells)

    def set_probs(self, probs):
        """Replace the shark-occupancy table probs[T][C] in place (both precisions' copies; the fp32 copy holds each
        value rounded to nearest, as at creation).  Bins, cells and everything else stay.  Returns when the table is
        written; work that reads the world on another stream must be ordered after it by the caller."""
        T, Cn = self.shape
        a = np.asarray(probs, dtype=np.float64)
        if a.shape != (T, Cn):
            raise ValueError("probs must have shape %s, got %s" % ((T, Cn), a.shape))
        a = np.ascontiguousarray(a)
        check(lib().auvrrt_env_set_probs(self._h, _p(a)))

    def probs(self, precision="f64"):
        """The shark-occupancy table the kernels of `precision` read, as a float64 array [T, C] (the fp32 table
        widened).  Read on the world's internal stream: a refresh enqueued on another stream must be ordered before
        this call by the caller."""
        out = np.zeros(self.shape)
        check(lib().auvrrt_env_get_probs(self._h, _prec(precision), _p(out)))
        return out

    def close(self):
        if self._h:
            lib().auvrrt_env_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# EnvHeader of csrc/env.cuh: 38 ints then 14 doubles
_HEADER_INTS = ["K", "E", "H", "T", "C", "NB", "NP", "NCAND", "convex", "hot_bytes", "total_bytes",
                "off_cx", "off_cy", "off_cr", "off_creff", "off_creff2", "off_px", "off_py",
                "off_hx", "off_hy", "off_hr", "off_hr2", "off_b0", "off_b1",
                "off_brk", "off_piece", "off_c1", "off_cell", "off_probs", "off_xb", "nxb", "off_pfirst",
                "off_grid", "gnx", "gny", "bins_uniform", "off_one", "pad1"]
_HEADER_DOUBLES = ["minx", "miny", "maxx", "maxy", "gx0", "gy0", "gs", "bin_s0", "bin_w", "xb0", "xbw", "pad2", "pad3"]


def env_host_blob(circles=(), boundary=(), habitats=(), bins=(), cells=(), probs=None, precision="f32"):
    """The flattened world model as the kernels read it, built on the host (no device needed): returns
    (header dict, raw bytes as a uint8 array).  Used by the CPU-only tests of the classification grid and the
    shark-cell index."""
    circles, boundary, habitats = _f64(circles, (-1, 3)), _f64(boundary, (-1, 2)), _f64(habitats, (-1, 3))
    bins, cells = _f64(bins, (-1, 2)), _f64(cells, (-1, 4))
    T, Cn = len(bins), len(cells)
    probs = _f64(probs if probs is not None else np.zeros((T, Cn)), (T, Cn))
    args = (_p(circles), len(circles), _p(boundary), len(boundary), _p(habitats), len(habitats), _p(bins), T, _p(cells), Cn,
            _p(probs), _prec(precision))
    n = int(lib().auvrrt_env_host_blob(*args, None, 0))
    if n < 0:
        raise ValueError(lib().auvrrt_last_error().decode())
    raw = np.zeros(n, np.uint8)
    lib().auvrrt_env_host_blob(*args, raw.ctypes.data_as(C.c_void_p), n)
    ni = len(_HEADER_INTS)
    hi = raw[:4 * ni].view(np.int32)
    hd = raw[4 * ni:4 * ni + 8 * len(_HEADER_DOUBLES)].view(np.float64)
    h = {k: int(v) for k, v in zip(_HEADER_INTS, hi)}
    h.update({k: float(v) for k, v in zip(_HEADER_DOUBLES, hd)})
    return h, raw


def nn(tree_xy, queries_xy, precision="f64", device=0):
    """RRT.get_closest_mps for every query: index of the nearest tree node."""
    t = _f64(tree_xy, (-1, 2))
    q = _f64(queries_xy, (-1, 2))
    tx, ty = np.ascontiguousarray(t[:, 0]), np.ascontiguousarray(t[:, 1])
    qx, qy = np.ascontiguousarray(q[:, 0]), np.ascontiguousarray(q[:, 1])
    out = np.zeros(len(q), np.int32)
    check(lib().auvrrt_nn(_p(tx), _p(ty), len(tx), _p(qx), _p(qy), len(q), _prec(precision), device,
                          _p(out, C.c_int32)))
    return out


def steer_arc(parents, u, uoff, params, precision="f64", device=0, wp_cap=32):
    """RRT.steer for n edges on explicit uniform streams.
    -> leaf[n,5], counts[n], waypoints[n,wp_cap,6], used[n], status[n]"""
    parents = _f64(parents, (-1, 5))
    n = len(parents)
    u = _f64(u, (-1,))
    uoff = np.ascontiguousarray(np.asarray(uoff, dtype=np.int64))
    params = _f64(params, (5,))
    leaf = np.zeros((n, 5))
    counts = np.zeros(n, np.int32)
    wp = np.zeros((n, wp_cap, 6))
    used = np.zeros(n, np.int32)
    status = np.zeros(n, np.int32)
    check(lib().auvrrt_steer_arc(_p(parents), n, _p(u), _p(uoff, C.c_int64), _p(params), _prec(precision),
                                 device, _p(leaf), _p(counts, C.c_int32), _p(wp), wp_cap,
                                 _p(used, C.c_int32), _p(status, C.c_int32)))
    return leaf, counts, wp, used, status


def steer_dubins(q0, q1, rho=1.0, W=0, precision="f64", device=0):
    """-> word[n] (255: none), seg[n,3], length[n], waypoints[n,W,3] (None if W < 2)"""
    q0, q1 = _f64(q0, (-1, 3)), _f64(q1, (-1, 3))
    n = len(q0)
    word = np.zeros(n, np.uint8)
    seg = np.zeros((n, 3))
    length = np.zeros(n)
    wp = np.zeros((n, W, 3)) if W >= 2 else None
    check(lib().auvrrt_steer_dubins(_p(q0), _p(q1), n, float(rho), int(W), _prec(precision), device,
                                    _p(word, C.c_uint8), _p(seg), _p(length), _p(wp) if wp is not None else None))
    return word, seg, length, wp


def _ragged(paths, width):
    off = np.zeros(len(paths) + 1, np.int64)
    for i, p in enumerate(paths):
        off[i + 1] = off[i] + len(p)
    flat = (np.concatenate([_f64(p, (-1, width)) for p in paths], axis=0) if len(paths) and off[-1] > 0
            else np.zeros((0, width)))
    return off, np.ascontiguousarray(flat)


def collide(env: Env, paths_xy, precision="f64"):
    """RRT.check_collision for a list of paths (each [k,2]); 1 = safe, 0 = not, 255 = ValueError."""
    off, flat = _ragged(paths_xy, 2)
    out = np.zeros(len(paths_xy), np.uint8)
    check(lib().auvrrt_collide(env.handle, _p(flat), _p(off, C.c_int64), len(paths_xy), _prec(precision),
                               _p(out, C.c_uint8)))
    return out


def collide_points(env: Env, points_xy, precision="f64"):
    """RRT.check_collision_obstacle for every point."""
    pts = _f64(points_xy, (-1, 2))
    out = np.zeros(len(pts), np.uint8)
    check(lib().auvrrt_collide_points(env.handle, _p(pts), len(pts), _prec(precision), _p(out, C.c_uint8)))
    return out


def cost(env: Env, paths_xyt, t_total, weights, bin_mask=None, n_habitats=-1, precision="f64"):
    """cost.habitat_shark_cost_func for a list of paths (each [k,3] = x, y, traj_time_stamp)."""
    off, flat = _ragged(paths_xyt, 3)
    tt = _f64(t_total, (-1,))
    w = _f64(weights, (3,))
    out = np.zeros((len(paths_xyt), 4))
    mask = None if bin_mask is None else np.ascontiguousarray(np.asarray(bin_mask, dtype=np.uint8)).reshape(-1)
    if mask is not None and len(mask) < len(env.bins):       # the library reads one byte per time bin
        raise ValueError("bin_mask needs one entry per time bin (%d), got %d" % (len(env.bins), len(mask)))
    check(lib().auvrrt_cost(env.handle, _p(flat), _p(off, C.c_int64), len(paths_xyt), _p(tt), _p(w),
                            _p(mask, C.c_uint8) if mask is not None else None, int(n_habitats),
                            _prec(precision), _p(out)))
    return out


def cost_point(env: Env, points_xy, visited, tb, weights, precision="f64"):
    pts = _f64(points_xy, (-1, 2))
    vis = np.ascontiguousarray(np.asarray(visited, dtype=np.uint8)).reshape(-1)
    if len(vis) < len(env.habitats):                         # the library reads one byte per habitat
        raise ValueError("visited needs one entry per habitat (%d), got %d" % (len(env.habitats), len(vis)))
    w = _f64(weights, (3,))
    out = np.zeros(len(pts))
    check(lib().auvrrt_cost_point(env.handle, _p(pts), len(pts), _p(vis, C.c_uint8), int(tb), _p(w),
                                  _prec(precision), _p(out)))
    return out


def edges_dubins(env: Env, q0, q1, rho=1.0, W=20, precision="f32"):
    q0, q1 = _f64(q0, (-1, 3)), _f64(q1, (-1, 3))
    n = len(q0)
    safe = np.zeros(n, np.uint8)
    word = np.zeros(n, np.uint8)
    length = np.zeros(n)
    check(lib().auvrrt_edges_dubins(env.handle, _p(q0), _p(q1), n, float(rho), int(W), _prec(precision),
                                    _p(safe, C.c_uint8), _p(word, C.c_uint8), _p(length)))
    return safe, word, length


def edges_dubins_cost(env: Env, q0, q1, rho=1.0, W=20, velocity=1.0, w3=-4.0, precision="f32"):
    """edges_dubins + each edge's share of the path cost over waypoints 1..W-1 (traj_time_stamp = arclength / velocity):
    cost [n][3] = sum of w3 * prob, waypoints inside a habitat, distinct habitats visited"""
    q0, q1 = _f64(q0, (-1, 3)), _f64(q1, (-1, 3))
    n = len(q0)
    safe = np.zeros(n, np.uint8)
    word = np.zeros(n, np.uint8)
    length = np.zeros(n)
    cost = np.zeros((n, 3))
    check(lib().auvrrt_edges_dubins_cost(env.handle, _p(q0), _p(q1), n, float(rho), int(W), float(velocity), float(w3),
                                         _prec(precision), _p(safe, C.c_uint8), _p(word, C.c_uint8), _p(length), _p(cost)))
    return safe, word, length, cost


def edges_arc(env: Env, parents, seeds, params, precision="f32"):
    parents = _f64(parents, (-1, 5))
    n = len(parents)
    seeds = np.ascontiguousarray(np.asarray(seeds, dtype=np.uint64))
    params = _f64(params, (5,))
    safe = np.zeros(n, np.uint8)
    counts = np.zeros(n, np.int32)
    leaf = np.zeros((n, 5))
    check(lib().auvrrt_edges_arc(env.handle, _p(parents), _p(seeds, C.c_uint64), n, _p(params),
                                 _prec(precision), _p(safe, C.c_uint8), _p(counts, C.c_int32), _p(leaf)))
    return safe, counts, leaf


def edges_arc_cost(env: Env, parents, seeds, params, w3, precision="f32"):
    """edges_arc + each edge's share of the path cost over its appended waypoints:
    cost [n][3] = sum of w3 * prob, waypoints inside a habitat, distinct habitats visited"""
    parents = _f64(parents, (-1, 5))
    n = len(parents)
    seeds = np.ascontiguousarray(np.asarray(seeds, dtype=np.uint64))
    params = _f64(params, (5,))
    safe = np.zeros(n, np.uint8)
    counts = np.zeros(n, np.int32)
    leaf = np.zeros((n, 5))
    cost = np.zeros((n, 3))
    check(lib().auvrrt_edges_arc_cost(env.handle, _p(parents), _p(seeds, C.c_uint64), n, _p(params), float(w3),
                                      _prec(precision), _p(safe, C.c_uint8), _p(counts, C.c_int32), _p(leaf), _p(cost)))
    return safe, counts, leaf, cost


def plan_params(iterations, mode=0, bin_interval=5.0, v=2.0, max_traj_time=500.0, dist_to_end=2.0,
                diff_max=0.5, freq=30.0, min_dist=0.5, weights=(-3.0, -3.0, -4.0), chain_cap=96,
                path_cap=0, trace=False, group=0, max_plan_time=5.0, dubins_rho=1.0, dubins_eta=20.0,
                near_radius=15.0, dubins_w=12):
    """mode 3 (Dubins-RRT with best-parent selection) reads dubins_rho / dubins_eta / near_radius / dubins_w"""
    return PlanParams(int(iterations), int(mode), float(bin_interval), float(v), float(max_traj_time),
                      float(dist_to_end), float(diff_max), float(freq), float(min_dist),
                      (C.c_double * 3)(*[float(x) for x in weights]), int(chain_cap), int(path_cap),
                      int(bool(trace)), int(group), float(max_plan_time), float(dubins_rho), float(dubins_eta),
                      float(near_radius), int(dubins_w), 0)


RECORD_DTYPE = np.dtype([("status", "i4"), ("n_nodes", "i4"), ("best_node", "i4"), ("best_iter", "i4"),
                         ("depth", "i4"), ("n_path", "i4"), ("n_cost_evals", "i4"), ("n_waypoints", "i4"),
                         ("n_uniforms", "i8"), ("n_primitives", "i8"), ("cost", "f8", 4),
                         ("path_length", "f8"), ("t_leaf", "f8")])
assert RECORD_DTYPE.itemsize == C.sizeof(PlanRecord)


def plan_batch(env: Env, starts, seeds, params: PlanParams, precision="f32", want_chain=True):
    """RRT.exploring for Q independent queries.
    -> dict(records[Q] structured, chain[Q,chain_cap], path[Q,path_cap,6] | None, trace | None)"""
    starts = _f64(starts, (-1, 5))
    Q = len(starts)
    seeds = np.ascontiguousarray(np.asarray(seeds, dtype=np.uint64))
    assert len(seeds) == Q
    rec = np.zeros(Q, RECORD_DTYPE)
    chain = np.zeros((Q, max(params.chain_cap, 1)), np.uint32) if (want_chain or params.path_cap > 0) else None
    path = np.zeros((Q, params.path_cap, 6)) if params.path_cap > 0 else None
    tr = None
    trace = None
    if params.trace:
        I = params.iterations
        trace = {"parent": np.zeros((Q, I), np.int32), "safe": np.zeros((Q, I), np.uint8),
                 "nwp": np.zeros((Q, I), np.int32), "leaf": np.zeros((Q, I, 5)), "upos": np.zeros((Q, I), np.int64)}
        tr = PlanTrace(_p(trace["parent"], C.c_int32), _p(trace["safe"], C.c_uint8), _p(trace["nwp"], C.c_int32),
                       _p(trace["leaf"]), _p(trace["upos"], C.c_int64))
    check(lib().auvrrt_plan_batch(env.handle, _p(starts), _p(seeds, C.c_uint64), Q, C.byref(params),
                                  _prec(precision), rec.ctypes.data_as(C.POINTER(PlanRecord)),
                                  _p(chain, C.c_uint32) if chain is not None else None,
                                  _p(path) if path is not None else None,
                                  C.byref(tr) if tr is not None else None))
    return {"records": rec, "chain": chain, "path": path, "trace": trace}


def materialize(env: Env, starts, seeds, chain, depth, params: PlanParams, precision="f32"):
    starts = _f64(starts, (-1, 5))
    Q = len(starts)
    seeds = np.ascontiguousarray(np.asarray(seeds, dtype=np.uint64))
    chain = np.ascontiguousarray(np.asarray(chain, dtype=np.uint32)).reshape(Q, max(params.chain_cap, 1))
    depth = np.ascontiguousarray(np.asarray(depth, dtype=np.int32))
    path = np.zeros((Q, params.path_cap, 6))
    n_path = np.zeros(Q, np.int32)
    check(lib().auvrrt_materialize(env.handle, _p(starts), _p(seeds, C.c_uint64), _p(chain, C.c_uint32),
                                   _p(depth, C.c_int32), Q, C.byref(params), _prec(precision), _p(path),
                                   _p(n_path, C.c_int32)))
    return path, n_path


def plan_group(params: PlanParams, Q, with_path=False):
    """The planner auvrrt_plan_batch(_dev) runs for a batch of Q queries: 32, 16 or 8 lanes per tree, or 1 (one thread
    per tree).  with_path: the batch writes paths (an out_path with path_cap > 0).  This is the group
    materialize / device.materialize_dev need to re-create that batch's plans.  Host logic only."""
    g = lib().auvrrt_plan_group(C.byref(params), int(Q), int(bool(with_path)))
    if g < 0:
        raise _lib.AuvrrtError("libauvrrt: %s" % lib().auvrrt_last_error().decode())
    return g


def calibrate_fp32(device=0, iters=4096):
    f, ms = C.c_double(0), C.c_double(0)
    check(lib().auvrrt_calibrate_fp32(device, iters, C.byref(f), C.byref(ms)))
    return f.value, ms.value


def flat_polys(cell_polys):
    """list of polygons (vertex arrays) -> (offsets[C+1] int64, vertices[V, 2] float64), the C ABI's ragged layout"""
    coff = np.zeros(len(cell_polys) + 1, np.int64)
    for i, p in enumerate(cell_polys):
        coff[i + 1] = coff[i] + len(p)
    cxy = _f64(np.concatenate([np.asarray(p, dtype=np.float64).reshape(-1, 2) for p in cell_polys]), (-1, 2)) \
        if len(cell_polys) else np.zeros((0, 2))
    return coff, cxy


def occupancy_grid(cell_polys, bounds, cell_size, bin_interval, detect_range, tracks, device=0):
    """SharkOccupancyGrid.convert: list of cell polygons (vertex arrays, cell_list order), boundary bounds,
    and one [n,3] (x, y, traj_time_stamp) track per shark -> (grid[T, rows, cols], bins[T, 2])"""
    coff, cxy = flat_polys(cell_polys)
    toff = np.zeros(len(tracks) + 1, np.int64)
    for i, t in enumerate(tracks):
        toff[i + 1] = toff[i] + len(t)
    txy = _f64(np.concatenate([np.asarray(t, dtype=np.float64).reshape(-1, 3) for t in tracks]), (-1, 3))
    b = _f64(bounds, (4,))
    T, rows, cols = C.c_int(0), C.c_int(0), C.c_int(0)
    check(lib().auvrrt_occupancy_dims(_p(b), float(cell_size), float(bin_interval), _p(txy), _p(toff, C.c_int64),
                                      len(tracks), C.byref(T), C.byref(rows), C.byref(cols)))
    out = np.zeros((max(T.value, 0), rows.value, cols.value))
    check(lib().auvrrt_occupancy_grid(_p(cxy), _p(coff, C.c_int64), len(cell_polys), _p(b), float(cell_size),
                                      float(bin_interval), float(detect_range), _p(txy), _p(toff, C.c_int64),
                                      len(tracks), device, _p(out), out.size))
    bins = np.array([[i * bin_interval, (i + 1) * bin_interval] for i in range(T.value)], dtype=np.float64).reshape(-1, 2)
    return out, bins
