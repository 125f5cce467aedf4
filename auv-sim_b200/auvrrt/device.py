"""Device-resident entry points on torch tensors.

torch is plumbing here (device memory, streams, torch.distributed); the arithmetic is in the
kernels behind the `_dev` functions of include/auvrrt.h.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

import copy

from . import _lib
from ._lib import F32, F64, PlanRecord, check, lib
from .api import RECORD_DTYPE, Env, _f64, _p, _prec, flat_polys, plan_group


def _rdtype(precision):
    return torch.float32 if _prec(precision) == F32 else torch.float64


def _stream_ptr(stream=None):
    s = stream if stream is not None else torch.cuda.current_stream()
    return C.c_void_p(s.cuda_stream)


def _vp(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


class DevicePlanner:
    """Batched RRT.exploring with everything resident in HBM: starts/seeds in, 96-byte records
    (+ chains of stream positions) out.  One instance owns the tree workspace.  `group` is the planner the last
    launch ran (api.plan_group), the evaluator best_paths re-creates its paths with."""

    def __init__(self, env: Env, params, precision="f32", max_queries=4096, want_chain=True, want_path=False):
        self.env, self.params, self.prec = env, params, _prec(precision)
        self.dev = torch.device("cuda", env.device)
        self.rdtype = _rdtype(precision)
        wsb = lib().auvrrt_plan_workspace_bytes_q(env.handle, C.byref(params), self.prec, int(max_queries))
        if wsb < 0:
            raise _lib.AuvrrtError(lib().auvrrt_last_error().decode())
        self.workspace = torch.empty(int(wsb), dtype=torch.uint8, device=self.dev)
        self.Q = int(max_queries)
        self.starts = torch.zeros((self.Q, 5), dtype=self.rdtype, device=self.dev)
        self.seeds = torch.zeros(self.Q, dtype=torch.int64, device=self.dev)      # uint64 bit patterns
        self.records = torch.zeros((self.Q, C.sizeof(PlanRecord)), dtype=torch.uint8, device=self.dev)
        ccap = max(params.chain_cap, 1)
        self.chain = torch.zeros((self.Q, ccap), dtype=torch.int32, device=self.dev) if (want_chain or want_path) else None
        self.path = (torch.zeros((self.Q, params.path_cap, 6), dtype=self.rdtype, device=self.dev)
                     if want_path and params.path_cap > 0 else None)
        self.group = None

    def set_queries(self, starts: np.ndarray, seeds: np.ndarray):
        q = len(seeds)
        assert q <= self.Q
        self.starts[:q].copy_(torch.from_numpy(np.asarray(starts, dtype=np.float64)).to(self.rdtype))
        self.seeds[:q].copy_(torch.from_numpy(np.asarray(seeds, dtype=np.uint64).view(np.int64)))
        self.n = q

    def launch(self, stream=None):
        """enqueue one pass over the current queries on `stream`; no synchronisation"""
        group = plan_group(self.params, self.n, self.path is not None)
        check(lib().auvrrt_plan_batch_dev(self.env.handle, _vp(self.starts), _vp(self.seeds), self.n,
                                          C.byref(self.params), self.prec, _vp(self.workspace),
                                          self.workspace.numel(), _vp(self.records), _vp(self.chain),
                                          _vp(self.path), None, _stream_ptr(stream)))
        self.group = group

    def best_paths(self, mission_off, path_cap, stream=None):
        """Each mission's best plan of the last launch and its path, enqueued on `stream` (default: the current stream)
        without synchronising.  mission_off int64 [M + 1] on the device: mission m is queries
        [mission_off[m], mission_off[m + 1]) (plan_best_dev).  Returns dict(best int64 [M] (query index or -1),
        cost float64 [M] (cost[0] or +inf), path [M, path_cap, 6] in the precision's float type, n_path int32 [M])
        as device tensors: row m of path re-creates plan best[m] (materialize_dev)."""
        if self.group is None:
            raise ValueError("best_paths: nothing launched yet")
        if self.chain is None:
            raise ValueError("best_paths: the planner was created without chains (want_chain=False)")
        n = self.n
        with torch.cuda.stream(stream if stream is not None else torch.cuda.current_stream(self.dev)):
            best, cost = plan_best_dev(self.records[:n], mission_off, stream=stream)
            pp = copy.copy(self.params)
            pp.group = self.group
            path, n_path = materialize_dev(self.env, self.starts[:n], self.seeds[:n], self.records[:n], self.chain[:n],
                                           best, pp, self.prec, path_cap, stream=stream)
        return {"best": best, "cost": cost, "path": path, "n_path": n_path}

    def records_numpy(self):
        return self.records[:self.n].cpu().numpy().view(RECORD_DTYPE).reshape(-1)


def plan_best_dev(records, mission_off, out_best=None, out_cost=None, stream=None):
    """Each mission's best plan (RRT.exploring with replicas: the least cost[0] of the records with status OK, depth
    >= 0 and a cost that is not NaN; the lowest index on ties, -0.0 == +0.0), enqueued on `stream` (default: the
    current stream) without synchronising or allocating in the library.  records uint8 [Q, 96] (plan records) and
    mission_off int64 [M + 1] on one device; mission m is records [mission_off[m], mission_off[m + 1]), offsets
    clamped into [0, Q].  out_best int64 [M] and out_cost float64 [M], allocated when None.
    Returns (out_best: global record index or -1, out_cost: its cost[0] or +inf)."""
    dev = records.device if isinstance(records, torch.Tensor) else None
    Q = records.shape[0] if isinstance(records, torch.Tensor) and records.dim() == 2 else -1
    _need("records", records, (torch.uint8,), (Q, C.sizeof(PlanRecord)), dev)
    M = mission_off.shape[0] - 1 if isinstance(mission_off, torch.Tensor) and mission_off.dim() == 1 else -2
    _need("mission_off", mission_off, (torch.int64,), (M + 1,), dev)
    if out_best is None:
        out_best = torch.empty(max(M, 0), dtype=torch.int64, device=dev)
    if out_cost is None:
        out_cost = torch.empty(max(M, 0), dtype=torch.float64, device=dev)
    _need("out_best", out_best, (torch.int64,), (max(M, 0),), dev)
    _need("out_cost", out_cost, (torch.float64,), (max(M, 0),), dev)
    check(lib().auvrrt_plan_best_dev(_vp(records), Q, _vp(mission_off), M, _vp(out_best), _vp(out_cost),
                                     _stream_on(dev, stream)))
    return out_best, out_cost


def materialize_dev(env: Env, starts, seeds, records, chain, pick, params, precision, path_cap, out=None, out_n=None,
                    stream=None):
    """api.materialize on device tensors through a pick list, enqueued on `stream` (default: the current stream)
    without synchronising: row m of the output re-creates plan pick[m] of one plan_batch_dev launch of Q queries, with
    the depth of its record.  starts [Q, 5] in the precision's float type, seeds int64 / uint64 [Q], records uint8
    [Q, 96], chain int32 / uint32 [Q, chain_cap], pick int64 [M]; params.group must name the planner that ran
    (api.plan_group of that launch; 0 is refused); params.path_cap is replaced by path_cap.
    out [M, path_cap, 6] in the precision's float type and out_n int32 [M], allocated when None.  n_path is the full
    row count (only path_cap rows are written); pick -1 gives 0, another pick outside [0, Q) or a depth outside
    [0, chain_cap] gives -1, and no row.  Returns (out, out_n)."""
    dev = torch.device("cuda", env.device)
    prec = _prec(precision)
    rdt = _rdtype(prec)
    Q = starts.shape[0] if isinstance(starts, torch.Tensor) and starts.dim() == 2 else -1
    _need("starts", starts, (rdt,), (Q, 5), dev)
    _need("seeds", seeds, (torch.int64, torch.uint64), (Q,), dev)
    _need("records", records, (torch.uint8,), (Q, C.sizeof(PlanRecord)), dev)
    _need("chain", chain, (torch.int32, torch.uint32), (Q, max(params.chain_cap, 1)), dev)
    M = pick.shape[0] if isinstance(pick, torch.Tensor) and pick.dim() == 1 else -1
    _need("pick", pick, (torch.int64,), (M,), dev)
    path_cap = int(path_cap)
    if path_cap < 1:
        raise ValueError("path_cap must be >= 1, got %d" % path_cap)
    if out is None:
        out = torch.empty((M, path_cap, 6), dtype=rdt, device=dev)
    if out_n is None:
        out_n = torch.empty(M, dtype=torch.int32, device=dev)
    _need("out", out, (rdt,), (M, path_cap, 6), dev)
    _need("out_n", out_n, (torch.int32,), (M,), dev)
    pp = copy.copy(params)
    pp.path_cap = path_cap
    check(lib().auvrrt_materialize_dev(env.handle, _vp(starts), _vp(seeds), _vp(records), _vp(chain), Q, _vp(pick), M,
                                       C.byref(pp), prec, _vp(out), _vp(out_n), _stream_on(dev, stream)))
    return out, out_n


def nn_dev(tree_x, tree_y, qx, qy, out_idx, scratch, precision, stream=None):
    check(lib().auvrrt_nn_dev(_vp(tree_x), _vp(tree_y), tree_x.numel(), _vp(qx), _vp(qy), qx.numel(),
                              _prec(precision), _vp(scratch), scratch.numel(), _vp(out_idx), _stream_ptr(stream)))


def nn_scratch(nq, device):
    return torch.empty(int(lib().auvrrt_nn_scratch_bytes(int(nq))), dtype=torch.uint8, device=device)


def edges_dubins_dev(env: Env, q0, q1, rho, W, out_safe, out_word, out_length, precision, stream=None):
    check(lib().auvrrt_edges_dubins_dev(env.handle, _vp(q0), _vp(q1), q0.shape[0], float(rho), int(W),
                                        _prec(precision), _vp(out_safe), _vp(out_word), _vp(out_length),
                                        _stream_ptr(stream)))


def edges_dubins_cost_dev(env: Env, q0, q1, rho, W, velocity, w3, out_safe, out_word, out_length, out_cost, precision, stream=None):
    check(lib().auvrrt_edges_dubins_cost_dev(env.handle, _vp(q0), _vp(q1), q0.shape[0], float(rho), int(W), float(velocity),
                                             float(w3), _prec(precision), _vp(out_safe), _vp(out_word), _vp(out_length),
                                             _vp(out_cost), _stream_ptr(stream)))


def edges_arc_cost_dev(env: Env, parents, seeds, params5, w3, out_safe, out_counts, out_leaf, out_cost, precision, stream=None):
    p = (C.c_double * 5)(*[float(x) for x in params5])
    check(lib().auvrrt_edges_arc_cost_dev(env.handle, _vp(parents), _vp(seeds), parents.shape[0], p, float(w3),
                                          _prec(precision), _vp(out_safe), _vp(out_counts), _vp(out_leaf), _vp(out_cost),
                                          _stream_ptr(stream)))


def edges_arc_dev(env: Env, parents, seeds, params5, out_safe, out_counts, out_leaf, precision, stream=None):
    p = (C.c_double * 5)(*[float(x) for x in params5])
    check(lib().auvrrt_edges_arc_dev(env.handle, _vp(parents), _vp(seeds), parents.shape[0], p,
                                     _prec(precision), _vp(out_safe), _vp(out_counts), _vp(out_leaf),
                                     _stream_ptr(stream)))


# ---- vectorised gym_rrt episodes (csrc/gym.cu) -----------------------------------------------------------------

def _need(name, t, dtypes, shape, device):
    if not isinstance(t, torch.Tensor):
        raise ValueError("%s must be a torch tensor, got %s" % (name, type(t).__name__))
    if t.device != device:
        raise ValueError("%s must be on %s, got %s" % (name, device, t.device))
    if t.dtype not in dtypes:
        raise ValueError("%s must be %s, got %s" % (name, " or ".join(str(d) for d in dtypes), t.dtype))
    if tuple(t.shape) != tuple(shape):
        raise ValueError("%s must have shape %s, got %s" % (name, tuple(shape), tuple(t.shape)))
    if not t.is_contiguous():
        raise ValueError("%s must be contiguous" % name)


def _gym_device(batch):
    return torch.device("cuda", batch.device)


def gym_reset_dev(batch, mask, starts, goals, seeds, stream=None):
    """Planner_RRT.__init__ for the episodes of `batch` (a gym.GymBatch) with mask[q] != 0, in place, enqueued on
    `stream` (default: the current stream).  mask: bool or uint8 [Q], or None for every episode (a full reset);
    starts float64 [Q, 3]; goals float64 [Q, 2]; seeds int64 or uint64 [Q] (bit patterns of the uint64 seeds).
    Rows of episodes outside the mask are not read.  A masked reset clears only the cells the episode's previous
    tree occupied, and needs one full reset of the batch before it."""
    dev, Q = _gym_device(batch), batch.Q
    if mask is not None:
        _need("mask", mask, (torch.bool, torch.uint8), (Q,), dev)
    _need("starts", starts, (torch.float64,), (Q, 3), dev)
    _need("goals", goals, (torch.float64,), (Q, 2), dev)
    _need("seeds", seeds, (torch.int64, torch.uint64), (Q,), dev)
    check(lib().auvrrt_gym_reset_dev(batch.handle, _vp(mask), _vp(starts), _vp(goals), _vp(seeds),
                                     _stream_ptr(stream if stream is not None else torch.cuda.current_stream(dev))))


def gym_step_dev(batch, actions, records, stream=None, *, full_candidates=False):
    """One RRTEnv.step for every episode of `batch`, enqueued on `stream`: actions int32 [Q] flat sub-cell ids
    (-1 or an empty cell: nothing happens, no draw), or None for one Planner_RRT.planning step; records uint8
    [Q, 88] (gym.GYM_RECORD_DTYPE rows) or None."""
    dev, Q = _gym_device(batch), batch.Q
    if actions is not None:
        _need("actions", actions, (torch.int32,), (Q,), dev)
    if records is not None:
        _need("records", records, (torch.uint8,), (Q, C.sizeof(_lib.GymRecord)), dev)
    check(lib().auvrrt_gym_step_dev(batch.handle, _vp(actions), 1, int(bool(full_candidates)), _vp(records),
                                    _stream_ptr(stream if stream is not None else torch.cuda.current_stream(dev))))


class _CountsArray:
    """the library's resident counts array as a __cuda_array_interface__ object; it holds the batch so that the
    handle outlives every tensor built on it (until batch.close())"""

    def __init__(self, batch, ptr):
        self.batch = batch
        self.__cuda_array_interface__ = {"shape": (batch.Q, batch.n_subcells), "typestr": "<u2",
                                         "data": (int(ptr), False), "version": 3}


def gym_counts_tensor(batch):
    """Zero-copy torch.uint16 view [Q, n_subcells] of the node count of every sub-cell of every episode
    (RRTEnv.convert_rrt_grid_to_1D_num_of_nodes_only), resident on the device.  It is the library's own array:
    every step and reset writes it in place.  The batch must have been created with track_counts=True."""
    ptr = batch.counts_device_ptr()
    if not ptr:
        raise ValueError("gym_counts_tensor: the batch was created without track_counts")
    return torch.as_tensor(_CountsArray(batch, ptr), device=_gym_device(batch))


# ---- shark-occupancy grids from device-resident tracks (csrc/occupancy.cu) ----------------------------------------

def _stream_on(dev, stream):
    return _stream_ptr(stream if stream is not None else torch.cuda.current_stream(dev))


class SharkOccupancy:
    """SharkOccupancyGrid.convert for fixed cells (polygons in cell_list order), boundary bounds, cell size, bin interval
    and detection range, on tracks that live on the device.  n_bins bins (b * bin_interval, (b + 1) * bin_interval);
    each call takes at most max_sharks tracks and max_points points.  The handle owns its cell tables, candidate-cell
    index and workspace: a call allocates nothing and synchronises nothing (it can be captured in a CUDA graph)."""

    def __init__(self, cell_polys, bounds, cell_size, bin_interval, detect_range, n_bins, max_sharks, max_points,
                 device=0):
        coff, cxy = flat_polys(cell_polys)
        b = _f64(bounds, (4,))
        self.dev = torch.device("cuda", int(device))
        self.C, self.n_bins = len(cell_polys), int(n_bins)
        self.max_sharks, self.max_points = int(max_sharks), int(max_points)
        self._h = C.c_void_p()
        check(lib().auvrrt_occ_create(_p(cxy), _p(coff, C.c_int64), self.C, _p(b), float(cell_size), float(bin_interval),
                                      float(detect_range), self.n_bins, self.max_sharks, self.max_points, int(device),
                                      C.byref(self._h)))
        T, rows, cols = C.c_int(0), C.c_int(0), C.c_int(0)
        check(lib().auvrrt_occ_shape(self._h, C.byref(T), C.byref(rows), C.byref(cols)))
        self.rows, self.cols = rows.value, cols.value

    @property
    def grid_shape(self):
        return self.n_bins, self.rows, self.cols

    def grid_dev(self, tracks, track_off, out=None, env=None, t_occ=None, stream=None):
        """Enqueue one conversion on `stream` (default: the current stream).  tracks float64 [n, 3] (x, y,
        traj_time_stamp of every point, sharks in dict order), track_off int64 [S + 1]; out float64 [n_bins, rows, cols]
        or None; env an api.Env whose probs[T][C] is replaced in place (it needs T == n_bins, the same cells and
        createBinList's bins) or None; t_occ int32 [1] or None, set to createBinList's T for these tracks.  Bins
        b < min(n_bins, t_occ) equal api.occupancy_grid's bit for bit.  Returns `out`."""
        n = tracks.shape[0] if isinstance(tracks, torch.Tensor) and tracks.dim() == 2 else -1
        _need("tracks", tracks, (torch.float64,), (n, 3), self.dev)
        S = track_off.shape[0] - 1 if isinstance(track_off, torch.Tensor) and track_off.dim() == 1 else -1
        _need("track_off", track_off, (torch.int64,), (S + 1,), self.dev)
        if out is not None:
            _need("out", out, (torch.float64,), self.grid_shape, self.dev)
        if t_occ is not None:
            _need("t_occ", t_occ, (torch.int32,), (1,), self.dev)
        if env is not None and not isinstance(env, Env):
            raise ValueError("env must be an auvrrt.api.Env, got %s" % type(env).__name__)
        check(lib().auvrrt_occ_grid_dev(self._h, _vp(tracks), _vp(track_off), S, n, _vp(out),
                                        env.handle if env is not None else None, _vp(t_occ), _stream_on(self.dev, stream)))
        return out

    def close(self):
        if self._h:
            lib().auvrrt_occ_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def env_set_probs_dev(env: Env, probs, stream=None):
    """Replace env's shark-occupancy table with probs (float64 [T, C] on env's device), enqueued on `stream` (default:
    the current stream) without synchronising.  Work that reads env on another stream must be ordered after it."""
    dev = torch.device("cuda", env.device)
    _need("probs", probs, (torch.float64,), env.shape, dev)
    check(lib().auvrrt_env_set_probs_dev(env.handle, _vp(probs), _stream_on(dev, stream)))
