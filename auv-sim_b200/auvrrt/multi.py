"""Multi-GPU driver: planning queries are independent (own start, seed, tree; read-only shared map),
so they are sharded contiguously across ranks with NO data-path collective; one collective at the
end gathers the fixed-size plan records (the "final min-cost plan gather" of the north star).
On GPUs (`plan_sharded_device`) the records stay in HBM from the planner kernel to the NCCL gather, the global
minimum is two 8-byte MIN all-reduces, and only the winner's path is re-created (on its owner) and broadcast.

One process per GPU, torch.distributed for the plumbing: backend "nccl" on GPUs (NVLink / NVSwitch),
"gloo" on CPU for the host-logic tests.  The gather payload is 96 bytes per query.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist

from .api import RECORD_DTYPE


def shard_range(n_queries: int, rank: int, world: int):
    """contiguous shard [lo, hi) of rank `rank`; the first n % world ranks get one extra query"""
    base, extra = divmod(int(n_queries), int(world))
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def _comm_device():
    return torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")


def gather_records(local: np.ndarray, n_queries: int, dtype=None) -> np.ndarray:
    """all-gather the per-query records of every rank, in global query order.
    `local` is this rank's structured array (RECORD_DTYPE unless `dtype` says otherwise) for its shard_range()."""
    RECORD_DTYPE = np.dtype(dtype) if dtype is not None else globals()["RECORD_DTYPE"]
    world, rank = dist.get_world_size(), dist.get_rank()
    dev = _comm_device()
    sizes = [shard_range(n_queries, r, world) for r in range(world)]
    cap = max(hi - lo for lo, hi in sizes)
    buf = torch.zeros((cap, RECORD_DTYPE.itemsize), dtype=torch.uint8)
    lo, hi = sizes[rank]
    assert len(local) == hi - lo, (len(local), lo, hi)
    if hi > lo:
        buf[:hi - lo] = torch.from_numpy(np.ascontiguousarray(local).view(np.uint8).reshape(hi - lo, -1))
    buf = buf.to(dev)
    out = torch.empty((world, cap, RECORD_DTYPE.itemsize), dtype=torch.uint8, device=dev)
    dist.all_gather_into_tensor(out.view(-1), buf.view(-1)) if dev.type == "cuda" else dist.all_gather(
        list(out.unbind(0)), buf)
    out = out.cpu().numpy()
    parts = [out[r, :h - l].reshape(-1).view(RECORD_DTYPE) for r, (l, h) in enumerate(sizes)]
    return np.concatenate(parts) if parts else np.zeros(0, RECORD_DTYPE)


def _orderable(cost: np.ndarray) -> np.ndarray:
    """float64 -> uint64 whose unsigned order equals the float order (NaN excluded)"""
    b = np.asarray(cost, dtype=np.float64).view(np.uint64)
    return np.where(b >> np.uint64(63), ~b, b | np.uint64(1 << 63))


def global_best(local: np.ndarray, lo: int) -> int:
    """global query index of the minimum-cost successful plan over all ranks (-1 if none).
    Every rank contributes its local minimum as (orderable cost bits, global index); the tiny
    all-gather is reduced identically on every rank, ties going to the lowest index -- the same rule
    as the reference's strict `<` (rrt_dubins.py:169)."""
    dev = _comm_device()
    ok = local["status"] == 0
    if ok.any():
        keys = _orderable(np.where(ok, local["cost"][:, 0], np.inf))
        j = int(np.lexsort((np.arange(len(local)), keys))[0])
        key, idx = int(keys[j]), lo + j
    else:
        key, idx = (1 << 64) - 1, -1
    mine = torch.tensor([key >> 32, key & 0xFFFFFFFF, idx], dtype=torch.int64, device=dev)
    world = dist.get_world_size()
    allc = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(allc, mine)
    c = torch.stack(allc).cpu().numpy()
    c = c[c[:, 2] >= 0]
    if len(c) == 0:
        return -1
    order = np.lexsort((c[:, 2], c[:, 1], c[:, 0]))
    return int(c[order[0], 2])


# ---------------------------------------------------------------------------------------------------------------
# Device-resident path (NCCL): records never leave HBM before the gather
# ---------------------------------------------------------------------------------------------------------------
_REC_BYTES = RECORD_DTYPE.itemsize                 # 96
_COST0_F64 = RECORD_DTYPE.fields["cost"][1] // 8   # cost[0] as the n-th double of a record
_INF_KEY = 0x7FF0000000000000                      # orderable key of +inf


def orderable_key_i64(cost_f64: torch.Tensor) -> torch.Tensor:
    """float64 tensor -> int64 tensor whose signed order equals the float order (no NaN)"""
    b = cost_f64.contiguous().view(torch.int64)
    return b ^ ((b >> 63) & 0x7FFFFFFFFFFFFFFF)


def local_min_key(records_dev: torch.Tensor, lo: int):
    """(orderable key of the minimum cost over this shard's successful plans, global index of its first occurrence);
    both int64 scalars on the device; (key(+inf), INT64_MAX) when no plan succeeded"""
    n = records_dev.shape[0]
    dev = records_dev.device
    big = torch.iinfo(torch.int64).max
    if n == 0:
        return (torch.tensor(_INF_KEY, dtype=torch.int64, device=dev), torch.tensor(big, dtype=torch.int64, device=dev))
    status = records_dev.view(torch.int32).view(n, _REC_BYTES // 4)[:, 0]
    cost0 = records_dev.view(torch.float64).view(n, _REC_BYTES // 8)[:, _COST0_F64]
    key = orderable_key_i64(torch.where(status == 0, cost0, torch.full_like(cost0, float("inf"))))
    kmin = key.min()
    idx = torch.where(key == kmin, torch.arange(n, device=dev, dtype=torch.int64) + lo, torch.full((n,), big, device=dev, dtype=torch.int64)).min()
    idx = torch.where(kmin == _INF_KEY, torch.full_like(idx, big), idx)
    return kmin, idx


def plan_sharded_device(env, starts, seeds, params, precision="f32", want_path=True, planner=None):
    """Config 5: all queries sharded contiguously over the ranks of the default (NCCL) process group, planned with
    everything resident in HBM, then
      1. one all_gather_into_tensor of the 96-byte plan records (every rank ends with all records, global order),
      2. the global minimum-cost plan by two 8-byte MIN all-reduces: the orderable cost key, then the lowest global
         query index among the ranks that hold that cost (the reference's strict `<`: the first minimum wins),
      3. the winner's path re-created on its owner rank from (start, seed, chain) and broadcast.
    Returns dict(records = uint8 tensor [Q, 96] on this rank's GPU, best = global index or -1, path = rows or None,
    local = this rank's DevicePlanner)."""
    from . import api
    from .device import DevicePlanner
    world, rank = dist.get_world_size(), dist.get_rank()
    starts = np.asarray(starts, dtype=np.float64).reshape(-1, 5)
    seeds = np.asarray(seeds, dtype=np.uint64)
    Q = len(seeds)
    sizes = [shard_range(Q, r, world) for r in range(world)]
    lo, hi = sizes[rank]
    cap = max(h - l for l, h in sizes)
    dev = torch.device("cuda", env.device)
    if planner is None:
        planner = DevicePlanner(env, params, precision, max(cap, 1), want_chain=True)
    planner.set_queries(starts[lo:hi], seeds[lo:hi])
    if hi > lo:
        planner.launch()
    local = planner.records[:hi - lo]
    # 1. gather (padded to the largest shard so that one collective of equal-size blocks does it)
    gathered = torch.empty((world, cap, _REC_BYTES), dtype=torch.uint8, device=dev)
    if cap > hi - lo:
        planner.records[hi - lo:cap].zero_()
    dist.all_gather_into_tensor(gathered.view(-1), planner.records[:cap].reshape(-1))
    if all(h - l == cap for l, h in sizes):
        allrec = gathered.view(world * cap, _REC_BYTES)[:Q]
    else:
        allrec = torch.cat([gathered[r, :h - l] for r, (l, h) in enumerate(sizes)], 0)
    # 2. global minimum, first index on ties
    kmin, idx = local_min_key(local, lo)
    gk = kmin.clone()
    dist.all_reduce(gk, op=dist.ReduceOp.MIN)
    gi = torch.where(kmin == gk, idx, torch.full_like(idx, torch.iinfo(torch.int64).max))
    dist.all_reduce(gi, op=dist.ReduceOp.MIN)
    best = int(gi.item())
    if best == torch.iinfo(torch.int64).max:
        best = -1
    # 3. the winner's path, from its owner
    path = None
    if want_path and best >= 0:
        owner = next(r for r, (l, h) in enumerate(sizes) if l <= best < h)
        n_rows = torch.zeros(1, dtype=torch.int64, device=dev)
        rows_dev = None
        if rank == owner:
            j = best - lo
            rec = planner.records[j:j + 1].cpu().numpy().view(RECORD_DTYPE).reshape(-1)
            import copy
            pp = copy.copy(params)
            pp.path_cap = 34 * (int(rec["depth"][0]) + 1)
            # re-create the path with the evaluator of the kernel that planned it (group 0: one thread per tree from
            # 32768 queries on, no paths being written)
            if pp.group == 0 and hi - lo >= 32768 and pp.mode != 3 and planner.path is None:
                pp.group = 1
            chain = planner.chain[j:j + 1].cpu().numpy().view(np.uint32)
            rows, n_path = api.materialize(env, starts[best:best + 1], seeds[best:best + 1], chain, rec["depth"], pp, precision)
            rows_dev = torch.from_numpy(np.ascontiguousarray(rows[0, :n_path[0]])).to(dev)
            n_rows[0] = int(n_path[0])
        dist.broadcast(n_rows, src=owner)
        if rank != owner:
            rows_dev = torch.empty((int(n_rows.item()), 6), dtype=torch.float64, device=dev)
        dist.broadcast(rows_dev, src=owner)
        path = rows_dev.cpu().numpy()
    return {"records": allrec, "best": best, "path": path, "local": planner, "shard": (lo, hi)}


def plan_sharded(env, starts, seeds, params, precision="f32", plan_fn=None):
    """Run all queries sharded over the ranks of the default process group and return
    (records for ALL queries in global order, index of the global minimum-cost plan).
    `plan_fn(env, starts, seeds, params, precision) -> {"records": ...}` defaults to the CUDA
    planner (auvrrt.api.plan_batch); tests inject a stand-in to exercise the host logic on gloo."""
    if plan_fn is None and dist.get_backend() == "nccl":
        r = plan_sharded_device(env, starts, seeds, params, precision, want_path=False)
        return r["records"].cpu().numpy().reshape(-1).view(RECORD_DTYPE), r["best"]
    if plan_fn is None:
        from . import api
        plan_fn = api.plan_batch
    world, rank = dist.get_world_size(), dist.get_rank()
    starts = np.asarray(starts, dtype=np.float64).reshape(-1, 5)
    seeds = np.asarray(seeds, dtype=np.uint64)
    Q = len(seeds)
    lo, hi = shard_range(Q, rank, world)
    local = plan_fn(env, starts[lo:hi], seeds[lo:hi], params, precision)["records"] if hi > lo else np.zeros(0, RECORD_DTYPE)
    allrec = gather_records(local, Q)
    best = global_best(local, lo)
    return allrec, best


def gym_plan_sharded(boundary, obstacles, starts, goals, seeds, max_step=200, run_fn=None, **batch_kw):
    """Planner_RRT.planning for every episode, episodes sharded contiguously over the ranks; returns the
    records of ALL episodes in global order (one all-gather of 88-byte records, no data-path collective).
    `run_fn(boundary, obstacles, starts, goals, seeds, max_step, **batch_kw) -> records` defaults to the CUDA
    planner (auvrrt.gym.GymBatch); tests inject a stand-in to exercise the host logic on gloo."""
    from .gym import GYM_RECORD_DTYPE
    if run_fn is None:
        def run_fn(boundary, obstacles, starts, goals, seeds, max_step, **kw):
            from .gym import GymBatch
            kw.setdefault("node_cap", max_step + 1)
            b = GymBatch(boundary, obstacles, len(seeds), **kw)
            try:
                b.reset(starts, goals, seeds)
                return b.plan(max_step)
            finally:
                b.close()
    world, rank = dist.get_world_size(), dist.get_rank()
    starts = np.asarray(starts, dtype=np.float64).reshape(-1, 3)
    goals = np.asarray(goals, dtype=np.float64).reshape(-1, 2)
    seeds = np.asarray(seeds, dtype=np.uint64)
    Q = len(seeds)
    lo, hi = shard_range(Q, rank, world)
    local = run_fn(boundary, obstacles, starts[lo:hi], goals[lo:hi], seeds[lo:hi], max_step, **batch_kw) if hi > lo \
        else np.zeros(0, GYM_RECORD_DTYPE)
    return gather_records(local, Q, GYM_RECORD_DTYPE)


def astar_sharded(env, queries, run_fn=None, **batch_kw):
    """lattice-A* queries sharded contiguously over the ranks -> (records of ALL queries in global order, index of
    the minimum-cost successful query, -1 if none; ties to the lowest index).  `env` is this rank's AstarEnv."""
    from .astar import ASTAR_QUERY_DTYPE, ASTAR_RECORD_DTYPE
    if run_fn is None:
        def run_fn(env, q, **kw):
            from .astar import astar_batch
            kw.setdefault("want_paths", False)
            return astar_batch(env, q, **kw)["records"]
    world, rank = dist.get_world_size(), dist.get_rank()
    queries = np.ascontiguousarray(queries, dtype=ASTAR_QUERY_DTYPE)
    Q = len(queries)
    lo, hi = shard_range(Q, rank, world)
    local = run_fn(env, queries[lo:hi], **batch_kw) if hi > lo else np.zeros(0, ASTAR_RECORD_DTYPE)
    allrec = gather_records(local, Q, ASTAR_RECORD_DTYPE)
    ok = allrec["status"] == 0
    best = -1
    if ok.any():
        keys = _orderable(np.where(ok, allrec["cost"], np.inf))
        best = int(np.lexsort((np.arange(Q), keys))[0])
    return allrec, best
