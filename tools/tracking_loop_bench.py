"""The device end of a tracking-loop step -- each mission's best plan (device.plan_best_dev) and its path
(device.materialize_dev) -- against today's host tail, and the whole step (refresh -> plan -> best -> path) replayed
from one CUDA graph against the same step launched eagerly.

Cases:
  a   one mission x 4096 replicas at config 2 (2048 iterations, fp32, group 0: the warp planner)
  b   4096 missions x 64 replicas, 512 iterations, fp32, group 0 (262,144 queries: the thread-per-tree planner)
  c   the selection alone on 2^20 synthetic records in one mission (the split kernel) and in 4096 missions of 256

Per case one JSON line goes to OUT/r07_tracking_loop.jsonl:
  select_ms, materialize_ms   device time of one call, CUDA events over --reps warmed calls
  select_gbs                  64 bytes per record (the two 32-byte sectors of status / depth and cost[0]) over
                              select_ms, and its share of hbm_gbs, a device-to-device copy of 4 GiB measured in the same
                              run (records of cases a / b fit the 126 MB L2 after the first pass: the rate is L2's)
  device_tail_ms              select + materialize, CUDA events
  host_tail_ms                records .cpu(), numpy argmin per mission, api.materialize, H2D copy of the paths; host
                              clock ending in a synchronise (median of --host-reps)
  step_eager_ms, step_graph_ms  refresh (config 3 tracks, Catalina's 986 cells, 9 bins) -> plan -> best -> path, launched
                              eagerly and replayed from a CUDA graph captured once; CUDA events, blocks alternated
  graph_exact                 the replayed step's best / cost / n_path / rows equal the eager step's bit for bit
and the GPU's name and power limit, read in the same run.  Not bench.py: that measures the flagship planner.

  python tools/tracking_loop_bench.py --out DIR [--reps 50] [--host-reps 5] [--step-reps 5] [--cases a,b,c]
"""
import argparse
import copy
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "auv-sim_b200"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

import bench  # noqa: E402
import occupancy_refresh_bench as orb  # noqa: E402
from auvrrt import api  # noqa: E402
from auvrrt import device as adev  # noqa: E402
from auvrrt.api import RECORD_DTYPE  # noqa: E402

SELECT_BYTES = 64
PATH_CAP = 4096           # 34 rows per edge (the parent + at most 32 waypoints + 1) x 97 plus slack: no path is cut


def hbm_gbs(dev):
    n = 1 << 29                                               # 4 GiB of float64 read and written
    a = torch.empty(n, dtype=torch.float64, device=dev)
    b = torch.empty_like(a)
    b.copy_(a)
    ms = orb.events_ms(lambda: b.copy_(a), 10)
    return 2 * 8 * n / (ms * 1e-3) / 1e9


def host_best(rec, R):
    """numpy per mission (R records each): first minimum of cost[0] over the eligible records"""
    c = rec["cost"][:, 0]
    ok = (rec["status"] == 0) & (rec["depth"] >= 0) & ~np.isnan(c)
    key = np.where(ok, np.where(c == 0, 0.0, c), np.nan).reshape(-1, R)
    has = ok.reshape(-1, R).any(1)
    j = np.nanargmin(np.where(has[:, None], key, 0.0), axis=1)
    return np.where(has, np.arange(len(has)) * R + j, -1)


def host_tail(pl, R, pp, starts, seeds, dev):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    rec = pl.records[:pl.n].cpu().numpy().view(RECORD_DTYPE).reshape(-1)
    chain = pl.chain[:pl.n].cpu().numpy().view(np.uint32)
    best = host_best(rec, R)
    sel = best[best >= 0]
    rows, n_path = api.materialize(pl.env, starts[sel], seeds[sel], chain[sel], rec["depth"][sel], pp, "f32")
    paths = torch.from_numpy(rows).to(dev)
    torch.cuda.synchronize()
    return time.perf_counter() - t0, paths


def loop_case(name, R, M, iters, env, occ, trk, toff, a):
    dev = torch.device("cuda", 0)
    Q = R * M
    starts, seeds = bench.make_queries(0, Q)
    pl = adev.DevicePlanner(env, api.plan_params(iters), "f32", Q, want_chain=True)
    pl.set_queries(starts, seeds)
    off = torch.arange(M + 1, dtype=torch.int64, device=dev) * R
    best = torch.empty(M, dtype=torch.int64, device=dev)
    cost = torch.empty(M, dtype=torch.float64, device=dev)
    path = torch.empty((M, PATH_CAP, 6), dtype=torch.float32, device=dev)
    n_path = torch.empty(M, dtype=torch.int32, device=dev)
    occ.grid_dev(trk, toff, env=env)
    pl.launch()
    pp = copy.copy(pl.params)
    pp.group, pp.path_cap = pl.group, PATH_CAP
    n = pl.n

    def select():
        adev.plan_best_dev(pl.records[:n], off, out_best=best, out_cost=cost)

    def materialize():
        adev.materialize_dev(env, pl.starts[:n], pl.seeds[:n], pl.records[:n], pl.chain[:n], best, pp, "f32", PATH_CAP,
                             out=path, out_n=n_path)

    def tail():
        select()
        materialize()

    for f in (select, materialize, tail):
        f()
    torch.cuda.synchronize()
    sel_ms = orb.events_ms(select, a.reps)
    mat_ms = orb.events_ms(materialize, a.reps)
    tail_ms = orb.events_ms(tail, a.reps)
    # the host tail on the same records, and whether it found the same plans
    host_tail(pl, R, pp, starts, seeds, dev)
    ht = [host_tail(pl, R, pp, starts, seeds, dev) for _ in range(a.host_reps)]
    hb = host_best(pl.records[:n].cpu().numpy().view(RECORD_DTYPE).reshape(-1), R)
    same_best = bool(np.array_equal(hb, best.cpu().numpy()))

    # the whole step: refresh -> plan -> best -> path, eager and from one graph
    def step():
        occ.grid_dev(trk, toff, env=env)
        pl.launch()
        return pl.best_paths(off, PATH_CAP)

    eager = step()
    torch.cuda.synchronize()
    want = {k: v.clone() for k, v in eager.items()}
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = step()
    g.replay()
    torch.cuda.synchronize()
    m = torch.arange(PATH_CAP, device=dev)[None, :] < want["n_path"].clamp(0, PATH_CAP)[:, None]
    exact = bool(torch.equal(out["best"], want["best"]) and torch.equal(out["n_path"], want["n_path"])
                 and torch.equal(out["cost"].view(torch.int64), want["cost"].view(torch.int64))
                 and torch.equal(out["path"][m], want["path"][m]))
    se, sg = [], []
    for _ in range(a.step_reps):
        se.append(orb.events_ms(step, 3))
        sg.append(orb.events_ms(g.replay, 3))
    return {"case": name, "missions": M, "replicas": R, "queries": Q, "iterations": iters, "group": pl.group,
            "path_cap": PATH_CAP, "select_ms": sel_ms, "materialize_ms": mat_ms, "device_tail_ms": tail_ms,
            "select_gbs": SELECT_BYTES * Q / (sel_ms * 1e-3) / 1e9,
            "host_tail_ms": 1e3 * float(np.median([t for t, _ in ht])), "host_reps": a.host_reps,
            "host_same_best": same_best, "step_eager_ms": float(np.median(se)), "step_graph_ms": float(np.median(sg)),
            "step_eager_ms_runs": se, "step_graph_ms_runs": sg, "graph_exact": exact,
            "plans_found": int((want["best"] >= 0).sum().item())}


def select_case(a):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_gpu_best_paths import ref_best, synthetic_records
    dev = torch.device("cuda", 0)
    rs = np.random.RandomState(7)
    Q = 1 << 20
    rec = synthetic_records(Q, rs)
    d = torch.from_numpy(np.ascontiguousarray(rec).view(np.uint8).reshape(Q, -1).copy()).to(dev)
    out = []
    for M in (1, 4096):
        offn = np.arange(M + 1, dtype=np.int64) * (Q // M)
        off = torch.from_numpy(offn).to(dev)
        best = torch.empty(M, dtype=torch.int64, device=dev)
        cost = torch.empty(M, dtype=torch.float64, device=dev)
        adev.plan_best_dev(d, off, out_best=best, out_cost=cost)
        torch.cuda.synchronize()
        wb, wc = ref_best(rec, offn)
        exact = bool(np.array_equal(best.cpu().numpy(), wb) and np.array_equal(cost.cpu().numpy().view(np.int64),
                                                                               wc.view(np.int64)))
        ms = orb.events_ms(lambda: adev.plan_best_dev(d, off, out_best=best, out_cost=cost), a.reps)
        out.append({"case": "c", "missions": M, "records": Q, "select_ms": ms,
                    "select_gbs": SELECT_BYTES * Q / (ms * 1e-3) / 1e9, "exact": exact,
                    "note": "96 MB of records: L2-resident after the first pass"})
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--host-reps", type=int, default=5)
    ap.add_argument("--step-reps", type=int, default=5)
    ap.add_argument("--cases", default="a,b,c")
    a = ap.parse_args()
    if not torch.cuda.is_available() or api.device_count() == 0:
        raise SystemExit("tracking_loop_bench.py: no CUDA device -- the product path has no CPU fallback")
    os.makedirs(a.out, exist_ok=True)
    info = orb.gpu_info()
    info["hbm_gbs"] = hbm_gbs(torch.device("cuda", 0))
    z = np.load(os.path.join(ROOT, "tests", "golden", "occupancy.npz"))
    polys = [z["cell_xy"][z["cell_off"][i]:z["cell_off"][i + 1]] for i in range(len(z["cell_off"]) - 1)]
    bounds = np.asarray(z["bounds"], np.float64)
    world, _, _ = bench.load_world()
    tracks = orb.cases()["config3"]
    n = sum(len(t) for t in tracks)
    occ = adev.SharkOccupancy(polys, bounds, orb.CS, orb.BI, orb.RG, orb.T, len(tracks), n)
    env = api.Env.from_map(world, np.array([[b * orb.BI, (b + 1) * orb.BI] for b in range(orb.T)]),
                           np.zeros((orb.T, len(polys))))
    trk = torch.from_numpy(np.ascontiguousarray(np.concatenate(tracks))).cuda()
    toff = torch.from_numpy(np.concatenate([[0], np.cumsum([len(t) for t in tracks])]).astype(np.int64)).cuda()
    path = os.path.join(a.out, "r07_tracking_loop.jsonl")
    with open(path, "w") as f:
        for c in a.cases.split(","):
            if c == "a":
                rows = [loop_case("a", bench.Q_PER_GPU, 1, bench.ITERS, env, occ, trk, toff, a)]
            elif c == "b":
                rows = [loop_case("b", 64, 4096, 512, env, occ, trk, toff, a)]
            else:
                rows = select_case(a)
            for r in rows:
                r.update(info)
                if "select_gbs" in r:
                    r["select_share_of_hbm"] = r["select_gbs"] / info["hbm_gbs"]
                line = json.dumps(r)
                print(line, flush=True)
                f.write(line + "\n")
    occ.close()
    env.close()


if __name__ == "__main__":
    main()
