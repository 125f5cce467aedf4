"""Refreshing a world's shark-occupancy cost on the device (auvrrt.device.SharkOccupancy.grid_dev(..., env=env))
against the host path it replaces, on the Catalina cells (986 polygons, 10 m lattice, 50 s bins, 50 m detection range,
9 bins).

Cases:
  config3  tests/golden/shark_tracks_raw.npz mapped as tracks_to_shark_dict maps it: 32 sharks x 815 points
  pf       a seeded particle-filter-sized set: 256 random-walk tracks x 4096 points over [0, 470] s

Per case one JSON line goes to OUT/r04_occupancy_refresh.jsonl:
  refresh_ms             device time of one refresh into an env, CUDA events over --refreshes warmed refreshes
  host_path_ms           api.occupancy_grid + the keep_zero_cells dicts (SharkOccupancyGrid.convert) + _world.grid_of +
                         api.Env(...), host clock ending in a synchronise (median of --host-reps), and each part
  plan_ms / refresh_plan_ms  one DevicePlanner.launch at config 2 (4096 queries x 2048 iterations, fp32) alone, and a
                         refresh followed by that launch, CUDA events, blocks of each alternated
  kernel_us              per-kernel device time per refresh from a torch.profiler run of its own
  launches_per_refresh   auvrrt_launch_count delta
  exact                  the refreshed table equals the table of api.occupancy_grid's grid, bit for bit
and the GPU's name and power limit, read in the same run.  Not bench.py: that measures the flagship planner.

  python tools/occupancy_refresh_bench.py --out DIR [--refreshes 200] [--plan-reps 5] [--host-reps 5]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "auv-sim_b200"), os.path.join(ROOT, "auv-sim_b200", "path_planning")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

import _world  # noqa: E402
import bench  # noqa: E402
from auvrrt import api  # noqa: E402
from auvrrt import device as adev  # noqa: E402

CS, BI, RG, T = 10.0, 50.0, 50.0, 9
TRACK_MAP = {"x0": 370.0, "y0": 4.0, "sx": 250.0 / 964.0, "sy": 150.0 / 496.0, "ox": -330.0, "oy": -60.0,
             "frame_dt": 0.03, "time_scale": 20.0}       # sharkOccupancyGrid.CATALINA_TRACK_MAP
KERNELS = ("k_occ_hist", "k_occ_norm", "k_occ_auv", "k_occ_avg", "k_occ_to_env")


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_w"] = float(out.splitlines()[0])
    except Exception as e:  # the number is then reported as unknown, not guessed
        info["power_limit_error"] = repr(e)
    return info


def cases():
    z = np.load(os.path.join(ROOT, "tests", "golden", "shark_tracks_raw.npz"))
    m = TRACK_MAP
    x, y = z["x"].astype(np.float64), z["y"].astype(np.float64)
    t = np.arange(x.shape[1]) * m["frame_dt"] * m["time_scale"]
    config3 = [np.stack([m["ox"] + (x[s] - m["x0"]) * m["sx"], m["oy"] + (y[s] - m["y0"]) * m["sy"], t], 1)
               for s in range(len(x))]
    rs = np.random.RandomState(2024)
    pf = [np.stack([rs.uniform(-330, -80) + np.cumsum(rs.normal(0, 0.6, 4096)),
                    rs.uniform(-60, 90) + np.cumsum(rs.normal(0, 0.6, 4096)), np.linspace(0.0, 470.0, 4096)], 1)
          for _ in range(256)]
    return {"config3": config3, "pf": pf}


def table_of(grid, polys, bounds):
    rc = [(int((p[:, 1].min() - bounds[1]) / CS), int((p[:, 0].min() - bounds[0]) / CS)) for p in polys]
    return np.stack([[g[r, c] for r, c in rc] for g in grid]).reshape(len(grid), len(polys))


def events_ms(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def host_path(polys, bounds, world, tracks, cell_bounds):
    """the four steps a caller needs without a device refresh; -> seconds per step"""
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    grid, bins = api.occupancy_grid(polys, bounds, CS, BI, RG, tracks)
    t1 = time.perf_counter()
    d = {}
    for b, key in enumerate([(i * BI, (i + 1) * BI) for i in range(len(bins))]):     # convert(keep_zero_cells=True)
        d[key] = {cb: float(grid[b, r, c]) for cb, (r, c) in cell_bounds}
    t2 = time.perf_counter()
    b_, cells, probs = _world.grid_of(d)
    t3 = time.perf_counter()
    env = api.Env(world["circles"], world["boundary"], world["habitats"], b_, cells, probs)
    torch.cuda.synchronize()
    t4 = time.perf_counter()
    env.close()
    return {"occupancy_grid": t1 - t0, "dicts": t2 - t1, "grid_of": t3 - t2, "env_create": t4 - t3, "total": t4 - t0}


def run_case(name, tracks, polys, bounds, world, a):
    dev = torch.device("cuda", 0)
    n = sum(len(t) for t in tracks)
    bins = np.array([[b * BI, (b + 1) * BI] for b in range(T)])
    occ = adev.SharkOccupancy(polys, bounds, CS, BI, RG, T, len(tracks), n)
    env = api.Env.from_map(world, bins, np.zeros((T, len(polys))))
    off = np.concatenate([[0], np.cumsum([len(t) for t in tracks])]).astype(np.int64)
    trk = torch.from_numpy(np.ascontiguousarray(np.concatenate(tracks))).to(dev)
    toff = torch.from_numpy(off).to(dev)
    t_occ = torch.zeros(1, dtype=torch.int32, device=dev)

    def refresh():
        occ.grid_dev(trk, toff, env=env)

    occ.grid_dev(trk, toff, env=env, t_occ=t_occ)
    torch.cuda.synchronize()
    grid, gbins = api.occupancy_grid(polys, bounds, CS, BI, RG, tracks)
    exact = bool(int(t_occ.item()) == len(gbins) == T and np.array_equal(env.probs("f64"), table_of(grid, polys, bounds)))
    l0 = api.launch_count()
    refresh()
    launches = api.launch_count() - l0
    for _ in range(10):
        refresh()
    refresh_ms = [events_ms(refresh, a.refreshes) for _ in range(3)]
    # host path
    cell_bounds = [((float(p[:, 0].min()), float(p[:, 1].min()), float(p[:, 0].max()), float(p[:, 1].max())),
                    (int((p[:, 1].min() - bounds[1]) / CS), int((p[:, 0].min() - bounds[0]) / CS))) for p in polys]
    host_path(polys, bounds, world, tracks, cell_bounds)
    hp = [host_path(polys, bounds, world, tracks, cell_bounds) for _ in range(a.host_reps)]
    host = {k: 1e3 * float(np.median([h[k] for h in hp])) for k in hp[0]}
    # config 2 launch alone and after a refresh, same env
    pp = api.plan_params(bench.ITERS)
    planner = adev.DevicePlanner(env, pp, "f32", bench.Q_PER_GPU, want_chain=True)
    starts, seeds = bench.make_queries(0, bench.Q_PER_GPU)
    planner.set_queries(starts, seeds)
    stream = torch.cuda.current_stream()
    for _ in range(3):
        planner.launch(stream)

    def both():
        refresh()
        planner.launch(stream)

    plan, rp = [], []
    for _ in range(a.plan_reps):
        plan.append(events_ms(lambda: planner.launch(stream), 5))
        rp.append(events_ms(both, 5))
    # per-kernel times, a run of its own
    nprof = 50
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(nprof):
            refresh()
        torch.cuda.synchronize()
    kus = {}
    for e in prof.key_averages():
        for k in KERNELS:
            if k in e.key:
                kus[k] = kus.get(k, 0.0) + (getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)) / nprof
    occ.close()
    env.close()
    return {"case": name, "sharks": len(tracks), "points": n, "bins": T, "cells": len(polys),
            "grid": list(occ.grid_shape), "refreshes_timed": a.refreshes,
            "refresh_ms": float(np.median(refresh_ms)), "refresh_ms_runs": refresh_ms,
            "host_path_ms": host, "host_reps": a.host_reps,
            "plan_config2": {"queries": bench.Q_PER_GPU, "iterations": bench.ITERS, "precision": "f32",
                             "plan_ms": float(np.median(plan)), "refresh_plan_ms": float(np.median(rp)),
                             "plan_ms_runs": plan, "refresh_plan_ms_runs": rp},
            "kernel_us": kus, "launches_per_refresh": launches, "exact": exact}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True)
    ap.add_argument("--refreshes", type=int, default=200)
    ap.add_argument("--plan-reps", type=int, default=5)
    ap.add_argument("--host-reps", type=int, default=5)
    ap.add_argument("--cases", default="config3,pf")
    a = ap.parse_args()
    if not torch.cuda.is_available() or api.device_count() == 0:
        raise SystemExit("occupancy_refresh_bench.py: no CUDA device -- the product path has no CPU fallback")
    os.makedirs(a.out, exist_ok=True)
    z = np.load(os.path.join(ROOT, "tests", "golden", "occupancy.npz"))
    polys = [z["cell_xy"][z["cell_off"][i]:z["cell_off"][i + 1]] for i in range(len(z["cell_off"]) - 1)]
    bounds = np.asarray(z["bounds"], np.float64)
    world, _, _ = bench.load_world()
    info = gpu_info()
    path = os.path.join(a.out, "r04_occupancy_refresh.jsonl")
    all_cases = cases()
    with open(path, "w") as f:
        for name in a.cases.split(","):
            r = run_case(name, all_cases[name], polys, bounds, world, a)
            r.update(info)
            line = json.dumps(r)
            print(line, flush=True)
            f.write(line + "\n")


if __name__ == "__main__":
    main()
