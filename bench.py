#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's config, one JSON line on rank 0.

metric  : Dubins/arc edge evaluations per second (steer + collide + cost) of the batched RRT planner
workload: configs[1] -- 4096 independent RRT queries per GPU x 2048 steer calls each, Catalina map
          (K=27 circles, E=5, H=10 habitats, T=10 x C=986 shark grid), reference default mode
          (traj_time_stamp=True, plan_time=True), fp32 fast build.
A "step" is one pass of the planner over the batch.  `value` has the queries resident in HBM;
`e2e` goes through the host-buffer C ABI (auvrrt_plan_batch) with host<->device copies inside.
N > 1 (torchrun): queries are sharded across ranks (weak scaling, no data-path collective) and the
96-byte plan records are gathered to rank 0 over NCCL inside the timed region.

--impl reference times the reference's own pure-Python planner (the unmodified modules installed into baseline/_ref
by baseline/install_ref.py) on all host cores, one query of the workload per process per step; without that install it
falls back to the fp64 C port of the reference (oracle/auvrrt_oracle.c).
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "auv-sim_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "edge_evals_per_s"
UNIT = "edges/s"
Q_PER_GPU = 4096
ITERS = 2048
FP32_NOMINAL_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12      # 74.4 (BASELINE.md section 4)


def ncu_traffic(kernel_key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu capture
    (profiles/traffic.json, written from `ncu --set full` reports by tools/ncu_summary.py), or None"""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get(kernel_key)
    except Exception:
        return None


def load_world():
    with open(os.path.join(ROOT, "tests", "golden", "catalina_map.json")) as f:
        world = json.load(f)
    g = np.load(os.path.join(ROOT, "tests", "golden", "shark_grid.npz"))
    return world, g["bins"], g["probs"]


def make_queries(q0, q1):
    """config 2: starts uniform in the box x in [-300,-100], y in [-100,100] restricted to the
    polygon (performance.py:56-62), theta = 0, t = 0; seed = global query id."""
    world, _, _ = load_world()
    poly = np.array(world["boundary"])
    rs = np.random.RandomState(12345)
    n = q1
    pts = []
    while len(pts) < n:
        c = np.stack([rs.uniform(-300, -100, 4 * n), rs.uniform(-100, 100, 4 * n)], 1)
        ax, ay = poly[:, 0], poly[:, 1]
        bx, by = np.roll(ax, -1), np.roll(ay, -1)
        cr = (bx - ax)[None] * (c[:, 1:2] - ay[None]) - (by - ay)[None] * (c[:, 0:1] - ax[None])
        inside = np.all(cr < 0, 1) | np.all(cr > 0, 1)
        # also keep the start out of the obstacle circles: a start inside one can never grow a tree
        # (the reference raises TypeError at rrt_dubins.py:174) and would be a degenerate cheap query
        circ = np.array(world["circles"])
        reff = np.maximum.accumulate(circ[::-1, 2])[::-1]
        d = np.hypot(c[:, 0:1] - circ[None, :, 0], c[:, 1:2] - circ[None, :, 1])
        inside &= np.all(d > reff[None] + 1e-6, 1)
        pts.extend(c[inside].tolist())
    starts = np.zeros((n, 5))
    starts[:, :2] = np.array(pts[:n])
    return starts[q0:q1], np.arange(q0, q1, dtype=np.uint64)


class ClockSampler(threading.Thread):
    """samples SM clock + throttle reasons through NVML while the timed region runs"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.004)

    def result(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


REF_DIR = os.path.join(ROOT, "baseline", "_ref")
PORT_THREADS = 16            # the C port is always timed on this many threads, so BENCH and SCALE ratios are comparable


def python_reference_available():
    return os.path.isfile(os.path.join(REF_DIR, "path_planning", "rrt_dubins.py"))


_py_ref_state = {}


def _py_ref_worker(qids):
    """one process of the pure-Python reference arm: plan the given queries with the UNMODIFIED reference modules
    (baseline/_ref, installed by baseline/install_ref.py) under the iteration-budget clock; returns
    (steer calls, seconds inside RRT.exploring, plans found)"""
    st = _py_ref_state
    if not st:
        os.environ["AUVRRT_REFERENCE"] = REF_DIR
        import importlib
        from oracle import harness as H
        H = importlib.reload(H)
        ref = H.load_reference()
        world = H.catalina_world(ref)
        csv = os.path.join(REF_DIR, "path_planning", "shark_data", "AUVGrid_prob_500_turn.csv")
        obstacles, poly, habitats, cells, shark = H.world_objects(ref, world, grid_csv=csv)
        st.update(H=H, ref=ref, habitats=habitats, rrt=ref.RRT(poly, obstacles, shark, cells))
    H, ref = st["H"], st["ref"]
    calls = found = 0
    secs = 0.0
    for qid, sx, sy in qids:
        res, c, dt = H.timed_exploring(ref, st["rrt"], ref.MPS(sx, sy), list(st["habitats"]), iterations=ITERS, seed=int(qid))
        calls += c; secs += dt; found += res is not None
    return calls, secs, found


class PythonReference:
    """the reference's own pure-Python planner on the host cores: a pool of processes, one query of the workload each
    per step (queries are independent: the embarrassingly parallel way its authors would run many)"""

    def __init__(self, procs=0):
        import multiprocessing as mp
        self.procs = procs or (os.cpu_count() or 1)
        self.pool = mp.get_context("spawn").Pool(self.procs)
        self.starts, _ = make_queries(0, max(self.procs, 1) * 16)

    def step(self, k, per_proc=1):
        """plan `per_proc` queries on each of the `procs` processes concurrently (query ids k*procs*per_proc ...);
        -> (edges/s over all processes, plans/s, wall, found)"""
        n = self.procs * per_proc
        ids = [(k * n + j) % len(self.starts) for j in range(n)]
        jobs = [[(i, float(self.starts[i, 0]), float(self.starts[i, 1])) for i in ids[p::self.procs]] for p in range(self.procs)]
        t0 = time.perf_counter()
        out = self.pool.map(_py_ref_worker, jobs, chunksize=1)
        wall = time.perf_counter() - t0
        calls = sum(o[0] for o in out)
        return calls / wall, len(ids) / wall, wall, sum(o[2] for o in out), max(o[1] for o in out)

    def single(self):
        """one query in one process: the single-core figure"""
        calls, secs, _ = self.pool.apply(_py_ref_worker, ([(0, float(self.starts[0, 0]), float(self.starts[0, 1]))],))
        return calls / secs

    def close(self):
        self.pool.close(); self.pool.join()


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for l in f:
                if l.startswith("model name"):
                    return l.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def cpu_baseline(nthreads=0, sample_queries=None):
    """the oracle port (fp64 C restatement of the pure-Python reference) on the host cores"""
    from oracle import orc
    world, bins, probs = load_world()
    ow = orc.OracleWorld.from_map(world, bins, probs)
    nt = nthreads or orc.num_threads()
    nq = sample_queries or max(32 * nt, 64)        # ~1.3 s wall, ~20-40 s of CPU work
    starts, seeds = make_queries(0, nq)
    pp = orc.plan_params(ITERS)
    t0 = time.perf_counter()
    res, counts, status = orc.exploring_batch(ow, starts, seeds, pp, nthreads=nt)
    dt = time.perf_counter() - t0
    return {"value": nq * ITERS / dt, "unit": UNIT, "cores": nt, "kind": "port",
            "sample": "%d of the %d queries x %d iterations, fp64 C port of the pure-Python reference "
                      "(oracle/auvrrt_oracle.c), %d threads, %.2f s wall" % (nq, Q_PER_GPU, ITERS, nt, dt),
            "plans_per_s": nq / dt, "seconds": dt}


def config_dict(n_gpus):
    return {"workload": "configs[1]: %d independent RRT-Dubins queries per GPU x %d steer calls, Catalina map "
                        "(K=27, E=5, H=10, T=10, C=986), time-bin parent pick (reference default mode)" % (Q_PER_GPU, ITERS),
            "queries_per_gpu": Q_PER_GPU, "iterations": ITERS, "global_queries": Q_PER_GPU * n_gpus,
            "parallelism": "queries sharded across %d GPU(s); NCCL gather of 96-byte plan records" % n_gpus,
            "l2": "flushed between timed steps (256 MiB write); tree workspace is larger than L2"}


def run_reference(args, rank, world_size):
    """the reference arm: the UNMODIFIED pure-Python planner (baseline/_ref) on all host cores when it is installed,
    else its fp64 C port.  A step = every host core plans one query of the workload (2048 steer calls)."""
    if rank != 0:
        return
    port = cpu_baseline(nthreads=PORT_THREADS)
    port_obj = {"value": port["value"], "unit": UNIT, "cores": port["cores"], "kind": "port", "sample": port["sample"]}
    if python_reference_available():
        pr = PythonReference()
        try:
            single = pr.single()
            vals = []
            for i in range(args.warmup + args.steps):
                r = pr.step(i)
                if i >= args.warmup:
                    vals.append(r)
        finally:
            pr.close()
        v = float(np.mean([r[0] for r in vals]))
        ms = float(np.mean([r[2] for r in vals])) * 1e3
        sample = ("%d of the %d queries x %d steer calls per step (one query per process, %d processes), unmodified "
                  "path_planning/rrt_dubins.py + cost.py from baseline/_ref under the iteration-budget clock, CPython %s, %s"
                  % (pr.procs, Q_PER_GPU, ITERS, pr.procs, sys.version.split()[0], cpu_model()))
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic", "config": config_dict(args.gpus),
                "plans_per_s": float(np.mean([r[1] for r in vals])),
                "cpu_baseline": {"value": v, "unit": UNIT, "cores": pr.procs, "kind": "reference", "sample": sample,
                                 "single_process_edges_per_s": single, "cpu_model": cpu_model(), "port": port_obj},
                "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "note": "the reference's own pure-Python planner; `port` is its fp64 C restatement (oracle/auvrrt_oracle.c) "
                        "on %d threads for comparison" % PORT_THREADS}
        print(json.dumps(line))
        return
    vals = []
    for i in range(args.warmup + args.steps):
        b = cpu_baseline(nthreads=PORT_THREADS)
        if i >= args.warmup:
            vals.append(b)
    v = float(np.mean([b["value"] for b in vals]))
    ms = float(np.mean([b["seconds"] for b in vals])) * 1e3
    b = vals[-1]
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": config_dict(args.gpus),
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": b["cores"], "kind": "port", "sample": b["sample"]},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "baseline/_ref is not installed (python baseline/install_ref.py in the build container): this arm "
                    "times the fp64 C port of the pure-Python reference"}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="f32", choices=["f32", "f64"])
    ap.add_argument("--group", type=int, default=0, help="lanes per tree: 0 auto, 32/16/8, 1 = thread per tree")
    ap.add_argument("--no-extras", action="store_true", help="skip micro-benchmarks / cpu baseline")
    ap.add_argument("--micro-edges", type=int, default=100_000_000)
    ap.add_argument("--queries", type=int, default=0, help="queries per GPU (default: the configs[1] size, 4096)")
    ap.add_argument("--config5-queries", type=int, default=1 << 20,
                    help="total queries of the sharded config-5 run (strong scaling, part of every line; 0 skips it)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (rank 0's plan records and chains) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    global Q_PER_GPU
    if args.queries > 0:
        Q_PER_GPU = args.queries
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world_size)
        return

    import torch
    import torch.distributed as dist
    from auvrrt import api, device as adev
    if not torch.cuda.is_available() or api.device_count() == 0:
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world_size > 1:
        dist.init_process_group("nccl", device_id=dev)
    world, bins, probs = load_world()
    env = api.Env.from_map(world, bins, probs, device=local_rank)
    pp = api.plan_params(ITERS, group=args.group)
    starts, seeds = make_queries(rank * Q_PER_GPU, (rank + 1) * Q_PER_GPU)
    planner = adev.DevicePlanner(env, pp, args.precision, Q_PER_GPU, want_chain=True)
    planner.set_queries(starts, seeds)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    gathered = torch.empty((world_size, Q_PER_GPU, planner.records.shape[1]), dtype=torch.uint8, device=dev) if world_size > 1 else None
    stream = torch.cuda.current_stream()

    def step():
        planner.launch(stream)
        if world_size > 1:   # the final min-cost plan gather: 96-byte records, rank 0 keeps the minimum
            dist.all_gather_into_tensor(gathered.view(-1), planner.records.view(-1))

    def barrier():
        torch.cuda.synchronize()
        if world_size > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = api.launch_count()
    evs = []
    barrier()
    for _ in range(args.steps):
        flush.fill_(1)                       # L2 flush, outside the event-timed region
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        step()
        e1.record(stream)
        evs.append((e0, e1))
    barrier()
    launches = api.launch_count() - launches0
    ms_total = sum(a.elapsed_time(b) for a, b in evs)
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world_size > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    sampler.stop_flag = True
    sampler.join()
    rec = planner.records_numpy()
    ok = int((rec["status"] == 0).sum())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, rec, planner.chain[:planner.n].cpu().numpy())

    # ---- end to end through the host-buffer C ABI (host arrays in, records + chains out)
    e2e_steps = max(2, min(args.steps, 3))
    api.plan_batch(env, starts, seeds, pp, args.precision)           # warm: allocates env-owned buffers
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        r = api.plan_batch(env, starts, seeds, pp, args.precision)
        if world_size > 1:
            dist.all_gather_into_tensor(gathered.view(-1), torch.from_numpy(r["records"].view(np.uint8).reshape(-1)).to(dev))
    barrier()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world_size > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s = float(te.item())
    rsz = 4 if args.precision == "f32" else 8

    c5 = None
    if args.config5_queries > 0 and not args.no_extras:
        try:
            del planner
            torch.cuda.empty_cache()
            c5 = config5(env, dev, args, api, adev, rank, world_size)
        except Exception as ex:
            c5 = {"error": repr(ex)}

    if rank != 0:
        if world_size > 1:
            dist.destroy_process_group()
        return

    edges = Q_PER_GPU * world_size * ITERS * args.steps
    value = edges / (ms_total * 1e-3)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world_size, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": args.precision, "data": "synthetic", "config": config_dict(world_size),
            "plans_per_s": Q_PER_GPU * world_size * args.steps / (ms_total * 1e-3),
            "queries_ok": ok, "gpu_launches": int(launches), "clocks": sampler.result(),
            "e2e": {"value": Q_PER_GPU * world_size * ITERS * e2e_steps / e2e_s, "unit": UNIT,
                    "h2d_bytes_per_step": Q_PER_GPU * (5 * rsz + 8),
                    "d2h_bytes_per_step": Q_PER_GPU * (96 + 4 * pp.chain_cap),
                    "plans_per_s": Q_PER_GPU * world_size * e2e_steps / e2e_s, "steps": e2e_steps}}

    # ---- roofline of the dominant kernel (k_plan): algorithmic FLOP per launch / event time
    K, E, H, T = len(world["circles"]), len(world["boundary"]), len(world["habitats"]), len(bins)
    W = float(rec["n_waypoints"].sum()); P = float(rec["n_primitives"].sum())
    acc = float((rec["n_nodes"] - 1).sum()) / (len(rec) * ITERS)
    R_rows = 35
    flop = 6 * W * K + 6 * W * E + 30 * P + acc * W * (2 * T + 2 * R_rows + 6 * H + 3)
    sfu = K * len(rec) * ITERS + 8 * P
    per_launch_s = ms_total * 1e-3 / args.steps
    try:
        cal_flops, _ = api.calibrate_fp32(local_rank, 8192)
    except Exception:
        cal_flops = None
    peak = (cal_flops or FP32_NOMINAL_TFLOPS * 1e12) / 1e12
    ach = flop * world_size / per_launch_s / 1e12 / world_size
    line["roofline"] = {"bound": "fp32", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                        "traffic": ncu_traffic("k_plan_f32_g32_q4096") if (world_size == 1 and Q_PER_GPU == 4096) else None, "kernel": ("k_plan_tpt<float>" if (args.group == 1 or (args.group == 0 and Q_PER_GPU >= 32768)) else "k_plan<float,%d>" % (args.group or 32)),
                        "peak_source": "FFMA calibration kernel measured live in this run" if cal_flops else "nominal 148 SM x 128 lanes x 2 x 1.965 GHz",
                        "nominal_peak": FP32_NOMINAL_TFLOPS,
                        "algorithmic_flop_per_edge": flop / (len(rec) * ITERS), "sfu_per_edge": sfu / (len(rec) * ITERS),
                        "waypoints_per_edge": W / (len(rec) * ITERS), "primitives_per_edge": P / (len(rec) * ITERS),
                        "note": "no tensor cores: no dense contraction on this path (BASELINE.json north_star)"}

    if c5 is not None:
        line["config5"] = c5
    if not args.no_extras and world_size == 1:
        port = cpu_baseline(nthreads=PORT_THREADS)
        port_obj = {k: v for k, v in port.items() if k in ("value", "unit", "cores", "kind", "sample")}
        line["cpu_baseline"] = port_obj
        if python_reference_available():
            try:
                pr = PythonReference()
                try:
                    single = pr.single()
                    PER_PROC = 8                       # ~10 s of wall clock: 8 queries x 2048 steer calls per process
                    r = pr.step(0, per_proc=PER_PROC)
                finally:
                    pr.close()
                line["cpu_baseline"] = {
                    "value": r[0], "unit": UNIT, "cores": pr.procs, "kind": "reference",
                    "sample": "%d of the %d queries x %d steer calls, %d queries per process on %d processes, unmodified "
                              "reference modules from baseline/_ref, %.1f s wall; %s" % (pr.procs * PER_PROC, Q_PER_GPU, ITERS, PER_PROC, pr.procs, r[2], cpu_model()),
                    "single_process_edges_per_s": single, "plans_per_s": r[1], "port": port_obj}
            except Exception as ex:
                line["cpu_baseline"]["python_reference_error"] = repr(ex)
        try:
            line["extras"] = extras(env, dev, args, api, adev)
        except Exception as ex:   # extras never invalidate the headline line
            line["extras"] = {"error": repr(ex)}
    elif not args.no_extras:
        line["cpu_baseline"] = None
    print(json.dumps(line))
    if world_size > 1:
        dist.destroy_process_group()


DUMP_BYTES = 63 << 20        # array data of --dump-outputs: under 64 MiB with the .npy headers


def dump_outputs(out_dir, rec, chain):
    """The planner's outputs of the last timed step, one float64 .npy per record field plus `chain` (the stream
    positions of each plan's nodes, exact in float64) and `query` (the query index of each row).  Above DUMP_BYTES a
    fixed seeded sample of the queries is written, so that two builds can be compared file for file."""
    fields = {name: rec[name] for name in rec.dtype.names}
    fields["chain"] = chain.view(np.uint32)
    row_bytes = 8 * (1 + sum(int(np.prod(a.shape[1:])) for a in fields.values()))
    rows = np.arange(len(rec))
    if len(rows) * row_bytes > DUMP_BYTES:
        rows = np.sort(np.random.RandomState(0).choice(len(rows), DUMP_BYTES // row_bytes, replace=False))
    out = {name: a[rows] for name, a in fields.items()}
    out["query"] = rows
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


def catalina_parents(world, n, dev, seed=3):
    """n tree-node-like parent states (x, y, theta, traj_time_stamp, length) uniform over the FREE space of the
    Catalina map: inside the boundary polygon and outside every (inflated) obstacle circle; theta uniform,
    traj_time_stamp uniform in [0, 400] s (inside the shark grid's time bins), length 0"""
    import torch
    poly = torch.tensor(world["boundary"], device=dev, dtype=torch.float32)
    circ = np.array(world["circles"])
    reff = np.maximum.accumulate(circ[::-1, 2])[::-1].copy()
    cx = torch.tensor(circ[:, 0], device=dev, dtype=torch.float32); cy = torch.tensor(circ[:, 1], device=dev, dtype=torch.float32)
    cr = torch.tensor(reff + 0.01, device=dev, dtype=torch.float32)
    g = torch.Generator(device=dev); g.manual_seed(seed)
    out = torch.empty((n, 5), device=dev, dtype=torch.float32)
    have = 0
    chunk = min(n, 1 << 24)
    ax, ay = poly[:, 0], poly[:, 1]
    bx, by = torch.roll(ax, -1), torch.roll(ay, -1)
    while have < n:
        x = torch.rand(chunk, device=dev, generator=g) * 549.8 - 467.4
        y = torch.rand(chunk, device=dev, generator=g) * 344.7 - 153.5
        cross = (bx - ax)[None] * (y[:, None] - ay[None]) - (by - ay)[None] * (x[:, None] - ax[None])
        ok = (cross < 0).all(1) | (cross > 0).all(1)
        ok &= (((x[:, None] - cx[None]) ** 2 + (y[:, None] - cy[None]) ** 2) > (cr * cr)[None]).all(1)
        x, y = x[ok], y[ok]
        m = min(n - have, x.numel())
        out[have:have + m, 0] = x[:m]; out[have:have + m, 1] = y[:m]
        have += m
    out[:, 2] = (torch.rand(n, device=dev, generator=g) * 2 - 1) * np.pi
    out[:, 3] = torch.rand(n, device=dev, generator=g) * 400.0
    out[:, 4] = 0
    return out


def micro_catalina(env, dev, n_edges, api, adev, cal_flops, timed):
    """SURVEY 8(d) "Catalina scale": independent arc edges (S1 steer + K1 collide + C1 cost) on the real map,
    K = 27 circles, E = 5, H = 10 habitats, T x C = 10 x 986 shark grid -- where the north star's 1e10 edges/s lives.
    One thread per edge (edges_tpe.cu).  Three runs on the same edges: classification grid with cost on (the
    product path) and off, and the all-pairs variant (every waypoint against every circle / polygon edge / habitat),
    whose executed work is what SURVEY's FLOP formula counts."""
    import torch
    world, bins_, _ = load_world()
    K, E, H, T = len(world["circles"]), len(world["boundary"]), len(world["habitats"]), len(bins_)
    par = catalina_parents(world, n_edges, dev)
    sd = torch.arange(n_edges, device=dev, dtype=torch.int64)
    safe = torch.zeros(n_edges, dtype=torch.uint8, device=dev); cnt = torch.zeros(n_edges, dtype=torch.int32, device=dev)
    leaf = torch.zeros((n_edges, 5), device=dev); cost = torch.zeros((n_edges, 3), device=dev)
    sp5 = [2.0, 0.5, 30.0, 0.5, 2.0]
    out = {}
    saved = {k: os.environ.get(k) for k in ("AUVRRT_EDGES_VARIANT", "AUVRRT_EDGES_BRUTE")}
    try:
        os.environ["AUVRRT_EDGES_VARIANT"] = "tpe"
        os.environ["AUVRRT_EDGES_BRUTE"] = "0"
        t_on, _ = timed(lambda: adev.edges_arc_cost_dev(env, par, sd, sp5, -4.0, safe, cnt, leaf, cost, "f32"), reps=3, warm=1)
        safe_grid = safe.clone(); cost_grid = cost.clone(); cnt_grid = cnt.clone()
        W = float(cnt.float().mean().item()); Pm = 14.5
        acc = float(safe.float().mean().item())
        t_off, _ = timed(lambda: adev.edges_arc_dev(env, par, sd, sp5, safe, cnt, leaf, "f32"), reps=3, warm=1)
        same_off = bool(torch.equal(safe, safe_grid))
        os.environ["AUVRRT_EDGES_BRUTE"] = "1"
        t_all, _ = timed(lambda: adev.edges_arc_cost_dev(env, par, sd, sp5, -4.0, safe, cnt, leaf, cost, "f32"), reps=3, warm=1)
        R_rows = 35
        flop_geo = 6 * W * K + 6 * W * E + 30 * Pm
        flop_cost = (W - 1) * (2 * T + 2 * R_rows + 6 * H + 3)        # every appended waypoint is costed (the parent is not)
        flop = flop_geo + flop_cost
        peak = cal_flops / 1e12
        out["micro_catalina_arc_cost"] = {
            "edges": n_edges, "circles": K, "polygon_edges": E, "habitats": H, "time_bins": T, "cells": int(len(world["cells"])),
            "waypoints_per_edge": W, "primitives_per_edge": Pm, "safe_fraction": acc,
            "edges_per_s": n_edges / t_on, "seconds": t_on,
            "kernel": "k_edges_arc_tpe<float,COST,grid> (one thread per edge, classification grid)",
            "algorithmic_flop_per_edge": flop, "equivalent_all_pairs_tflops": n_edges * flop / t_on / 1e12,
            "equivalent_frac": n_edges * flop / t_on / cal_flops,
            "edges_with_shark_cost": float((cost_grid[:, 0] != 0).float().mean().item()),
            "note": "the grid decides most waypoint tests with one load, so the all-pairs FLOP count is an equivalent here; "
                    "the executed-work roofline is micro_catalina_arc_cost_allpairs (same edges, same results)"}
        # what bounds the grid kernel is instruction issue, not FLOPs: executed warp-instructions per edge (ncu, profiles/
        # r02_tpe_final.txt) x measured edges/s against 148 SMs x 4 schedulers x 1 instruction per clock
        wi = ncu_traffic("k_edges_arc_tpe_f32_cost_grid_warp_instr_per_edge")
        if wi:
            issue_peak = 148 * 4 * 1.965e9
            out["micro_catalina_arc_cost"]["roofline"] = {
                "bound": "issue", "achieved": n_edges / t_on * wi / 1e9, "peak": issue_peak / 1e9, "unit": "Gwarp-instr/s",
                "frac": n_edges / t_on * wi / issue_peak, "warp_instructions_per_edge": wi,
                "source": "smsp__inst_executed.sum / edges from the committed ncu capture of this kernel; peak = 148 SMs x 4 schedulers x 1.965 GHz"}
        out["micro_catalina_arc"] = {"edges": n_edges, "edges_per_s": n_edges / t_off, "seconds": t_off, "identical_booleans": same_off,
                                     "algorithmic_flop_per_edge": flop_geo, "equivalent_frac": n_edges * flop_geo / t_off / cal_flops,
                                     "kernel": "k_edges_arc_tpe<float,no cost,grid>"}
        d = (cost - cost_grid).abs()
        out["micro_catalina_arc_cost_allpairs"] = {
            "edges": n_edges, "edges_per_s": n_edges / t_all, "seconds": t_all,
            "kernel": "k_edges_arc_tpe<float,COST,all pairs> (FFMA2 over circle pairs)",
            "roofline": {"bound": "fp32", "achieved": n_edges * flop / t_all / 1e12, "peak": peak, "unit": "TFLOP/s",
                         "frac": n_edges * flop / t_all / cal_flops, "algorithmic_flop_per_edge": flop,
                         "peak_source": "FFMA calibration kernel measured live in this run"},
            "booleans_differ_fraction": float((safe != safe_grid).float().mean().item()),
            "counts_identical": bool(torch.equal(cnt, cnt_grid)),
            "cost_terms_max_abs_diff": [float(d[:, j].max().item()) for j in range(3)]}
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    del par, sd, safe, cnt, leaf, cost
    torch.cuda.empty_cache()
    return out


def config5(env, dev, args, api, adev, rank, world_size):
    """BASELINE.json configs[4]: Q planning queries (default 2^20) sharded contiguously over the ranks, planned by the
    thread-per-tree kernel with everything resident in HBM, one NCCL all-gather of the 96-byte records, the global
    minimum-cost plan by two 8-byte MIN all-reduces, the winner's path re-created on its owner and broadcast
    (auvrrt.multi.plan_sharded_device).  STRONG scaling: the same Q at every N."""
    import torch
    import torch.distributed as dist
    from auvrrt import multi
    Q = int(args.config5_queries)
    own_pg = False
    if not dist.is_initialized():
        import socket
        sock = socket.socket(); sock.bind(("127.0.0.1", 0)); port = sock.getsockname()[1]; sock.close()
        dist.init_process_group("nccl", init_method="tcp://127.0.0.1:%d" % port, rank=0, world_size=1, device_id=dev)
        own_pg = True
    try:
        pp5 = api.plan_params(ITERS, group=1)
        starts, seeds = make_queries(0, Q)
        lo, hi = multi.shard_range(Q, rank, world_size)
        cap = max(multi.shard_range(Q, r, world_size)[1] - multi.shard_range(Q, r, world_size)[0] for r in range(world_size))
        planner = adev.DevicePlanner(env, pp5, "f32", cap, want_chain=True)

        def sync():
            torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
        multi.plan_sharded_device(env, starts, seeds, pp5, "f32", want_path=False, planner=planner)      # warm-up
        reps, ts = 2, []
        for _ in range(reps):
            sync()
            t0 = time.perf_counter()
            r = multi.plan_sharded_device(env, starts, seeds, pp5, "f32", want_path=True, planner=planner)
            sync()
            ts.append(time.perf_counter() - t0)
        t = torch.tensor([min(ts)], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        secs = float(t.item())
        out = None
        if rank == 0:
            rec = r["records"]
            n = rec.shape[0]
            status = rec.view(torch.int32).view(n, 24)[:, 0]
            best = r["best"]
            # a fixed sample of query ids, planned again by this rank alone with the same kernel: identical records?
            ids = np.linspace(0, Q - 1, 64).astype(np.int64)
            sp = adev.DevicePlanner(env, pp5, "f32", len(ids), want_chain=False)
            sp.set_queries(starts[ids], seeds[ids]); sp.launch(); torch.cuda.synchronize()
            same = bool(torch.equal(sp.records[:len(ids)], rec[torch.from_numpy(ids).to(dev)]))
            bc = rec[best:best + 1].cpu().numpy().view(api.RECORD_DTYPE)["cost"].reshape(-1)[0] if best >= 0 else None
            out = {"queries": Q, "iterations": ITERS, "n_gpus": world_size, "scaling": "strong", "seconds": secs,
                   "plans_per_s": Q / secs, "edges_per_s": Q * ITERS / secs, "queries_ok": int((status == 0).sum().item()),
                   "best_query": best, "best_cost": None if bc is None else float(bc),
                   "best_path_rows": None if r["path"] is None else int(len(r["path"])),
                   "gather_bytes_per_rank": int(cap * 96), "sample_records_equal_single_gpu": same,
                   "kernel": "k_plan_tpt<float> (one thread per tree)",
                   "includes": "planner launch on every rank, NCCL all-gather of records, 2 MIN all-reduces, winner's path "
                               "materialised on its owner and broadcast; wall clock, max over ranks"}
        del planner
        torch.cuda.empty_cache()
        return out
    finally:
        if own_pg:
            dist.destroy_process_group()


def extras(env, dev, args, api, adev):
    """secondary measurements: NN scan against the HBM roofline, config-4 micro-benchmark, fp64 build"""
    import torch
    out = {}
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    hbm = peaks.get("hbm_gbs", 6650.0)

    def timed(fn, reps=5, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record(); torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e-3)
        return float(np.mean(ts)), float(np.min(ts))

    # NN scan: one query over a tree larger than L2 (2^27 nodes, 1 GiB of fp32 x/y)
    n = 1 << 27
    tx = torch.rand(n, device=dev) * 550 - 467
    ty = torch.rand(n, device=dev) * 345 - 153
    qx = torch.tensor([-200.0], device=dev); qy = torch.tensor([0.0], device=dev)
    idx = torch.zeros(1, dtype=torch.int32, device=dev)
    scr = adev.nn_scratch(1, dev)
    mean_s, min_s = timed(lambda: adev.nn_dev(tx, ty, qx, qy, idx, scr, "f32"))
    gbs = 8.0 * n / mean_s / 1e9
    out["roofline_nn"] = {"bound": "hbm", "achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm,
                          "traffic": ncu_traffic("k_nn_partial_f32_n2p27"), "kernel": "k_nn_partial<float>", "nodes": n, "queries": 1,
                          "peak_source": "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650",
                          "algorithmic_bytes": "8 B per node per pass"}
    del tx, ty

    # Catalina scale: independent steer + collide + cost edges, one thread per edge
    try:
        cal_c, _ = api.calibrate_fp32(dev.index, 8192)
        out.update(micro_catalina(env, dev, int(args.micro_edges), api, adev, cal_c, timed))
    except Exception as ex:
        out["micro_catalina_arc_cost"] = {"error": repr(ex)}

    # throughput planner (one thread per tree) at config-5 scale: 65536 queries resident on one GPU
    try:
        Qb = 262144
        ppt = api.plan_params(ITERS, group=1)
        st, sd = make_queries(0, Qb)
        pl = adev.DevicePlanner(env, ppt, "f32", Qb, want_chain=True)
        pl.set_queries(st, sd)
        mean_s, min_s = timed(lambda: pl.launch(), reps=2, warm=1)
        rec = pl.records_numpy()
        world, bins_, _ = load_world()
        Wt, Pt = float(rec["n_waypoints"].sum()), float(rec["n_primitives"].sum())
        acc = float((rec["n_nodes"] - 1).sum()) / (len(rec) * ITERS)
        flop = 6 * Wt * 27 + 6 * Wt * 5 + 30 * Pt + acc * Wt * (2 * 10 + 2 * 35 + 6 * 10 + 3)
        cal_t, _ = api.calibrate_fp32(dev.index, 8192)
        out["throughput_planner_group1"] = {"queries": Qb, "iterations": ITERS, "edges_per_s": Qb * ITERS / mean_s,
                                            "plans_per_s": Qb / mean_s, "seconds": mean_s,
                                            "queries_ok": int((rec["status"] == 0).sum()), "kernel": "k_plan_tpt<float>",
                                            "achieved_tflops": flop / mean_s / 1e12, "frac_of_fp32_peak": flop / mean_s / cal_t,
                                            "note": "config-5 scale on one GPU: one thread per tree"}
        del pl
        torch.cuda.empty_cache()
    except Exception as ex:
        out["throughput_planner_group1"] = {"error": repr(ex)}

    # planner mode 1 (get_random_mps + get_closest_mps, rrt_dubins.py:136-139, :505-513): the IN-PLANNER nearest-node scan.
    # Every steer call scans the query's own tree (x[], y[] SoA, 8 B per node, lane-strided, coalesced); 4096 trees of
    # <= 2049 nodes are 64 MB of coordinates, resident in the 126 MB L2, so the scan is L2-bandwidth work.
    try:
        Q1, I1 = 4096, ITERS
        pp1 = api.plan_params(I1, mode=1)
        st1, sd1 = make_queries(0, Q1)
        pl1 = adev.DevicePlanner(env, pp1, "f32", Q1, want_chain=True)
        pl1.set_queries(st1, sd1)
        mean_s, _ = timed(lambda: pl1.launch(), reps=3, warm=1)
        rec1 = pl1.records_numpy()
        # nodes scanned: the tree grows by one node per accepted edge, about linearly over the I steer calls
        scanned = float(((rec1["n_nodes"].astype(np.float64) + 1.0) * 0.5 * I1).sum())
        out["planner_mode1_nn_scan"] = {"queries": Q1, "iterations": I1, "seconds": mean_s, "edges_per_s": Q1 * I1 / mean_s,
                                        "nodes_scanned": scanned, "scan_bytes": 8.0 * scanned,
                                        "scan_gbs_over_whole_kernel": 8.0 * scanned / mean_s / 1e9,
                                        "nodes_mean_final": float(rec1["n_nodes"].mean()),
                                        "kernel": "k_plan<float,32,mode 1> (warp-cooperative scan of the tree's x[], y[] SoA)",
                                        "note": "GB/s of node coordinates read by the nearest-node scans, over the duration of the WHOLE "
                                                "planner kernel (steer / collide / cost included); the L2 throughput ncu measures for "
                                                "this kernel is in profiles/r02_plan_mode1_nn.txt"}
        del pl1
        torch.cuda.empty_cache()
    except Exception as ex:
        out["planner_mode1_nn_scan"] = {"error": repr(ex)}

    # planner mode 3: Dubins-RRT with best-parent selection (row X1; the build's own definition, parity unpinned)
    try:
        Q3, I3, W3 = 4096, 1024, 12
        pp3 = api.plan_params(I3, mode=3, v=1.0, max_traj_time=200.0, dubins_rho=1.0, dubins_eta=20.0, near_radius=15.0, dubins_w=W3)
        st3, sd3 = make_queries(0, Q3)
        pl3 = adev.DevicePlanner(env, pp3, "f32", Q3, want_chain=True)
        pl3.set_queries(st3, sd3)
        mean_s, _ = timed(lambda: pl3.launch(), reps=3, warm=1)
        rec3 = pl3.records_numpy()
        cand = float(rec3["n_waypoints"].sum()) / W3
        out["planner_mode3_dubins"] = {"queries": Q3, "iterations": I3, "waypoints_per_edge": W3, "seconds": mean_s,
                                       "plans_per_s": Q3 / mean_s, "iterations_per_s": Q3 * I3 / mean_s,
                                       "candidate_edges_per_s": cand / mean_s, "candidates_per_iteration": cand / (Q3 * I3),
                                       "queries_ok": int((rec3["status"] == 0).sum()), "nodes_mean": float(rec3["n_nodes"].mean()),
                                       "kernel": "k_plan<float,32,mode 3> (lane = candidate parent, warp min-reduction)",
                                       "note": "sample -> nearest + near nodes -> six-word Dubins steer + collide + cost per lane -> best parent"}
        del pl3
        torch.cuda.empty_cache()
    except Exception as ex:
        out["planner_mode3_dubins"] = {"error": repr(ex)}

    # config 4: Dubins edges vs 500 synthetic circles, 20 waypoints per edge
    rs = np.random.RandomState(1234)
    K = 500
    circles = np.stack([rs.uniform(-467.4, 82.4, K), rs.uniform(-153.5, 191.2, K), rs.uniform(1, 5, K)], 1)
    world, _, _ = load_world()
    env4 = api.Env(circles=circles, boundary=world["boundary"], device=dev.index)
    ne = int(args.micro_edges)
    g = torch.Generator(device=dev); g.manual_seed(1)
    q0 = torch.stack([torch.rand(ne, device=dev, generator=g) * 549.8 - 467.4,
                      torch.rand(ne, device=dev, generator=g) * 344.7 - 153.5,
                      (torch.rand(ne, device=dev, generator=g) * 2 - 1) * np.pi], 1).contiguous()
    ang = (torch.rand(ne, device=dev, generator=g) * 2 - 1) * np.pi
    dist_ = torch.rand(ne, device=dev, generator=g) * 38 + 2
    q1 = torch.stack([q0[:, 0] + dist_ * torch.cos(ang), q0[:, 1] + dist_ * torch.sin(ang),
                      (torch.rand(ne, device=dev, generator=g) * 2 - 1) * np.pi], 1).contiguous()
    del ang, dist_
    safe = torch.zeros(ne, dtype=torch.uint8, device=dev); word = torch.zeros(ne, dtype=torch.uint8, device=dev)
    length = torch.zeros(ne, device=dev)
    flop_edge = 6 * 20 * K + 6 * 20 * 5 + 140 + 24 * 20
    cal, _ = api.calibrate_fp32(dev.index, 8192)
    os.environ["AUVRRT_EDGES_BRUTE"] = "1"       # all-pairs kernel: the algorithmic-FLOP roofline measurement
    mean_s, min_s = timed(lambda: adev.edges_dubins_dev(env4, q0, q1, 1.0, 20, safe, word, length, "f32"), reps=3, warm=1)
    safe_brute = safe.clone()
    out["micro_config4"] = {"edges": ne, "circles": K, "waypoints": 20, "edges_per_s": ne / mean_s,
                            "algorithmic_flop_per_edge": flop_edge, "achieved_tflops": ne * flop_edge / mean_s / 1e12,
                            "fp32_peak_tflops_calibrated": cal / 1e12, "frac": ne * flop_edge / mean_s / cal,
                            "safe_fraction": float(safe.float().mean().item()), "kernel": "k_edges_dubins<float,20> (all pairs)"}
    os.environ["AUVRRT_EDGES_BRUTE"] = "0"       # broad-phase cull through the classification grid: same booleans
    mean_c, _ = timed(lambda: adev.edges_dubins_dev(env4, q0, q1, 1.0, 20, safe, word, length, "f32"), reps=3, warm=1)
    out["micro_config4_culled"] = {"edges": ne, "edges_per_s": ne / mean_c, "kernel": "k_edges_dubins_culled<float>",
                                   "identical_booleans": bool(torch.equal(safe, safe_brute)),
                                   "equivalent_all_pairs_tflops": ne * flop_edge / mean_c / 1e12,
                                   "note": "same results as the all-pairs kernel; the grid skips circles that cannot touch a waypoint's cell"}
    safe_culled = safe.clone()

    # config 4 with the reference's own steer (S1 random arcs, P = 14.5 primitives, W = 11.9 waypoints on average)
    # against the same 500 circles + the Catalina polygon, cost off and cost on (habitats + shark grid)
    try:
        world, bins_, probs_ = load_world()
        env4c = api.Env(circles=circles, boundary=world["boundary"], habitats=world["habitats"], bins=bins_,
                        cells=world["cells"], probs=probs_, device=dev.index)
        # the Dubins edges with cost on (habitats + shark grid at every waypoint, t = arclength / v): SURVEY 8(d) "cost off and on"
        cost_d = torch.zeros((ne, 3), device=dev)
        mean_dc, _ = timed(lambda: adev.edges_dubins_cost_dev(env4c, q0, q1, 1.0, 20, 1.0, -4.0, safe, word, length, cost_d, "f32"),
                           reps=3, warm=1)
        flop_dc = flop_edge + 19 * (2 * 10 + 2 * 35 + 6 * 10 + 3)
        out["micro_config4_culled_cost"] = {"edges": ne, "edges_per_s": ne / mean_dc, "kernel": "k_edges_dubins_culled<float,COST>",
                                            "identical_booleans": bool(torch.equal(safe, safe_culled)),
                                            "algorithmic_flop_per_edge": flop_dc,
                                            "equivalent_all_pairs_tflops": ne * flop_dc / mean_dc / 1e12,
                                            "edges_with_shark_cost": float((cost_d[:, 0] != 0).float().mean().item()),
                                            "edges_touching_a_habitat": float((cost_d[:, 1] > 0).float().mean().item())}
        del cost_d
        na = int(args.micro_edges)
        g = torch.Generator(device=dev); g.manual_seed(2)
        par = torch.stack([torch.rand(na, device=dev, generator=g) * 549.8 - 467.4,
                           torch.rand(na, device=dev, generator=g) * 344.7 - 153.5,
                           (torch.rand(na, device=dev, generator=g) * 2 - 1) * np.pi,
                           torch.rand(na, device=dev, generator=g) * 400.0,
                           torch.zeros(na, device=dev)], 1).contiguous()
        sd = torch.arange(na, device=dev, dtype=torch.int64)
        safe_a = torch.zeros(na, dtype=torch.uint8, device=dev); cnt_a = torch.zeros(na, dtype=torch.int32, device=dev)
        sp5 = [2.0, 0.5, 30.0, 0.5, 2.0]
        mean_off, _ = timed(lambda: adev.edges_arc_dev(env4c, par, sd, sp5, safe_a, cnt_a, None, "f32"), reps=3, warm=1)
        safe_off = safe_a.clone()
        W_mean = float(cnt_a.float().mean().item())            # waypoints per edge incl. the parent
        cost_a = torch.zeros((na, 3), device=dev)
        mean_on, _ = timed(lambda: adev.edges_arc_cost_dev(env4c, par, sd, sp5, -4.0, safe_a, cnt_a, None, cost_a, "f32"), reps=3, warm=1)
        Pm = 14.5
        flop_off = 6 * W_mean * K + 6 * W_mean * 5 + 30 * Pm
        flop_on = flop_off + W_mean * (2 * 10 + 2 * 35 + 6 * 10 + 3)
        out["micro_config4_arc"] = {"edges": na, "circles": K, "waypoints_mean": W_mean, "edges_per_s": na / mean_off,
                                    "algorithmic_flop_per_edge": flop_off, "equivalent_all_pairs_tflops": na * flop_off / mean_off / 1e12,
                                    "equivalent_frac": na * flop_off / mean_off / cal, "safe_fraction": float(safe_off.float().mean().item()),
                                    "kernel": "k_edges_arc_tpe<float,no cost,grid> (one thread per edge, classification grid)",
                                    "note": "the grid skips circles that cannot touch a waypoint's cell, so the all-pairs FLOP count is an equivalent, not executed work"}
        out["micro_config4_arc_cost"] = {"edges": na, "edges_per_s": na / mean_on, "algorithmic_flop_per_edge": flop_on,
                                         "equivalent_all_pairs_tflops": na * flop_on / mean_on / 1e12, "equivalent_frac": na * flop_on / mean_on / cal,
                                         "identical_booleans": bool(torch.equal(safe_a, safe_off)),
                                         "edges_with_shark_cost": float((cost_a[:, 0] != 0).float().mean().item()),
                                         "kernel": "k_edges_arc_tpe<float,COST,grid> (steer + collide + cost, one thread per edge)"}
        # the same edges all pairs (every waypoint against all 500 circles, the boundary edges and the habitats, packed
        # FFMA2 loops): executed work = the FLOP formula, so this is the arc kernel's executed-work roofline at K = 500
        nb_ = max(1 << 20, na // 16)
        saved_b = os.environ.get("AUVRRT_EDGES_BRUTE")
        try:
            os.environ["AUVRRT_EDGES_BRUTE"] = "1"
            safe_b = torch.zeros(nb_, dtype=torch.uint8, device=dev); cnt_b = torch.zeros(nb_, dtype=torch.int32, device=dev)
            cost_b = torch.zeros((nb_, 3), device=dev)
            mean_ap, _ = timed(lambda: adev.edges_arc_cost_dev(env4c, par[:nb_], sd[:nb_], sp5, -4.0, safe_b, cnt_b, None, cost_b, "f32"),
                               reps=2, warm=1)
            Wb = float(cnt_b.float().mean().item())
            flop_ap = 6 * Wb * K + 6 * Wb * 5 + 30 * Pm + (Wb - 1) * (2 * 10 + 2 * 35 + 6 * 10 + 3)
            out["micro_config4_arc_cost_allpairs"] = {
                "edges": nb_, "circles": K, "edges_per_s": nb_ / mean_ap, "seconds": mean_ap,
                "kernel": "k_edges_arc_tpe<float,COST,all pairs> (FFMA2 over circle / habitat / boundary-edge pairs)",
                "roofline": {"bound": "fp32", "achieved": nb_ * flop_ap / mean_ap / 1e12, "peak": cal / 1e12, "unit": "TFLOP/s",
                             "frac": nb_ * flop_ap / mean_ap / cal, "algorithmic_flop_per_edge": flop_ap,
                             "peak_source": "FFMA calibration kernel measured live in this run"},
                "booleans_differ_fraction": float((safe_b != safe_a[:nb_]).float().mean().item()),
                "counts_identical": bool(torch.equal(cnt_b, cnt_a[:nb_]))}
            del safe_b, cnt_b, cost_b
        finally:
            if saved_b is None:
                os.environ.pop("AUVRRT_EDGES_BRUTE", None)
            else:
                os.environ["AUVRRT_EDGES_BRUTE"] = saved_b
        del par, sd, safe_a, cnt_a, cost_a, safe_off
        torch.cuda.empty_cache()
    except Exception as ex:
        out["micro_config4_arc"] = {"error": repr(ex)}
    del q0, q1, safe, word, length, safe_culled
    torch.cuda.empty_cache()

    # SURVEY 8(f) N1: vectorised gym_rrt Planner_RRT (RRTEnv's planner, freq = 10), one thread per episode
    try:
        from auvrrt import gym as agym
        from oracle import orc
        OBST = [(12.0, 38.0, 4.0), (17.0, 34.0, 5.0), (20.0, 29.0, 4.0), (25.0, 25.0, 3.0), (29.0, 20.0, 4.0),
                (34.0, 17.0, 3.0), (37.0, 8.0, 5.0)]                      # gym_rrt/envs/rrt_dubins.py:509-517
        Qg, max_step = 262144, 200
        rg = np.random.default_rng(5)
        gs = np.column_stack([rg.uniform(5, 15, Qg), rg.uniform(5, 15, Qg), rg.uniform(-np.pi, np.pi, Qg)])
        gg = np.column_stack([rg.uniform(35, 45, Qg), rg.uniform(35, 45, Qg)])
        gseed = np.arange(Qg, dtype=np.uint64)
        gb = agym.GymBatch((0, 0, 50, 50), OBST, Qg, freq=10.0, node_cap=max_step + 1, precision=agym.F32, device=dev.index)
        d_recs = torch.zeros(Qg * 88, dtype=torch.uint8, device=dev)

        def gym_run():
            gb.reset(gs, gg, gseed)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _lib_check(agym.lib().auvrrt_gym_step_dev(gb.handle, None, max_step, 0, d_recs.data_ptr(),
                                                      torch.cuda.current_stream().cuda_stream))
            e1.record(); torch.cuda.synchronize()
            return e0.elapsed_time(e1) * 1e-3
        from auvrrt._lib import check as _lib_check
        gym_run()
        ts = [gym_run() for _ in range(3)]
        recs = np.frombuffer(d_recs.cpu().numpy().tobytes(), dtype=agym.GYM_RECORD_DTYPE)
        steps = float(recs["steps"].sum())
        nthreads = orc.num_threads()
        qs = min(Qg, 512 * nthreads)
        w = orc.gym_world((0, 0, 50, 50), OBST, freq=10.0)
        t0 = time.perf_counter()
        crec, _ = orc.gym_plan_batch(w, gs[:qs], gg[:qs], gseed[:qs], max_step=max_step)
        ct = time.perf_counter() - t0
        out["gym_planner"] = {"episodes": Qg, "max_step": max_step, "steps_per_s": steps / float(np.mean(ts)),
                              "episodes_per_s": Qg / float(np.mean(ts)), "seconds": float(np.mean(ts)),
                              "found_fraction": float(recs["done"].mean()), "kernel": "k_gym_run<float>",
                              "cpu_port_steps_per_s": float(crec[:, 0].sum()) / ct, "cpu_cores": nthreads,
                              "cpu_found_fraction": float(crec[:, 1].mean()),
                              "note": "Planner_RRT.planning(max_step=200) per episode, main()'s obstacle course"}
        gb.close()
    except Exception as ex:
        out["gym_planner"] = {"error": repr(ex)}

    # SURVEY 8(f) N4: batched lattice A* (astar_fixLenSOG, main()'s weights and 300 m limit), one warp per query, fp64
    try:
        from auvrrt import astar as aastar
        from oracle import orc
        world, bins_, probs_ = load_world()
        ga = np.load(os.path.join(ROOT, "tests", "golden", "astar.npz"))
        aenv = aastar.AstarEnv(world["circles"], world["boundary"], world["habitats"], bins_, ga["cells_rounded"], probs_,
                               centroid=ga["centroid"], cells_are_rounded=True, device=dev.index)
        Qa = 148 * 128
        ra = np.random.default_rng(9)
        qa = aastar.make_queries(np.round(np.column_stack([ra.uniform(-300, -100, Qa), ra.uniform(20, 90, Qa)]), 2), 300.0)
        d_q = torch.from_numpy(qa.view(np.uint8).reshape(Qa, 64).copy()).to(dev)
        d_rec = torch.zeros(Qa * 40, dtype=torch.uint8, device=dev)
        wsb = int(aastar.lib().auvrrt_astar_workspace_bytes(Qa, 2048))
        d_ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
        from auvrrt._lib import check as _chk

        def astar_run():
            _chk(aastar.lib().auvrrt_astar_batch_dev(aenv.handle, d_q.data_ptr(), Qa, 2048, 0, d_ws.data_ptr(), wsb, d_rec.data_ptr(),
                                                     None, None, None, None, torch.cuda.current_stream().cuda_stream))
        mean_s, _ = timed(astar_run, reps=3, warm=1)
        arec = np.frombuffer(d_rec.cpu().numpy().tobytes(), dtype=aastar.ASTAR_RECORD_DTYPE)
        nthreads = orc.num_threads()
        qs = 8 * nthreads
        ow = orc.astar_world(world["circles"], world["boundary"], ga["centroid"], world["habitats"], bins_, ga["cells_rounded"], probs_)
        oq = np.column_stack([qa["start"], qa["path_len_limit"], qa["weights"], qa["velocity"]])[:qs]
        t0 = time.perf_counter()
        crec, _, cst = orc.astar_batch(ow, oq)
        ct = time.perf_counter() - t0
        out["lattice_astar"] = {"queries": Qa, "path_len_limit": 300.0, "queries_per_s": Qa / mean_s,
                                "expansions_per_s": float(arec["n_expanded"].sum()) / mean_s, "seconds": mean_s,
                                "ok_fraction": float((arec["status"] == 0).mean()), "kernel": "k_astar (fp64, warp per query)",
                                "cpu_port_queries_per_s": qs / ct, "cpu_port_expansions_per_s": float(crec[:, 0].sum()) / ct,
                                "cpu_cores": nthreads,
                                "note": "bit-identical to the reference; the Python reference needs ~14 s per query"}
        aenv.close()
    except Exception as ex:
        out["lattice_astar"] = {"error": repr(ex)}
    return out


if __name__ == "__main__":
    main()
