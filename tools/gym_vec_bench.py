"""Throughput of the device-resident vectorised RRTEnv (gym_rrt.envs.DeviceVecRRTEnv) against the host loop
through VecRRTEnv, on main()'s course (gym_rrt/envs/rrt_dubins.py: (0, 0, 50, 50), the seven obstacles of
oracle.harness.GYM_MAIN_OBSTACLES, freq = 10, 2 m cells x 8 subsections = 5000 actions, fp32, 200-step episodes).

Two device policies, timed apart from the env with CUDA events:
  uniform   a uniform random sub-cell id: most name an empty cell, so this is the env's overhead floor;
  occupied  a random occupied sub-cell, argmax of noise x (obs > 0), as an agent acting on the observation would.
Per configuration one JSON line goes to OUT/gym_vec_bench.jsonl: env calls/s and episode steps/s, the policy's time,
the per-step device time of k_gym_reset_masked and k_gym_run from a torch.profiler run of its own, library
launches per step (auvrrt_launch_count), episodes finished per second, and the GPU's name and power limit read in
the same run.  Not bench.py: that measures the flagship planner.

  python tools/gym_vec_bench.py --out DIR [--Q 4096,65536,262144] [--steps 300] [--warmup 30]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "auv-sim_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

from auvrrt import api  # noqa: E402
from gym_rrt.envs import DeviceVecRRTEnv, VecRRTEnv  # noqa: E402
from oracle.harness import GYM_MAIN_OBSTACLES  # noqa: E402

WORLD = dict(boundary=(0, 0, 50, 50), obstacles=GYM_MAIN_OBSTACLES)
ENV_KW = dict(freq=10, cell_side_length=2, subsections_in_cell=8, precision="f32", max_nodes=201)
MAX_EPISODE_STEPS = 200


def episodes(Q, seed=1):
    rs = np.random.default_rng(seed)
    starts = np.column_stack([rs.uniform(5, 15, Q), rs.uniform(5, 15, Q), rs.uniform(-np.pi, np.pi, Q)])
    goals = np.column_stack([rs.uniform(35, 45, Q), rs.uniform(35, 45, Q)])
    return starts, goals, np.arange(Q, dtype=np.uint64) + 1000


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_w"] = float(out.splitlines()[0])
    except Exception as e:  # the number is then reported as unknown, not guessed
        info["power_limit_error"] = repr(e)
    return info


def make_policy(name, n_actions, gen):
    if name == "uniform":
        return lambda obs: torch.randint(0, n_actions, (obs.shape[0],), device=obs.device, generator=gen, dtype=torch.int32)
    # torch has no uint16 comparison; node counts stay below 2^15, so the int16 view is exact
    return lambda obs: torch.argmax(torch.rand(obs.shape, device=obs.device, generator=gen) * (obs.view(torch.int16) > 0),
                                    dim=1).to(torch.int32)


def kernel_ms(prof, name, n):
    tot = 0.0
    for e in prof.key_averages():
        if name in e.key:
            tot += getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
    return tot / 1e3 / n


def run_device(Q, policy_name, steps, warmup, prof_steps):
    env = DeviceVecRRTEnv(WORLD["boundary"], WORLD["obstacles"], Q, max_episode_steps=MAX_EPISODE_STEPS, **ENV_KW)
    s, g, sd = episodes(Q)
    obs = env.reset(s, g, sd)
    gen = torch.Generator(device="cuda").manual_seed(0)
    policy = make_policy(policy_name, env.n_actions, gen)
    for _ in range(warmup):
        obs, *_ = env.step(policy(obs))
    finished = torch.zeros((), dtype=torch.int64, device="cuda")
    terminated = torch.zeros((), dtype=torch.int64, device="cuda")
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
    torch.cuda.synchronize()
    l0 = api.launch_count()
    for i in range(steps):
        ev[i][0].record()
        act = policy(obs)
        ev[i][1].record()
        obs, rew, term, trunc, info = env.step(act)
        ev[i][2].record()
        finished += (term | trunc).sum()
        terminated += term.sum()
    torch.cuda.synchronize()
    launches = api.launch_count() - l0
    pol_ms = sum(e[0].elapsed_time(e[1]) for e in ev)
    env_ms = sum(e[1].elapsed_time(e[2]) for e in ev)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(prof_steps):
            obs, *_ = env.step(policy(obs))
        torch.cuda.synchronize()
    r = {"kind": "device", "Q": Q, "policy": policy_name, "steps": steps,
         "env_ms_per_step": env_ms / steps, "env_calls_per_s": steps / (env_ms / 1e3),
         "episode_steps_per_s": Q * steps / (env_ms / 1e3),
         "policy_ms_per_step": pol_ms / steps,
         "reset_kernel_ms_per_step": kernel_ms(prof, "k_gym_reset_masked", prof_steps),
         "run_kernel_ms_per_step": kernel_ms(prof, "k_gym_run", prof_steps),
         "launches_per_step": launches / steps,
         "episodes_finished_per_s": int(finished) / (env_ms / 1e3),
         "episodes_terminated_per_s": int(terminated) / (env_ms / 1e3),
         "episodes_finished": int(finished)}
    env.close()
    return r


def run_host(Q, policy_name, steps, warmup):
    env = VecRRTEnv(WORLD["boundary"], WORLD["obstacles"], Q, **ENV_KW)
    s, g, sd = episodes(Q)
    obs = env.reset(s, g, sd)
    rs = np.random.default_rng(0)

    def policy(obs):
        if policy_name == "uniform":
            return rs.integers(0, env.n_actions, Q).astype(np.int32)
        return np.argmax((obs > 0) * rs.random(obs.shape, dtype=np.float32), axis=1).astype(np.int32)

    for _ in range(warmup):
        obs, *_ = env.step(policy(obs))
    pol = tot = 0.0
    for _ in range(steps):
        t0 = time.perf_counter()
        act = policy(obs)
        t1 = time.perf_counter()
        obs, rew, done, recs = env.step(act)          # ends in a device synchronise (records and counts copied back)
        t2 = time.perf_counter()
        pol += t1 - t0
        tot += t2 - t1
    env.close()
    return {"kind": "host_VecRRTEnv", "Q": Q, "policy": policy_name, "steps": steps, "env_ms_per_step": tot * 1e3 / steps,
            "env_calls_per_s": steps / tot, "episode_steps_per_s": Q * steps / tot,
            "policy_ms_per_step": pol * 1e3 / steps, "obs_bytes_per_step": 2 * Q * env.n_actions}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True)
    ap.add_argument("--Q", default="4096,65536,262144")
    ap.add_argument("--host-Q", default="4096,65536")
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=30)
    ap.add_argument("--prof-steps", type=int, default=50)
    ap.add_argument("--host-steps", type=int, default=10)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gym_vec_bench: no CUDA device (this measures the GPU; there is no CPU fallback)")
    os.makedirs(a.out, exist_ok=True)
    info = gpu_info()
    path = os.path.join(a.out, "gym_vec_bench.jsonl")
    with open(path, "w") as f:
        def emit(r):
            r.update(info)
            line = json.dumps(r)
            print(line, flush=True)
            f.write(line + "\n")
            f.flush()
        for Q in [int(x) for x in a.Q.split(",") if x]:
            for pol in ("uniform", "occupied"):
                emit(run_device(Q, pol, a.steps, a.warmup, a.prof_steps))
        for Q in [int(x) for x in a.host_Q.split(",") if x]:
            for pol in ("uniform", "occupied"):
                emit(run_host(Q, pol, a.host_steps, 2))
    print("wrote", path)


if __name__ == "__main__":
    main()
