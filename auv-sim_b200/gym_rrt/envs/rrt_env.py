"""Drop-in for gym_rrt/envs/rrt_env.py of auv-sim (/root/reference/gym_rrt/envs/rrt_env.py:86-452): the
environment whose action is "grow the tree from this sub-cell".  `RRTEnv` keeps the reference's
single-episode surface (init_env / reset / step(chosen_grid_cell_idx, step_num) -> state, reward, done,
info) without needing `gym` or matplotlib; `VecRRTEnv` is the same environment for Q episodes stepped
in one kernel launch, which is what the GPU is for; `DeviceVecRRTEnv` keeps those Q episodes and their
observations on the GPU as torch tensors and resets each one in place when it ends.  No CPU fallback."""
import numpy as np

from gym_rrt.envs.rrt_dubins import Planner_RRT
from auvrrt import gym as _gym

RRT_PLANNER_FREQ = 10            # rrt_env.py:27
R_FOUND_PATH, R_CREATE_NODE, R_INVALID_NODE = 300, 0, -1      # rrt_env.py:40-42


class RRTEnv:
    metadata = {'render.modes': ['human']}

    def __init__(self):
        self.auv_init_pos = None
        self.shark_init_pos = None
        self.state = None
        self.obstacle_array = []
        self.obstacle_array_for_rendering = []
        self.habitats_array_for_rendering = []
        self.rrt_planner = None
        self.precision = "f32"
        self.seed_value = None
        # nodes one episode may hold (start included).  The reference's tree is unbounded and its RL drivers step an
        # episode up to 1000 times (2000 at test time, solveRL-RRT.py:35-36), each step adding at most one node, so the
        # default leaves room for the longest of those; init_env(max_steps=...) changes it.
        self.max_steps = 2000
        self._episode = 0

    def seed(self, seed=None):
        self.seed_value = seed

    def init_env(self, auv_init_pos, shark_init_pos, boundary_array, grid_cell_side_length, num_of_subsections,
                 obstacle_array=[], habitat_grid=None, max_steps=None):
        if max_steps is not None:
            self.max_steps = int(max_steps)
        self.auv_init_pos = auv_init_pos
        self.shark_init_pos = shark_init_pos
        self.obstacle_array_for_rendering = obstacle_array
        self.habitats_array_for_rendering = [] if habitat_grid is None else habitat_grid.habitat_array
        self.obstacle_array = np.array([[o.x, o.y, o.z, o.size] for o in obstacle_array])
        self.boundary_array = boundary_array
        self.cell_side_length = grid_cell_side_length
        self.num_of_subsections = num_of_subsections
        return self.reset()

    def _grid_rows(self):
        """[cell.x, cell.y, subsection.theta] for every sub-cell in env_grid order (rrt_env.py:250-263)"""
        rows = []
        for row in self.rrt_planner.env_grid:
            for cell in row:
                for sub in cell.subsection_cells:
                    rows.append([cell.x, cell.y, sub.theta])
        return np.array(rows, dtype=np.float64).reshape(-1, 3)

    def _observe(self):
        counts = self.rrt_planner.node_counts().astype(np.int64)
        self.state["rrt_grid"] = np.column_stack([self._static_grid, counts.astype(np.float64)])
        self.state["has_node"] = (counts > 0).astype(np.int64)
        self.state["rrt_grid_num_of_nodes_only"] = counts

    def reset(self):
        a, s = self.auv_init_pos, self.shark_init_pos
        self.rrt_planner = Planner_RRT(a, s, self.boundary_array, self.obstacle_array_for_rendering,
                                       self.habitats_array_for_rendering, cell_side_length=self.cell_side_length,
                                       freq=RRT_PLANNER_FREQ, subsections_in_cell=self.num_of_subsections,
                                       seed=None if self.seed_value is None else self.seed_value + self._episode,
                                       precision=self.precision, track_counts=True, node_cap=self.max_steps + 1)
        self._episode += 1            # a seeded env replays a different stream every episode
        self._static_grid = self._grid_rows()
        self.state = {'auv_pos': np.array([a.x, a.y, a.z, a.theta]), 'shark_pos': np.array([s.x, s.y, s.z, s.theta]),
                      'obstacles_pos': self.obstacle_array, 'path': None}
        self._observe()
        return self.state

    def step(self, chosen_grid_cell_idx, step_num=None):
        """chosen_grid_cell_idx = (row * cols + col) * subsections + subsection (rrt_env.py:206-222)"""
        done, path = self.rrt_planner.generate_one_node(int(chosen_grid_cell_idx), step_num)
        self._observe()
        if path is not None:
            self.state["path"] = path
        if done and path is not None:
            reward = R_FOUND_PATH
        elif path is not None:
            reward = R_CREATE_NODE
        else:
            reward = R_INVALID_NODE
        return self.state, reward, done, {}


class VecRRTEnv:
    """Q RRTEnv episodes stepped together (one launch per step)."""

    def __init__(self, boundary, obstacles, n_envs, *, cell_side_length=2, subsections_in_cell=8, freq=RRT_PLANNER_FREQ,
                 max_nodes=257, precision="f32", device=0, **planner_kw):
        circles = [(float(o.x), float(o.y), float(o.size)) if hasattr(o, "x") else tuple(map(float, o)) for o in obstacles]
        b = boundary
        rect = (b[0].x, b[0].y, b[1].x, b[1].y) if hasattr(b[0], "x") else tuple(map(float, b))
        self.batch = _gym.GymBatch(rect, circles, n_envs, freq=freq, cell_side_length=cell_side_length,
                                   subsections_in_cell=subsections_in_cell, node_cap=max_nodes, track_counts=True,
                                   precision=_gym.F64 if precision == "f64" else _gym.F32, device=device, **planner_kw)
        self.n_envs = int(n_envs)
        self.n_actions = self.batch.n_subcells

    def reset(self, starts, goals, seeds):
        """starts [Q][3] = x, y, theta; goals [Q][2] -> observation counts [Q][n_actions] (uint16)"""
        self.batch.reset(starts, goals, seeds)
        return self.batch.counts()

    def step(self, actions, observe=True):
        """-> (counts or None, rewards [Q], done [Q] bool, records)"""
        recs = self.batch.step(actions)
        return (self.batch.counts() if observe else None), _gym.GymBatch.rewards(recs), recs["done"] != 0, recs

    def path(self, q):
        return self.batch.path(q)

    def close(self):
        self.batch.close()


_SEED_MASK = (1 << 63) - 1


class DeviceVecRRTEnv:
    """Q RRTEnv episodes resident on the GPU, stepped with torch CUDA tensors and reset one by one as they end.

    Every tensor stays on the device and `step` never synchronises with the host: it enqueues one masked reset
    (episodes that ended in the previous step), one step of every episode and a few elementwise torch ops on the
    current stream.  Auto-reset follows gymnasium's "next-step" mode: an episode that ends in step t reports its
    terminal observation in step t; in step t+1 it starts over (its action is ignored) and that step reports
    reward 0, terminated = truncated = False and info["reset"] = True.

    Episode e of slot q (e = 0 is the one `reset` starts) uses the seed (seeds[q] + e * Q) & (2**63 - 1), so
    seeds = base + arange(Q) keeps every episode's sample sequence distinct.  `starts` [Q, 3] and `goals` [Q, 2]
    (float64, on the device) are read at each slot's reset; overwrite them in place to give the next episode of a
    slot a new start or goal."""

    def __init__(self, boundary, obstacles, n_envs, *, cell_side_length=2, subsections_in_cell=8, freq=RRT_PLANNER_FREQ,
                 max_nodes=257, precision="f32", device=0, max_episode_steps=200, **planner_kw):
        import torch
        circles = [(float(o.x), float(o.y), float(o.size)) if hasattr(o, "x") else tuple(map(float, o)) for o in obstacles]
        b = boundary
        rect = (b[0].x, b[0].y, b[1].x, b[1].y) if hasattr(b[0], "x") else tuple(map(float, b))
        self.batch = _gym.GymBatch(rect, circles, n_envs, freq=freq, cell_side_length=cell_side_length,
                                   subsections_in_cell=subsections_in_cell, node_cap=max_nodes, track_counts=True,
                                   precision=_gym.F64 if precision == "f64" else _gym.F32, device=device, **planner_kw)
        self.n_envs = Q = int(n_envs)
        self.n_actions = self.batch.n_subcells
        self.max_episode_steps = int(max_episode_steps)
        self.device = dev = torch.device("cuda", device)
        self.starts = torch.zeros((Q, 3), dtype=torch.float64, device=dev)
        self.goals = torch.zeros((Q, 2), dtype=torch.float64, device=dev)
        self.seeds = torch.zeros(Q, dtype=torch.int64, device=dev)            # uint64 bit patterns
        self.episode = torch.zeros(Q, dtype=torch.int64, device=dev)          # episodes started in each slot - 1
        self.elapsed = torch.zeros(Q, dtype=torch.int32, device=dev)          # step calls since the slot's reset
        self.records = torch.zeros((Q, _gym.GYM_RECORD_DTYPE.itemsize), dtype=torch.uint8, device=dev)
        self._ended = torch.zeros(Q, dtype=torch.bool, device=dev)            # ended in the last step: reset in the next
        self.obs = _dev().gym_counts_tensor(self.batch)
        self._ready = False

    def _to_dev(self, a, dtype, shape):
        import torch
        t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))
        return t.to(device=self.device, dtype=dtype).reshape(shape)

    def reset(self, starts, goals, seeds):
        """Full reset of every slot: starts [Q, 3] = x, y, theta; goals [Q, 2]; seeds [Q] (arrays or tensors; uint64
        values, or int64 bit patterns).  -> the observation: the live uint16 counts view [Q, n_actions]."""
        import torch
        Q = self.n_envs
        self.starts.copy_(self._to_dev(starts, torch.float64, (Q, 3)))
        self.goals.copy_(self._to_dev(goals, torch.float64, (Q, 2)))
        if not isinstance(seeds, torch.Tensor):
            seeds = torch.from_numpy(np.ascontiguousarray(np.asarray(seeds, dtype=np.uint64).reshape(Q)).view(np.int64))
        elif seeds.dtype == torch.uint64:
            seeds = seeds.view(torch.int64)
        self.seeds.copy_(seeds.to(device=self.device, dtype=torch.int64).reshape(Q))
        self.episode.zero_()
        self.elapsed.zero_()
        self._ended = torch.zeros_like(self._ended)
        _dev().gym_reset_dev(self.batch, None, self.starts, self.goals, self.seeds & _SEED_MASK)
        self._ready = True
        return self.obs

    def step(self, actions):
        """actions: int32 CUDA tensor [Q] of flat sub-cell ids.  -> (obs, reward, terminated, truncated, info):
        obs is the live uint16 counts view [Q, n_actions], OVERWRITTEN by the next step (clone it to keep it);
        reward float32 (300 goal reached, 0 node added, -1 otherwise: RRTEnv.step); terminated bool (goal reached);
        truncated bool (max_episode_steps step calls since the slot's reset, or a status != 0: the episode can no
        longer step); info["reset"] bool (the slot started a new episode in this step), info["status"] int32
        (AUVRRT_ST_*), info["records"] the raw uint8 [Q, 88] gym records (overwritten by the next step too)."""
        import torch
        if not self._ready:
            raise RuntimeError("DeviceVecRRTEnv.step before reset")
        D = _dev()
        D._need("actions", actions, (torch.int32,), (self.n_envs,), self.device)
        stream = torch.cuda.current_stream(self.device)
        was_reset = self._ended
        self.episode += was_reset
        seeds = (self.seeds + self.episode * self.n_envs) & _SEED_MASK
        D.gym_reset_dev(self.batch, was_reset, self.starts, self.goals, seeds, stream)
        acts = torch.where(was_reset, -1, actions).to(torch.int32)
        D.gym_step_dev(self.batch, acts, self.records, stream)
        fields = self.records.view(torch.int32)                  # [Q, 22]: GYM_RECORD_DTYPE's int32 words
        status = fields[:, 0].clone()
        live = ~was_reset
        self.elapsed = torch.where(was_reset, 0, self.elapsed + 1)
        terminated = (fields[:, 1] != 0) & live
        truncated = ((self.elapsed >= self.max_episode_steps) | (status != 0)) & live
        reward = torch.where(fields[:, 1] != 0, float(R_FOUND_PATH),
                             torch.where(fields[:, 6] != 0, float(R_CREATE_NODE), float(R_INVALID_NODE)))
        reward = torch.where(live, reward, 0.0).to(torch.float32)
        self._ended = terminated | truncated
        return self.obs, reward, terminated, truncated, {"reset": was_reset, "status": status, "records": self.records}

    def path(self, q):
        return self.batch.path(q)

    def close(self):
        self.batch.close()


def _dev():
    from auvrrt import device
    return device
