"""GPU: the planner kernels (warp per tree, 16/8-lane groups, thread per tree) against the fp64
oracle on parameter sets the golden traces do not cover: more arc primitives than lanes (chunked
steer), the time-bin reset quirk (max_traj_time not a multiple of bin_interval), other bin widths /
velocities / weights, no shark grid, no habitats, no obstacles, a non-convex boundary, nearest-node
mode with few iterations, and starts that cannot grow a tree."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import envelope_worlds as ew  # noqa: E402
from oracle import orc  # noqa: E402


@pytest.fixture(scope="module")
def api():
    import auvrrt
    assert auvrrt.api.device_count() > 0
    return auvrrt.api


@pytest.fixture(scope="module")
def env(api, catalina_map, shark_grid):
    e = api.Env.from_map(catalina_map, shark_grid[0], shark_grid[1])
    yield e
    e.close()


@pytest.fixture(scope="module")
def oworld(catalina_map, shark_grid):
    return orc.OracleWorld.from_map(catalina_map, shark_grid[0], shark_grid[1])


def _compare(api, env, ow, starts, seeds, kw, groups=(32, 1), iters=200):
    okw = dict(kw)
    pp_o = orc.plan_params(iters, **okw)
    want = [orc.exploring(ow, s, pp_o, seed=int(sd)) for s, sd in zip(starts, seeds)]
    for G in groups:
        pp = api.plan_params(iters, trace=True, chain_cap=200, group=G, **kw)
        r = api.plan_batch(env, starts, seeds, pp, "f64")
        for j, o in enumerate(want):
            rec = r["records"][j]
            assert rec["status"] == o["status"], (G, j, rec["status"], o["status"])
            if o["status"] in (orc.OK, orc.NO_PATH):
                for k in ("parent", "safe", "nwp", "upos"):
                    assert np.array_equal(r["trace"][k][j], o[k]), (G, j, k)
                assert np.allclose(r["trace"]["leaf"][j], o["leaf"], rtol=1e-9, atol=1e-9)
                assert rec["n_nodes"] == o["n_nodes"] and rec["n_uniforms"] == o["n_uniforms"]
                assert rec["n_cost_evals"] == len(o["cost_evals"])
            if o["status"] == orc.OK:
                assert rec["best_iter"] == o["best_iter"]
                assert np.allclose(rec["cost"], o["result"][1:], rtol=1e-9, atol=1e-12)
                assert abs(rec["path_length"] - o["result"][0]) <= 1e-9 * max(1.0, o["result"][0])
    return want


def test_parameter_sets_on_catalina(api, catalina_map, shark_grid):
    bins, probs = shark_grid
    env = api.Env.from_map(catalina_map, bins, probs)
    ow = orc.OracleWorld.from_map(catalina_map, bins, probs)
    starts = np.array([[-200.0, 0.0, 0.0, 0.0, 0.0], [-150.0, 40.0, 1.0, 0.0, 0.0], [-250.0, 60.0, -2.0, 12.5, 3.0]])
    seeds = [11, 12, 13]
    sets = [
        dict(freq=50.0),                                            # up to 49 primitives: chunked steer in every group size
        dict(freq=70.0, dist_to_end=1.0, diff_max=0.9),             # many invalid primitives, 3 chunks of 32
        dict(max_traj_time=498.0),                                  # bin 100 is re-created on every overflow insert (:149-150)
        dict(max_traj_time=123.0, bin_interval=7.0, v=1.0),
        dict(bin_interval=0.4, max_traj_time=60.0, v=0.5),          # 150 bins: per-bin metadata in global memory (BS = false)
        dict(weights=(0.1, -0.7, 1.3)),
        dict(min_dist=0.0), dict(min_dist=1.5),
        dict(mode=1), dict(mode=1, freq=40.0, max_traj_time=120.0),
        dict(mode=2, max_plan_time=5.0), dict(mode=2, max_plan_time=0.7, freq=12.0, max_traj_time=90.0),
    ]
    for kw in sets:
        _compare(api, env, ow, starts, seeds, kw, groups=(32, 16, 8, 1))


def test_degenerate_worlds(api, catalina_map, shark_grid):
    bins, probs = shark_grid
    starts = np.array([[-200.0, 0.0, 0.0, 0.0, 0.0], [-100.0, -20.0, 0.5, 0.0, 0.0]])
    seeds = [5, 6]
    worlds = [
        dict(circles=[], boundary=catalina_map["boundary"], habitats=catalina_map["habitats"], bins=bins,
             cells=catalina_map["cells"], probs=probs),                                   # no obstacles
        dict(circles=catalina_map["circles"], boundary=catalina_map["boundary"], habitats=[], bins=bins,
             cells=catalina_map["cells"], probs=probs),                                   # no habitats (H == 0, cost.py:204)
        dict(circles=catalina_map["circles"], boundary=catalina_map["boundary"], habitats=catalina_map["habitats"]),   # no shark grid
        dict(circles=catalina_map["circles"][:3], habitats=catalina_map["habitats"][:2], bins=bins[:2],
             cells=catalina_map["cells"][:50], probs=probs[:2, :50],
             boundary=[[-400.0, -100.0], [50.0, -100.0], [50.0, 150.0], [-150.0, 150.0], [-150.0, 20.0], [-400.0, 20.0]]),  # non-convex
    ]
    for w in worlds:
        env = api.Env(**w)
        ow = orc.OracleWorld(**w)
        _compare(api, env, ow, starts, seeds, dict(max_traj_time=150.0), iters=300)
        _compare(api, env, ow, starts, seeds, dict(max_traj_time=150.0, mode=1), iters=150)
        env.close()


@pytest.mark.parametrize("world", [w for w in ew.NAMES if w != "catalina"])
def test_envelope_worlds(api, world):
    """the envelope worlds (envelope_worlds.py): fp64 traces of every group size in every parent-pick mode, exact"""
    w = ew.assert_flags(world)
    env = api.Env(**w)
    ow = orc.OracleWorld(**w)
    starts = ew.free_starts(world, 2, 7)
    I = 96 if world == "huge" else 200
    for kw in (dict(max_traj_time=150.0), dict(max_traj_time=150.0, mode=1), dict(max_traj_time=150.0, mode=2, max_plan_time=3.0)):
        _compare(api, env, ow, starts, [5, 6], kw, groups=(32, 16, 8, 1), iters=I)
    env.close()


def test_trees_that_cannot_grow(api, catalina_map, shark_grid):
    bins, probs = shark_grid
    env = api.Env.from_map(catalina_map, bins, probs)
    ow = orc.OracleWorld.from_map(catalina_map, bins, probs)
    starts = np.array([[9.39, -3.2, 0.0, 0.0, 0.0],        # inside an obstacle
                       [500.0, 500.0, 0.0, 0.0, 0.0],      # outside the boundary (and outside the grid)
                       [-200.0, 0.0, 0.0, 600.0, 0.0]])    # already past the horizon: overflow bin only
    want = _compare(api, env, ow, starts, [1, 2, 3], dict(), iters=64)
    assert [w["status"] for w in want[:2]] == [orc.NO_PATH, orc.NO_PATH]


def test_fp32_thread_per_tree_vs_warp_per_tree(api, catalina_map, shark_grid):
    """the two fp32 planners order their arithmetic differently, so trees diverge; both must still be
    valid planners: same statuses, similar tree sizes and costs over a batch"""
    bins, probs = shark_grid
    env = api.Env.from_map(catalina_map, bins, probs)
    Q = 512
    starts = np.tile([-200.0, 0.0, 0.0, 0.0, 0.0], (Q, 1))
    seeds = np.arange(Q)
    a = api.plan_batch(env, starts, seeds, api.plan_params(1024, group=32), "f32")["records"]
    b = api.plan_batch(env, starts, seeds, api.plan_params(1024, group=1), "f32")["records"]
    assert np.all(a["status"] == 0) and np.all(b["status"] == 0)
    assert abs(a["n_nodes"].mean() - b["n_nodes"].mean()) < 0.02 * a["n_nodes"].mean()
    assert abs(a["cost"][:, 0].mean() - b["cost"][:, 0].mean()) < 0.1
    assert np.mean(a["n_uniforms"] == b["n_uniforms"]) > 0.02        # some trees stay identical for all 1024 steps


# ------------------------------------------------------------------------------------ mode 3: Dubins-RRT, best parent
def _mode3_params(api_or_orc, iters, **kw):
    return api_or_orc.plan_params(iters, mode=3, v=1.0, max_traj_time=200.0, dubins_rho=1.0, dubins_eta=20.0,
                                  near_radius=15.0, dubins_w=12, **kw)


def test_mode3_dubins_best_parent_f64_matches_oracle(api, env, oworld):
    """planner mode 3 (six-word Dubins steer toward the sample + best-parent selection; the build's own definition,
    parity unpinned) in the fp64 build against its independent oracle restatement, decision by decision"""
    Q, I = 6, 384
    starts = np.tile([-200.0, 0.0, 0.0, 0.0, 0.0], (Q, 1))
    starts[3:, :2] = [[-150.0, 40.0], [-250.0, -20.0], [-120.0, -40.0]]
    seeds = np.arange(Q) + 900
    r = api.plan_batch(env, starts, seeds, _mode3_params(api, I, trace=True, path_cap=2048, chain_cap=255), "f64")
    n_found = 0
    for q in range(Q):
        o = orc.exploring(oworld, starts[q], _mode3_params(orc, I), seed=int(seeds[q]))
        assert np.array_equal(r["trace"]["parent"][q], o["parent"]), q          # chosen parents (-1: no safe candidate)
        assert np.array_equal(r["trace"]["safe"][q], o["safe"]) and np.array_equal(r["trace"]["upos"][q], o["upos"])
        assert np.allclose(r["trace"]["leaf"][q], o["leaf"], rtol=1e-9, atol=1e-9)
        rec = r["records"][q]
        assert rec["status"] == o["status"] and rec["n_nodes"] == o["n_nodes"] and rec["n_cost_evals"] == len(o["cost_evals"])
        assert rec["n_waypoints"] == o["n_waypoints_total"]
        if o["status"] == 0:
            n_found += 1
            assert rec["best_iter"] == o["best_iter"] and rec["best_node"] == o["best_node"]
            assert np.allclose(rec["cost"], o["result"][1:], rtol=1e-9, atol=1e-12)
            assert np.isclose(rec["path_length"], o["result"][0], rtol=1e-9)
            assert rec["n_path"] == o["n_path"]
            assert np.allclose(r["path"][q][:o["n_path"]], o["path"], rtol=1e-9, atol=1e-9)
            # ... and the same path re-created from (start, seed, chain)
            pp = _mode3_params(api, I, path_cap=2048, chain_cap=255)
            rows, n_path = api.materialize(env, starts[q:q + 1], seeds[q:q + 1], r["chain"][q:q + 1], r["records"]["depth"][q:q + 1], pp, "f64")
            assert n_path[0] == o["n_path"] and np.allclose(rows[0, :n_path[0]], o["path"], rtol=1e-9, atol=1e-9)
            # the incremental cost equals cost.habitat_shark_cost_func on the explicit path (leaf -> root order)
            pth = o["path"][::-1]
            want = orc.cost(pth[:, [0, 1, 4]], float(pth[0, 4]), oworld, [-3.0, -3.0, -4.0])
            assert np.allclose(rec["cost"], want, rtol=1e-9, atol=1e-12)
    assert n_found >= 3


def test_mode3_dubins_best_parent_f32(api, env, oworld):
    """fp32 build of mode 3: valid plans, statistics close to the fp64 build's"""
    Q, I = 64, 512
    starts = np.tile([-200.0, 0.0, 0.0, 0.0, 0.0], (Q, 1))
    seeds = np.arange(Q) + 5000
    r32 = api.plan_batch(env, starts, seeds, _mode3_params(api, I, path_cap=2048, chain_cap=255), "f32")["records"]
    r64 = api.plan_batch(env, starts, seeds, _mode3_params(api, I), "f64")["records"]
    assert (r32["status"] <= 1).all() and (r32["status"] == 0).mean() > 0.7
    assert abs(r32["n_nodes"].mean() - r64["n_nodes"].mean()) < 0.05 * r64["n_nodes"].mean()
    ok = (r32["status"] == 0) & (r64["status"] == 0)
    assert abs(r32["cost"][ok, 0].mean() - r64["cost"][ok, 0].mean()) < 0.1 * abs(r64["cost"][ok, 0].mean())
    # the first iterations of a tree are decided identically (same sample, one or two candidates)
    same_first = (r32["n_waypoints"] > 0).all()
    assert same_first
