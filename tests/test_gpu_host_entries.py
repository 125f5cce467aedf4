"""GPU: the host-buffer entries of the C ABI (api.cu) and the device check of the handle constructors.

(A) One call of each host-buffer entry launches a fixed number of kernels: the entry's own, plus in fp32 one
    k_convert per non-empty real input and one k_convert_back per real output that is copied back.  The counts are
    pinned, so a change to how the entries stage their buffers cannot add or drop a conversion unnoticed.
(B) A device ordinal past the last device is AUVRRT_ERR_ARG for the gym and lattice-A* constructors, as it is for
    every api.cu entry.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SP5 = [2.0, 0.5, 30.0, 0.5, 2.0]
W3 = -4.0
START = [-200.0, 0.0, 0.0, 0.0, 0.0]

# entry -> (launches in fp64, launches in fp32)
LAUNCHES = {
    "nn": (2, 6),
    "steer_arc": (1, 4),
    "steer_dubins": (1, 6),
    "steer_dubins_no_waypoints": (1, 5),
    "collide": (1, 2),
    "collide_points": (1, 2),
    "cost": (1, 4),
    "cost_point": (1, 3),
    "edges_dubins": (1, 4),
    "edges_dubins_cost": (1, 5),
    "edges_arc": (1, 3),
    "edges_arc_cost": (1, 4),
    "plan_batch": (1, 1),
    "materialize": (1, 3),
}


@pytest.fixture(scope="module")
def api():
    import auvrrt
    assert auvrrt.api.device_count() > 0
    return auvrrt.api


@pytest.fixture(scope="module")
def env(api, catalina_map, shark_grid):
    e = api.Env.from_map(catalina_map, *shark_grid)
    yield e
    e.close()


def _calls(api, env, prec):
    rs = np.random.RandomState(11)
    n = 64
    parents = np.tile(START, (n, 1)) + np.column_stack([rs.uniform(-20, 20, (n, 2)), rs.uniform(-3, 3, n), np.zeros((n, 2))])
    seeds = np.arange(n) + 500
    q0 = parents[:, :3]
    q1 = q0 + np.column_stack([rs.uniform(-10, 10, (n, 2)), rs.uniform(-3, 3, n)])
    paths = [parents[i:i + 1, :2] + rs.uniform(-5, 5, (8, 2)) for i in range(n)]
    timed = [np.column_stack([p, np.linspace(0, 50, len(p))]) for p in paths]
    u = rs.uniform(0, 1, 100 * n)
    uoff = np.arange(n + 1) * 100
    pp = api.plan_params(64, path_cap=64)
    Q = 8
    starts, qseeds = np.tile(START, (Q, 1)), np.arange(Q)

    def materialize():
        r = api.plan_batch(env, starts, qseeds, pp, prec)
        depth = r["records"]["depth"]
        ok = (depth >= 0) & (depth <= pp.chain_cap)
        assert ok.any()
        return lambda: api.materialize(env, starts[ok], qseeds[ok], r["chain"][ok], depth[ok], pp, prec)

    return {
        "nn": lambda: api.nn(parents[:, :2], q1[:3, :2], prec),
        "steer_arc": lambda: api.steer_arc(parents, u, uoff, SP5, prec),
        "steer_dubins": lambda: api.steer_dubins(q0, q1, 1.0, 8, prec),
        "steer_dubins_no_waypoints": lambda: api.steer_dubins(q0, q1, 1.0, 0, prec),
        "collide": lambda: api.collide(env, paths, prec),
        "collide_points": lambda: api.collide_points(env, parents[:, :2], prec),
        "cost": lambda: api.cost(env, timed, np.full(n, 60.0), [-3.0, -3.0, -4.0], precision=prec),
        "cost_point": lambda: api.cost_point(env, parents[:, :2], np.zeros(64, np.uint8), 1, [-3.0, -3.0, -4.0], prec),
        "edges_dubins": lambda: api.edges_dubins(env, q0, q1, 1.0, 20, prec),
        "edges_dubins_cost": lambda: api.edges_dubins_cost(env, q0, q1, 1.0, 20, 1.0, W3, prec),
        "edges_arc": lambda: api.edges_arc(env, parents, seeds, SP5, prec),
        "edges_arc_cost": lambda: api.edges_arc_cost(env, parents, seeds, SP5, W3, prec),
        "plan_batch": lambda: api.plan_batch(env, starts, qseeds, pp, prec),
        "materialize": materialize(),
    }


@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("entry", sorted(LAUNCHES))
def test_host_entry_launch_count(api, env, entry, prec):
    call = _calls(api, env, prec)[entry]
    l0 = api.launch_count()
    call()
    assert api.launch_count() - l0 == LAUNCHES[entry][prec == "f32"]


def test_constructors_reject_a_device_past_the_last(api, catalina_map, shark_grid):
    from auvrrt import AuvrrtError, astar, gym
    past = api.device_count()
    with pytest.raises(AuvrrtError, match=r"out of range .*\(status 1\)"):
        gym.GymBatch((0, 0, 50, 50), [(12.0, 38.0, 4.0)], 4, device=past)
    bins, probs = shark_grid
    cells = np.tile([-250.0, -50.0, -240.0, -40.0], (probs.shape[1], 1))
    with pytest.raises(AuvrrtError, match=r"out of range .*\(status 1\)"):
        astar.AstarEnv(catalina_map["circles"], catalina_map["boundary"], catalina_map["habitats"], bins, cells, probs,
                       device=past)
