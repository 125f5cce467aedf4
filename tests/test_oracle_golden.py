"""CPU: pin the fp64 C oracle (oracle/auvrrt_oracle.c) against golden vectors produced by the
UNMODIFIED reference (oracle/make_golden.py).  Bit-exact: same libm, no FMA contraction."""
import json
import os

import numpy as np
import pytest

from oracle import orc


@pytest.fixture(scope="module")
def world(catalina_map, shark_grid):
    bins, probs = shark_grid
    return orc.OracleWorld.from_map(catalina_map, bins, probs)


def test_stream_matches_harness():
    from oracle import harness as H
    for seed in (0, 1, 12345, 2**40 + 7):
        blk = H.stream_block(seed, 5, 64)
        blk23 = H.stream_block(seed, 5, 64, f32u=True)
        for j in range(64):
            assert orc.stream_u(seed, 5 + j) == blk[j] == H.stream_u53(seed, 5 + j)
            assert orc.stream_u(seed, 5 + j, True) == blk23[j] == H.stream_u23(seed, 5 + j)
            assert np.float32(blk23[j]) == blk23[j] and 0.0 <= blk23[j] < 1.0


def test_steer_arc_bit_exact(golden_dir):
    from oracle import harness as H
    z = np.load(os.path.join(golden_dir, "steer_arc.npz"))
    d2e, dmax, freq, mind = z["params"]
    n = len(z["parents"])
    for i in range(n):
        u = H.steer_arc_uniforms(i, int(z["uoff"][i + 1] - z["uoff"][i]))
        st, leaf, wp, used = orc.steer_arc(z["parents"][i], u, d2e, dmax, freq, mind, z["velocity"][i])
        assert st == orc.OK and used == len(u)
        assert np.array_equal(leaf, z["leaf"][i])
        ref_wp = z["wp"][z["woff"][i]:z["woff"][i + 1]]
        assert len(wp) + 1 == z["nwp"][i]
        assert np.array_equal(wp, ref_wp)


def test_collision_catalina_both_orders(golden_dir, catalina_map):
    z = np.load(os.path.join(golden_dir, "steer_arc.npz"))
    fwd = orc.OracleWorld.from_map(catalina_map)
    rev_map = dict(catalina_map, circles=list(reversed(catalina_map["circles"])))
    rev = orc.OracleWorld.from_map(rev_map)
    for i in range(len(z["parents"])):
        wp = z["wp"][z["woff"][i]:z["woff"][i + 1]]
        pts = np.vstack([z["parents"][i][None, :2], wp[:, :2]])
        assert orc.check_collision(pts, fwd) == z["safe_fwd"][i]
        assert orc.check_collision(pts, rev) == z["safe_rev"][i]
    assert z["safe_fwd"].sum() != z["safe_rev"].sum()  # the running-min quirk is order dependent


def test_collision_hand_cases(golden_dir):
    with open(os.path.join(golden_dir, "collision_hand.json")) as f:
        cases = json.load(f)
    for c in cases:
        w = orc.OracleWorld(circles=c["circles"], boundary=c["boundary"])
        assert bool(orc.check_collision(c["points"], w)) == c["safe"], c


def test_orient2d_exact_against_fractions():
    from fractions import Fraction as F
    rs = np.random.RandomState(7)
    for _ in range(3000):
        a, b = rs.uniform(-500, 500, 2), rs.uniform(-500, 500, 2)
        t = rs.uniform(0, 1)
        c = a + t * (b - a)                       # (nearly) collinear third point
        c = c + rs.choice([0.0, 1e-16, -1e-16, 1e-13], 2) * np.abs(c)
        d = (F(a[0]) - F(c[0])) * (F(b[1]) - F(c[1])) - (F(a[1]) - F(c[1])) * (F(b[0]) - F(c[0]))
        want = (d > 0) - (d < 0)
        assert orc.lib().orc_orient2d(a[0], a[1], b[0], b[1], c[0], c[1]) == want


def test_nn_golden(golden_dir):
    z = np.load(os.path.join(golden_dir, "nn.npz"))
    for i in range(int(z["n"])):
        tree, qs, idx = z["tree%d" % i], z["q%d" % i], z["idx%d" % i]
        for q, want in zip(qs, idx):
            assert orc.nn(tree, q) == want


def test_cost_golden(golden_dir, catalina_map, shark_grid):
    bins, probs = shark_grid
    z = np.load(os.path.join(golden_dir, "cost.npz"))
    for i in range(len(z["t_total"])):
        m = dict(catalina_map, habitats=catalina_map["habitats"][:int(z["n_hab"][i])])
        w = orc.OracleWorld.from_map(m, bins, probs)
        pts = z["pts"][z["off"][i]:z["off"][i + 1]]
        out = orc.cost(pts, z["t_total"][i], w, z["weights"][i])
        assert np.array_equal(out, z["out"][i]), (i, out, z["out"][i])


def test_cost_hand_cases(golden_dir):
    with open(os.path.join(golden_dir, "cost_hand.json")) as f:
        cases = json.load(f)
    for c in cases:
        bins = [g[0] for g in c["grid"]]
        cells = [cb for cb, _ in c["grid"][0][1]] if c["grid"] else []
        probs = [[p for _, p in g[1]] for g in c["grid"]]
        w = orc.OracleWorld(habitats=c["habitats"], bins=bins, cells=cells,
                            probs=probs if c["grid"] else None)
        out = orc.cost(c["points"], c["t_total"], w, c["weights"])
        assert np.array_equal(out, np.array(c["out"], dtype=np.float64)), c


def test_exploring_traces_bit_exact(exploring_golden, world):
    z, meta = exploring_golden
    for m in meta:
        tag = m["tag"]
        pp = orc.plan_params(m["iterations"], mode={"A": 0, "B": 1, "C": 2}[m["mode"]], max_plan_time=10.0)
        r = orc.exploring(world, [m["start"][0], m["start"][1], 0.0, 0.0, 0.0], pp, seed=m["seed"])
        assert r["status"] == (orc.OK if m["found"] else orc.NO_PATH)
        assert np.array_equal(r["parent"], z[tag + "_parent"])
        assert np.array_equal(r["safe"], z[tag + "_safe"])
        assert np.array_equal(r["nwp"], z[tag + "_nwp"])
        assert np.array_equal(r["upos"], z[tag + "_upos"])
        assert r["n_uniforms"] == m["n_uniforms"] and r["n_nodes"] == m["nodes"]
        if tag + "_leaf" in z:
            assert np.array_equal(r["leaf"], z[tag + "_leaf"])
        else:
            assert np.array_equal(r["leaf"][::16], z[tag + "_leaf_stride"])
        assert np.array_equal(r["cost_evals"], z[tag + "_cost_evals"])
        if m["found"]:
            assert np.array_equal(r["result"], z[tag + "_result"])
            assert np.array_equal(r["path"], z[tag + "_path"])
