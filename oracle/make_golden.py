"""TEST INFRASTRUCTURE ONLY -- writes tests/golden/* by running the UNMODIFIED reference.

Run in the build container (needs /root/reference):   python oracle/make_golden.py
The reference has no tests and no golden vectors of its own (SURVEY.md section 4), so every
fixture here is an output of the reference's own functions under oracle/harness.py:

  catalina_map.json   Cartesian map from catalina.create_environs (catalina.py:32-65) + lattice cells
  shark_grid.npz      createSharkGrid (rrt_dubins.py:612-630) on shark_data/AUVGrid_prob_500_turn.csv
  steer_arc.npz       RRT.steer (rrt_dubins.py:237-295) on recorded uniform streams
  collision.npz       RRT.check_collision (rrt_dubins.py:530-549), both obstacle orders + hand cases
  cost.npz            cost.habitat_shark_cost_func (cost.py:145-207) on recorded paths + hand cases
  nn.npz              RRT.get_closest_mps (rrt_dubins.py:505-513) incl. exact ties
  exploring.npz       RRT.exploring traces (rrt_dubins.py:92-176), time-bin mode and NN mode
"""
import io
import json
import math
import os
import sys
import zipfile

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import harness as H  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
GRID_CSV = os.path.join(H.REFERENCE_ROOT, "path_planning", "shark_data", "AUVGrid_prob_500_turn.csv")


def ragged(list_of_arrays, width):
    off = np.zeros(len(list_of_arrays) + 1, dtype=np.int64)
    for i, a in enumerate(list_of_arrays):
        off[i + 1] = off[i] + len(a)
    flat = (np.concatenate([np.asarray(a, dtype=np.float64).reshape(-1, width)
                            for a in list_of_arrays], axis=0)
            if list_of_arrays else np.zeros((0, width)))
    return off, flat


def savez_lzma(path, **arrays):
    """np.savez with LZMA instead of deflate (np.load reads both): keeps the larger fixtures under 1 MB"""
    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_LZMA) as zf:
        for name, a in arrays.items():
            buf = io.BytesIO()
            np.lib.format.write_array(buf, np.asanyarray(a), allow_pickle=False)
            zf.writestr(name + ".npy", buf.getvalue())


def random_state_in_polygon(ref, poly, rs):
    minx, miny, maxx, maxy = poly.bounds
    while True:
        x, y = rs.uniform(minx, maxx), rs.uniform(miny, maxy)
        if ref.Point(x, y).within(poly):
            return x, y


def main():
    os.makedirs(OUT, exist_ok=True)
    ref = H.load_reference()
    MPS = ref.MPS
    mod = ref.rrt_dubins

    # ---- map -------------------------------------------------------------------------------
    world = H.catalina_world(ref)
    with open(os.path.join(OUT, "catalina_map.json"), "w") as f:
        json.dump(world, f, indent=0)
    obstacles, poly, habitats, cells, shark = H.world_objects(ref, world, grid_csv=GRID_CSV)
    bins, probs = H.shark_arrays(shark, cells)
    np.savez_compressed(os.path.join(OUT, "shark_grid.npz"), bins=bins, probs=probs)
    print("map: K=%d E=%d H=%d C=%d T=%d" % (len(obstacles), len(world["boundary"]), len(habitats),
                                               len(cells), len(bins)))

    rrt = ref.RRT(poly, obstacles, shark, cells)
    rrt.t_start = 0.0
    rs = np.random.RandomState(20261017)

    # ---- steer + collision -----------------------------------------------------------------
    N = 1500
    parents, ustreams, leaves, wps, nwp = [], [], [], [], []
    safe_fwd, safe_rev = [], []
    saved = (mod.random, mod.time)
    mod.time = H.BudgetClock(1 << 60)
    obstacles_rev = list(reversed(obstacles))
    velocities = []
    try:
        for i in range(N):
            x, y = random_state_in_polygon(ref, poly, rs)
            th = rs.uniform(-12.0, 12.0)
            t0 = rs.uniform(0.0, 480.0)
            ln = rs.uniform(0.0, 900.0)
            v = [1.0, 2.0, 0.5][i % 3]
            parent = MPS(x, y, theta=th, traj_time_stamp=t0, length=ln)
            player = H.RecordingRandom(i) if i % 5 == 4 else H.StreamPlayer(seed=1000 + i)
            mod.random = player
            new = rrt.steer(parent, 2, 0.5, 30, 0.5, v, True)
            used = (np.array(player.log) if isinstance(player, H.RecordingRandom)
                    else H.stream_block(1000 + i, 0, player.pos))
            assert np.array_equal(used, H.steer_arc_uniforms(i, len(used)))   # so only the counts are stored
            parents.append([x, y, th, t0, ln])
            velocities.append(v)
            ustreams.append(used.reshape(-1, 1))
            leaves.append([new.x, new.y, new.theta, new.traj_time_stamp, new.length])
            nwp.append(len(new.path))
            wps.append(H.path_to_array(new.path[1:]))
            safe_fwd.append(rrt.check_collision(new, obstacles))
            safe_rev.append(rrt.check_collision(new, obstacles_rev))
    finally:
        mod.random, mod.time = saved
    uoff, uflat = ragged(ustreams, 1)
    woff, wflat = ragged(wps, 6)
    savez_lzma(
        os.path.join(OUT, "steer_arc.npz"), parents=np.array(parents), velocity=np.array(velocities),
        params=np.array([2.0, 0.5, 30.0, 0.5]), uoff=uoff, leaf=np.array(leaves),
        nwp=np.array(nwp, dtype=np.int32), woff=woff, wp=wflat,
        safe_fwd=np.array(safe_fwd, dtype=np.uint8), safe_rev=np.array(safe_rev, dtype=np.uint8))
    print("steer: %d edges, %d uniforms, %d waypoints, safe %d / %d (rev %d)" % (
        N, len(uflat), len(wflat), sum(safe_fwd), N, sum(safe_rev)))

    # ---- collision hand cases (explicit paths) ----------------------------------------------
    # running-min quirk (rrt_dubins.py:535-542): dList is never reset between obstacles.
    hand = []

    def cc(points, circles, boundary):
        p = ref.Polygon(boundary)
        r = ref.RRT(p, [MPS(c[0], c[1], size=c[2]) for c in circles], {}, [])
        node = MPS(points[-1][0], points[-1][1])
        node.path = [MPS(q[0], q[1]) for q in points]
        return bool(r.check_collision(node, r.obstacle_list))

    big = [(-1000.0, -1000.0), (1000.0, -1000.0), (1000.0, 1000.0), (-1000.0, 1000.0)]
    sq = [(0.0, 0.0), (10.0, 0.0), (10.0, 10.0), (0.0, 10.0)]
    lshape = [(0.0, 0.0), (10.0, 0.0), (10.0, 4.0), (4.0, 4.0), (4.0, 10.0), (0.0, 10.0)]
    cases = [
        ([(3.0, 0.0)], [(0.0, 0.0, 1.0), (100.0, 0.0, 5.0)], big),     # unsafe via running min
        ([(3.0, 0.0)], [(100.0, 0.0, 5.0), (0.0, 0.0, 1.0)], big),     # safe in reversed order
        ([(3.0, 0.0)], [(0.0, 0.0, 3.0)], big),                        # d == r collides (<=)
        ([(3.0, 0.0)], [(0.0, 0.0, 2.9999999999999996)], big),         # just outside
        ([(5.0, 5.0)], [], sq),                                        # inside
        ([(0.0, 5.0)], [], sq),                                        # on an edge -> not within
        ([(10.0, 10.0)], [], sq),                                      # on a vertex -> not within
        ([(5.0, 0.0)], [], sq),                                        # on a horizontal edge
        ([(5.0, 5.0), (11.0, 5.0)], [], sq),                           # second point outside
        ([(2.0, 8.0)], [], lshape), ([(8.0, 8.0)], [], lshape),        # concave polygon
        ([(4.0, 7.0)], [], lshape), ([(7.0, 4.0)], [], lshape),        # on reflex edges
        ([(4.0, 4.0)], [], lshape), ([(3.999999999999999, 3.9999999999999996)], [], lshape),
        ([(2.0, 4.0)], [], lshape),                                    # level with a vertex, inside
        ([(1e-300, 5.0)], [], sq), ([(5.0, 9.999999999999998)], [], sq),
    ]
    # a point within rounding distance of a slanted edge, both sides (exact predicate needed)
    a, b = (0.1, 0.1), (0.7, 0.3)
    tri = [a, b, (0.2, 0.9)]
    for tt in (0.25, 0.5, 0.75):
        px = a[0] + tt * (b[0] - a[0])
        py = a[1] + tt * (b[1] - a[1])
        for dy in (0.0, 1.4e-17, -1.4e-17, 5.6e-17, -5.6e-17):
            cases.append(([(px, py + dy)], [], tri))
    for pts, circ, bnd in cases:
        hand.append({"points": [list(p) for p in pts], "circles": [list(c) for c in circ],
                     "boundary": [list(p) for p in bnd], "safe": cc(pts, circ, bnd)})
    with open(os.path.join(OUT, "collision_hand.json"), "w") as f:
        json.dump(hand, f)
    print("collision hand cases:", [int(h["safe"]) for h in hand])

    # ---- nearest node ---------------------------------------------------------------------
    nn_cases = []
    for n in (1, 2, 7, 33, 257, 1500, 4096):
        tx = rs.uniform(-467, 82, n)
        ty = rs.uniform(-153, 191, n)
        if n >= 7:  # exact ties: duplicate nodes and mirror-image nodes
            tx[5], ty[5] = tx[2], ty[2]
            tx[n - 1], ty[n - 1] = tx[3], ty[3]
        nodes = [MPS(float(a_), float(b_)) for a_, b_ in zip(tx, ty)]
        qs, idx = [], []
        for k in range(24):
            if k == 0 and n >= 7:
                q = (float(tx[2]), float(ty[2]))
            elif k == 1 and n >= 7:  # equidistant from nodes 0 and 1 exactly (midpoint on a grid)
                tx[0], ty[0], tx[1], ty[1] = -100.0, 20.0, -96.0, 20.0
                nodes[0], nodes[1] = MPS(-100.0, 20.0), MPS(-96.0, 20.0)
                q = (-98.0, 20.0 + 1e-9 * 0)
            else:
                q = (float(rs.uniform(-467, 82)), float(rs.uniform(-153, 191)))
            got = rrt.get_closest_mps(MPS(q[0], q[1]), nodes)
            qs.append(q)
            idx.append([i for i, m in enumerate(nodes) if m is got][0])
        nn_cases.append((np.array([[m.x, m.y] for m in nodes]), np.array(qs), np.array(idx)))
    np.savez_compressed(os.path.join(OUT, "nn.npz"),
                        **{"tree%d" % i: c[0] for i, c in enumerate(nn_cases)},
                        **{"q%d" % i: c[1] for i, c in enumerate(nn_cases)},
                        **{"idx%d" % i: c[2].astype(np.int32) for i, c in enumerate(nn_cases)},
                        n=np.array(len(nn_cases)))

    # ---- exploring traces -------------------------------------------------------------------
    ex = {}
    paths_for_cost = []
    specs = []
    for s in range(16):
        specs.append(("A", s, (-200.0, 0.0), 2048 if s < 8 else 512))
    for s in range(16, 24):
        x, y = random_state_in_polygon(ref, ref.Polygon([(-300, -100), (-100, -100), (-100, 100), (-300, 100)]), rs)
        while not ref.Point(x, y).within(poly):
            x, y = rs.uniform(-300, -100), rs.uniform(-100, 100)
        specs.append(("A", s, (float(x), float(y)), 1024))
    for s in range(32, 40):
        specs.append(("B", s, (-200.0, 0.0), 1024 if s < 36 else 384))
    for s in range(48, 52):
        specs.append(("C", s, (-200.0, 0.0), 768))      # wall-clock parent pick on the simulated clock (N4)
    meta = []
    for mode, seed, start, iters in specs:
        rrt = ref.RRT(poly, obstacles, shark, cells)
        res, tr = H.traced_exploring(
            ref, rrt, MPS(start[0], start[1]), habitats, iterations=iters,
            rng=H.StreamPlayer(seed=seed), bin_interval=5, v=2, shark_interval=50,
            traj_time_stamp=(mode != "C"), max_plan_time=10.0, max_traj_time=500.0,
            plan_time=(mode != "B"), weights=(-3, -3, -4))
        tag = "%s%d" % (mode, seed)
        ex[tag + "_parent"] = tr["parent"].astype(np.int16)
        ex[tag + "_safe"] = tr["safe"]
        ex[tag + "_nwp"] = tr["nwp"].astype(np.uint8)
        ex[tag + "_upos"] = tr["upos"].astype(np.int32)
        ex[tag + "_cost_evals"] = tr["cost_evals"]
        if seed % 8 < 2:
            ex[tag + "_leaf"] = tr["leaf"]
        else:
            ex[tag + "_leaf_stride"] = tr["leaf"][::16]
        if res is not None:
            ex[tag + "_path"] = H.path_to_array(res["path"][0])
            ex[tag + "_result"] = np.array([res["path length"], res["cost"][0]] + list(res["cost"][1]))
            paths_for_cost.append((res["path"][0], res["path"][0][-1].traj_time_stamp))
            split = res["path"][1]
            ex[tag + "_split_counts"] = np.array([len(v_) for v_ in split.values()], dtype=np.int32)
        meta.append({"tag": tag, "mode": mode, "seed": seed, "start": list(start),
                     "iterations": iters, "n_uniforms": int(tr["n_uniforms"]),
                     "nodes": int(tr["safe"].sum()) + 1, "found": res is not None,
                     "cost": None if res is None else res["cost"][0]})
        print(meta[-1])
    ex["meta"] = np.array(json.dumps(meta))
    savez_lzma(os.path.join(OUT, "exploring.npz"), **ex)

    # ---- cost ---------------------------------------------------------------------------------
    cost_mod = ref.cost
    cpaths, ctime, cweights, cout, chab = [], [], [], [], []
    wsets = [(-3, -3, -4), (-1, -1, -1), (1, 0.5, 2), (-3, -3, -4)]
    for i, (path, tleaf) in enumerate(paths_for_cost):
        w = wsets[i % len(wsets)]
        order = list(reversed(path)) if i % 2 == 0 else list(path)   # leaf->root as the planner calls it
        habs = habitats if i % 3 else habitats[:4]
        c = cost_mod.habitat_shark_cost_func(order, tleaf, habs, shark, list(w))
        cpaths.append(np.array([[p.x, p.y, p.traj_time_stamp] for p in order]))
        ctime.append(tleaf)
        cweights.append(w)
        chab.append(len(habs))
        cout.append([c[0]] + list(c[1]))
    coff, cflat = ragged(cpaths, 3)
    np.savez_compressed(os.path.join(OUT, "cost.npz"), off=coff, pts=cflat, t_total=np.array(ctime),
                        weights=np.array(cweights, dtype=np.float64), n_hab=np.array(chab),
                        out=np.array(cout))
    # hand cases incl. the `x <= maxy` typo (cost.py:182) and the no-bin skip (cost.py:178-179)
    hand = []

    def hc(points, t_total, habs, grid, w):
        path = [MPS(p[0], p[1], traj_time_stamp=p[2]) for p in points]
        hl = [MPS(h[0], h[1], size=h[2]) for h in habs]
        sd = {}
        for (t0, t1), cellsp in grid:
            sd[(t0, t1)] = {tuple(cb): pr for cb, pr in cellsp}
        c = cost_mod.habitat_shark_cost_func(path, t_total, hl, sd, list(w))
        hand.append({"points": points, "t_total": t_total, "habitats": habs,
                     "grid": [[[t0, t1], [[list(cb), pr] for cb, pr in cellsp]] for (t0, t1), cellsp in grid],
                     "weights": list(w), "out": [c[0]] + list(c[1])})

    g2 = [((0, 100), [((0, 0, 10, 10), 0.5), ((0, 10, 10, 20), 0.25)])]
    hc([[5.0, 15.0, 1.0]], 10.0, [], g2, (-3, -3, -4))              # typo: first cell wins -> -0.2
    hc([[5.0, 15.0, 500.0]], 10.0, [[5.0, 15.0, 3.0]], g2, (-3, -3, -4))  # no bin -> skipped entirely
    hc([[15.0, 5.0, 1.0]], 10.0, [], g2, (-3, -3, -4))              # x outside -> no match
    hc([[9.0, 25.0, 1.0], [9.5, 0.0, 2.0]], 0.0, [[9.0, 25.0, 1.0], [9.0, 25.0, 5.0]], g2, (2, 3, 5))
    hc([[1.0, 1.0, 50.0], [1.0, 1.0, 50.0]], 7.0, [[0.0, 0.0, 2.0]],
       [((0, 50), [((0, 0, 10, 10), 0.5)]), ((50, 100), [((0, 0, 10, 10), 0.125)])], (-3, -3, -4))
    hc([], 5.0, [[0.0, 0.0, 2.0]], g2, (-3, -3, -4))
    hc([[3.0, 0.0, 1.0]], 4.0, [[0.0, 0.0, 3.0], [3.0, 0.0, 1.0]], [], (-3, -3, -4))  # empty dict: skip
    hc([[12.0, 0.5, 1.0]], 4.0, [], [((0, 10), [((0, 0, 20, 11), 1.0), ((0, 0, 20, 30), 2.0)])], (-1, -1, -1))
    with open(os.path.join(OUT, "cost_hand.json"), "w") as f:
        json.dump(hand, f)
    print("cost: %d paths; hand outs %s" % (len(cpaths), [h["out"][0] for h in hand]))


if __name__ == "__main__":
    main()
