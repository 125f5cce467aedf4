"""GPU: kernel instantiations the Catalina-default tests never launch.

(1) fp32 planner variants on the Catalina map: the default fast kernels (the single-chunk warp-per-tree kernel, the
    thread-per-tree FAST form) against the generic instantiations the launchers pick for other worlds and
    parameters, forced by their switches.  The variants make the same decisions: identical traces.
(2) Batches past the first wave of resident trees / edge batches: workspace reuse in k_plan, slot refill in
    k_plan_tpt, the batch loop and the automatic 1024-thread shape of k_edges_arc_tpe, and the fp32 nearest-node scan
    on ragged sizes.  The sizes follow from hardware upper bounds (64 warps, 2048 threads per SM, 148 SMs), so they
    hold whatever the occupancy query returns.
(3) The fp32 planner against the fp32-stream oracle on the envelope worlds (envelope_worlds.py).
"""
import numpy as np
import pytest

import envelope_worlds as ew

pytestmark = pytest.mark.gpu

from oracle import orc  # noqa: E402

RTOL32 = 1e-5
TRACE_KEYS = ("parent", "safe", "nwp", "upos")


@pytest.fixture(scope="module")
def api():
    import auvrrt
    assert auvrrt.api.device_count() > 0
    return auvrrt.api


@pytest.fixture(scope="module")
def env(api):
    e = api.Env(**ew.assert_flags("catalina"))
    yield e
    e.close()


@pytest.fixture(scope="module")
def oworld():
    return orc.OracleWorld(**ew.build("catalina")[0])


def _starts(Q, seed=0):
    rs = np.random.RandomState(seed)
    s = np.tile([-200.0, 0.0, 0.0, 0.0, 0.0], (Q, 1))
    s[:, 0] += rs.uniform(-30, 30, Q)
    s[:, 1] += rs.uniform(-20, 20, Q)
    return s


def _same_plans(a, b, tag):
    for k in TRACE_KEYS:
        assert np.array_equal(a["trace"][k], b["trace"][k]), (tag, k)
    ra, rb = a["records"], b["records"]
    for k in ("status", "n_nodes", "n_uniforms", "n_waypoints", "n_cost_evals", "depth"):
        assert np.array_equal(ra[k], rb[k]), (tag, k)
    assert np.array_equal(a["chain"], b["chain"]), tag
    # the cost sums of one edge may be reduced in another lane order: the last bits only
    assert np.allclose(ra["cost"], rb["cost"], rtol=1e-6, atol=1e-7), tag


# ------------------------------------------------------------------------------------ (1) fp32 planner variants
VARIANTS = {"generic": {"AUVRRT_PLAN_GENERIC": "1"},             # MODE < 0: the mode read at run time
            "bins_global": {"AUVRRT_PLAN_BINS_GLOBAL": "1"},     # per-bin metadata in the tree workspace (BS = false)
            "stage_kb8": {"AUVRRT_PLAN_STAGE_KB": "8"}}          # nothing staged: the multi-chunk kernel on global loads


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_fp32_warp_planner_variants_agree(api, env, monkeypatch, mode):
    """groups 32 / 16 / 8 and the generic instantiations give the default kernel's decisions, in every parent-pick
    mode; freq = 40 (more primitives than lanes: chunked steer) likewise across groups"""
    Q, I = 48, 384
    starts, seeds = _starts(Q, mode), np.arange(Q) + 700 * (mode + 1)
    kw = dict(mode=mode, max_plan_time=5.0) if mode == 2 else dict(mode=mode)
    for extra in (dict(), dict(freq=40.0)):
        pp = dict(kw, **extra)
        base = api.plan_batch(env, starts, seeds, api.plan_params(I, trace=True, group=32, **pp), "f32")
        assert (base["records"]["n_nodes"] > 1).mean() > 0.9
        for G in (16, 8):
            _same_plans(base, api.plan_batch(env, starts, seeds, api.plan_params(I, trace=True, group=G, **pp), "f32"),
                        (mode, extra, G))
        for name, sw in VARIANTS.items():
            with monkeypatch.context() as m:
                for k, v in sw.items():
                    m.setenv(k, v)
                for G in (32, 8):
                    _same_plans(base, api.plan_batch(env, starts, seeds, api.plan_params(I, trace=True, group=G, **pp), "f32"),
                                (mode, extra, name, G))


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_fp32_thread_per_tree_generic_agrees(api, env, monkeypatch, mode):
    """the thread-per-tree planner's FAST form (straight-line lookups, hot part staged) against its generic form
    (nothing staged: AUVRRT_TPT_STAGE_KB=0), and 150 time bins (the bins' bitmap off)"""
    Q, I = 300, 256
    starts, seeds = _starts(Q, 10 + mode), np.arange(Q) + 9000 + 1000 * mode
    for extra in (dict(), dict(bin_interval=0.4, max_traj_time=60.0, v=0.5)):
        pp = api.plan_params(I, trace=True, group=1, mode=mode, **extra)
        fast = api.plan_batch(env, starts, seeds, pp, "f32")
        with monkeypatch.context() as m:
            m.setenv("AUVRRT_TPT_STAGE_KB", "0")
            _same_plans(fast, api.plan_batch(env, starts, seeds, pp, "f32"), (mode, extra))


# ------------------------------------------------------------------------------------ (2) past the first wave
def _resample_identical(api, env, starts, seeds, pp, prec, full, n=256):
    """re-run a sample of queries (the last 64 among them) in a batch of their own: the same records and chains"""
    Q = len(starts)
    rs = np.random.RandomState(Q)
    sub = np.unique(np.concatenate([rs.choice(Q - 64, n - 64, replace=False), np.arange(Q - 64, Q)]))
    r = api.plan_batch(env, starts[sub], seeds[sub], pp, prec)
    assert np.array_equal(r["records"], full["records"][sub])
    assert np.array_equal(r["chain"], full["chain"][sub])
    return sub


@pytest.mark.parametrize("G,Q,I,prec", [(32, 12_000, 256, "f32"), (8, 40_000, 128, "f32"), (32, 9_600, 48, "f64")])
def test_warp_planner_reuses_workspace(api, env, oworld, G, Q, I, prec):
    """more queries than lane groups can be resident (148 SMs x 2048 threads / G): every group plans several trees in
    its workspace slot, one after the other"""
    assert Q > 148 * 2048 // G
    starts, seeds = _starts(Q, G), np.arange(Q) + 123
    pp = api.plan_params(I, group=G)
    full = api.plan_batch(env, starts, seeds, pp, prec)
    rec = full["records"]
    assert set(np.unique(rec["status"])) <= {0, 1} and (rec["status"] == 0).any() and (rec["status"] == 1).any()
    sub = _resample_identical(api, env, starts, seeds, pp, prec, full)
    if prec == "f64":
        res, counts, status = orc.exploring_batch(oworld, starts[sub], seeds[sub], orc.plan_params(I))
        r = rec[sub]
        assert np.array_equal(r["status"], status)
        assert np.array_equal(r["n_nodes"], counts[:, 0]) and np.array_equal(r["n_cost_evals"], counts[:, 1])
        assert np.array_equal(r["n_waypoints"], counts[:, 2])
        ok = status == 0
        assert np.allclose(r["cost"][ok], res[ok, 1:], rtol=1e-9, atol=1e-12)
        assert np.allclose(r["path_length"][ok], res[ok, 0], rtol=1e-9)


def test_thread_per_tree_refills_slots(api, env):
    """320,000 trees on at most 148 x 2048 / 256 x 256 = 302,848 slots: slots take a second tree"""
    Q, I = 320_000, 96
    starts, seeds = _starts(Q, 5), np.arange(Q, dtype=np.uint64) * 7 + 11
    pp = api.plan_params(I, group=1)
    full = api.plan_batch(env, starts, seeds, pp, "f32")
    rec = full["records"]
    assert set(np.unique(rec["status"])) <= {0, 1} and (rec["n_nodes"] > 1).mean() > 0.95
    assert (rec["n_cost_evals"] > 0).any() and (rec["n_cost_evals"] == 0).any()
    _resample_identical(api, env, starts, seeds, pp, "f32", full)


def _arc_parents(n, seed):
    rs = np.random.RandomState(seed)
    p = np.stack([rs.uniform(-300, -100, n), rs.uniform(-60, 100, n), rs.uniform(-6, 6, n),
                  rs.uniform(0, 520, n), rs.uniform(0, 500, n)], 1)
    return p.astype(np.float32).astype(np.float64)


def _check_arc_vs_oracle(api, env, oworld, parents, seeds, out):
    safe, counts, leaf, _ = out
    ws, wn, wl = orc.edges_arc_batch(oworld, parents, seeds, velocity=2.0, f32u=True)
    n = len(parents)
    assert (safe != ws).sum() <= max(1, 0.002 * n) and (counts != wn).sum() <= max(1, 0.002 * n)
    ok = (counts == wn) & (safe == ws)
    d = np.abs(leaf[ok] - wl[ok])
    assert np.all(d[:, :2] <= RTOL32 * np.maximum(np.abs(wl[ok][:, :2]), 100.0))
    assert np.all(d[:, 2:] <= RTOL32 * np.maximum(np.abs(wl[ok][:, 2:]), 1.0))


def test_edges_arc_tpe_batch_loop(api, env, oworld):
    """3.2M edges in the automatic shape (1024-thread CTAs from 148 x 8192 edges on: each CTA sweeps the batch loop
    more than twice) against the same edges in 200k chunks (256-thread CTAs, one batch each); a 4,000-edge sample,
    the final batch among it, against the oracle; and ragged sizes around the warp and batch widths"""
    n = 3_200_000
    parents, seeds = _arc_parents(n, 31), np.arange(n, dtype=np.uint64) + 17
    params, w3 = [2.0, 0.5, 30.0, 0.5, 2.0], -4.0
    big = api.edges_arc_cost(env, parents, seeds, params, w3, "f32")
    step = 200_000
    for i in range(0, n, step):
        part = api.edges_arc_cost(env, parents[i:i + step], seeds[i:i + step], params, w3, "f32")
        for a, b in zip(big, part):
            assert np.array_equal(a[i:i + step], b), i
    rs = np.random.RandomState(2)
    sub = np.unique(np.concatenate([rs.choice(n, 3000, replace=False), np.arange(n - 1000, n)]))
    _check_arc_vs_oracle(api, env, oworld, parents[sub], seeds[sub], [a[sub] for a in big])
    for m in (1, 31, 33, 2047, 2049, 8191, 8193):
        p, s = _arc_parents(m, m), np.arange(m, dtype=np.uint64) + 3 * m
        _check_arc_vs_oracle(api, env, oworld, p, s, api.edges_arc_cost(env, p, s, params, w3, "f32"))


def _nn_numpy(tree, q):
    """orc.nn's rule restated: the lowest index among the smallest sqrt(dx*dx + dy*dy), in fp64"""
    d = np.sqrt((tree[:, 0] - q[0]) ** 2 + (tree[:, 1] - q[1]) ** 2)
    return int(np.argmin(d))


@pytest.mark.parametrize("n", [1, 2, 3, 5, 4097, 4098, 4099, 5_000_003])
def test_nn_fp32_ragged(api, n):
    """the fp32 scan: 16-byte loads of four nodes, the tail of n % 4 nodes, the fp32 pre-filter; duplicated nearest
    nodes (the lowest index wins) and a node equal to the query"""
    rs = np.random.RandomState(n % 1000)
    tree = rs.uniform(-500, 500, (n, 2)).astype(np.float32).astype(np.float64)
    for nq in (1, 2, 3, 4, 5, 9):
        qs = rs.uniform(-500, 500, (nq, 2)).astype(np.float32).astype(np.float64)
        t = tree.copy()
        if n >= 3:
            t[n - 1] = qs[0]                          # a node on the query, in the tail
            t[n // 2] = t[n // 3] = qs[-1] + [0.25, -0.5]     # the nearest node of the last query, twice
            t[0] = qs[-1] + [0.25, -0.5]                  # ... and once more at index 0 when nothing is nearer
            t = t.astype(np.float32).astype(np.float64)
        got = api.nn(t, qs, "f32")
        want = [orc.nn(t, q) if n < 100_000 else _nn_numpy(t, q) for q in qs]
        assert list(got) == want, (n, nq)


# ------------------------------------------------------------------------------------ (3) envelope worlds
ENVELOPE = [w for w in ew.NAMES if w not in ("catalina", "huge")]


@pytest.mark.parametrize("world", ENVELOPE)
def test_fp32_planner_first_divergence_envelope(api, world):
    """fp32 warp-per-tree and thread-per-tree planners against the oracle on the fp32 stream and fp32-rounded start,
    decision by decision, as test_gpu_parity's first-divergence test does on Catalina.  Measured on a B200 (1000 W):
    every world, both planners, 24 of 24 trees follow the oracle for all 256 iterations, except one tree of the offset
    world (warp per tree) that diverges between iterations 128 and 256."""
    w = ew.assert_flags(world)
    e = api.Env(**w)
    ow = orc.OracleWorld(**w)
    Q, I = 24, 256
    starts = ew.free_starts(world, Q, 3).astype(np.float32).astype(np.float64)
    seeds = np.arange(Q) + 31000
    for G in (32, 1):
        r = api.plan_batch(e, starts, seeds, api.plan_params(I, trace=True, group=G), "f32")["trace"]
        first = np.full(Q, I)
        for q in range(Q):
            o = orc.exploring(ow, starts[q], orc.plan_params(I), seed=int(seeds[q]), f32u=True)
            d = (r["parent"][q] != o["parent"]) | (r["safe"][q] != o["safe"]) | (r["nwp"][q] != o["nwp"])
            if d.any():
                first[q] = int(np.argmax(d))
            n = first[q]
            if n > 0:
                assert np.all(np.abs(r["leaf"][q][:n, :2] - o["leaf"][:n, :2]) <= 2e-5 * np.maximum(np.abs(o["leaf"][:n, :2]), 100.0))
        hist = np.histogram(first, bins=[0, 16, 64, 128, 256, 257])[0]
        print(world, G, "first divergence:", dict(zip(["<16", "<64", "<128", "<256", "never"], hist)))
        assert (first >= I).mean() >= 0.75 and (first < 64).mean() <= 0.05, (world, G, hist)
    e.close()
