"""GPU: the device-resident entry points bench.py times, and auvrrt_materialize, which config 5 and the
thread-per-tree planner rely on for paths.

(A) auvrrt_plan_batch_dev (auvrrt.device.DevicePlanner) launches the kernels auvrrt_plan_batch launches, so its
    records, chains and paths equal the host entry's byte for byte: at the headline shape, across workspace reuse,
    partial batches, the caller's stream, seeds with the high bit set and without the optional buffers.
(B) auvrrt_materialize re-creates the in-kernel path bit for bit in every parent-pick mode, precision and group
    size, and for thread-per-tree chains; overflowed chains, short path buffers and plans without a path.
(C) The _dev edge entries and nn_dev against their host entries, on Catalina and on the warp-per-edge world.
"""
import ctypes as C

import numpy as np
import pytest
import torch

import envelope_worlds as ew

pytestmark = pytest.mark.gpu

from oracle import orc  # noqa: E402

SENTINEL = 0xA5
ERR_ARG = 1
ST_OK, ST_NO_PATH, ST_OVERFLOW = 0, 1, 5


@pytest.fixture(scope="module")
def api():
    import auvrrt
    assert auvrrt.api.device_count() > 0 and torch.cuda.is_available()
    return auvrrt.api


@pytest.fixture(scope="module")
def adev(api):
    from auvrrt import device
    return device


@pytest.fixture(scope="module")
def worlds(api):
    """(Env, OracleWorld) of catalina, coast, offset (and huge for the edge kernels), built once per module"""
    cache = {}

    def get(name):
        if name not in cache:
            w = ew.assert_flags(name)
            cache[name] = (api.Env(**w), orc.OracleWorld(**w))
        return cache[name]
    yield get
    for e, _ in cache.values():
        e.close()


@pytest.fixture(scope="module")
def cat(worlds):
    return worlds("catalina")


@pytest.fixture(scope="module")
def bench_queries():
    import bench               # config 2's starts and seeds, exactly as the benchmark makes them
    return bench.make_queries


# ------------------------------------------------------------------------------------ helpers
def _fill(t):
    if t is not None:
        t.view(torch.uint8).fill_(SENTINEL)


def _launch(pl, stream=None):
    for t in (pl.records, pl.chain, pl.path):
        _fill(t)
    pl.launch(stream)
    torch.cuda.synchronize()


def _dev_out(pl, n):
    """(records uint8 [Q, 96], chain uint32 or None, path in the build's float type or None) of all max_queries rows"""
    rec = pl.records.cpu().numpy()
    chain = pl.chain.cpu().numpy().view(np.uint32) if pl.chain is not None else None
    path = pl.path.cpu().numpy() if pl.path is not None else None
    return rec, chain, path


def _path_mask(n_path, cap):
    return np.arange(cap)[None, :] < np.minimum(n_path, cap)[:, None]


def _assert_equals_host(out, want, n, tag=""):
    """rows < n equal the host entry byte for byte (paths over the rows each query wrote)"""
    rec, chain, path = out
    hrec = want["records"]
    assert np.array_equal(rec[:n], hrec.view(np.uint8).reshape(n, -1)), ("records", tag)
    if chain is not None:
        assert np.array_equal(chain[:n], want["chain"]), ("chain", tag)
    if path is not None:
        m = _path_mask(hrec["n_path"], path.shape[1])
        assert np.array_equal(path[:n].astype(np.float64)[m], want["path"][m]), ("path", tag)


def _assert_sentinel_tail(out, n, tag=""):
    for a in out:
        if a is not None:
            assert (a[n:].view(np.uint8) == SENTINEL).all(), ("rows >= n were written", tag)


def _records(raw):
    from auvrrt.api import RECORD_DTYPE
    return np.ascontiguousarray(raw).view(RECORD_DTYPE).reshape(-1)


# ------------------------------------------------------------------------------------ (A) auvrrt_plan_batch_dev
def test_headline_shape_equals_host_entry(api, adev, cat, bench_queries):
    """bench.py's headline: 4096 queries x 2048 iterations, group 0, fp32, launched three times on one planner as the
    warm-up does; then fp64 at 256 iterations, a 64-query sample of it against the fp64 oracle"""
    env, ow = cat
    Q = 4096
    starts, seeds = bench_queries(0, Q)
    for prec, I in (("f32", 2048), ("f64", 256)):
        pp = api.plan_params(I)
        want = api.plan_batch(env, starts, seeds, pp, prec)
        pl = adev.DevicePlanner(env, pp, prec, Q, want_chain=True)
        pl.set_queries(starts, seeds)
        for k in range(3):
            _launch(pl)
            _assert_equals_host(_dev_out(pl, Q), want, Q, (prec, k))
        rec = want["records"]
        print(prec, "status OK:", int((rec["status"] == 0).sum()), "of", Q)
        assert (rec["status"] == 0).mean() > 0.5
    sub = np.random.RandomState(7).choice(Q, 64, replace=False)
    res, counts, status = orc.exploring_batch(ow, starts[sub], seeds[sub], orc.plan_params(256))
    r = _records(_dev_out(pl, Q)[0][sub])
    assert np.array_equal(r["status"], status) and (status == 0).any()
    assert np.array_equal(r["n_nodes"], counts[:, 0]) and np.array_equal(r["n_cost_evals"], counts[:, 1])
    assert np.array_equal(r["n_waypoints"], counts[:, 2])
    ok = status == 0
    assert np.allclose(r["cost"][ok], res[ok, 1:], rtol=1e-9, atol=1e-12)
    assert np.allclose(r["path_length"][ok], res[ok, 0], rtol=1e-9)


def test_workspace_reuse_across_batches(api, adev, cat, bench_queries):
    """batch A, then batch B (other starts and seeds), then A again on one workspace: A's bytes"""
    env, _ = cat
    Q = 4096
    sa, da = bench_queries(0, Q)
    sb, db = bench_queries(Q, 2 * Q)
    sb = sb[::-1].copy()
    pp = api.plan_params(512, path_cap=256)
    want = api.plan_batch(env, sa, da, pp, "f32")
    pl = adev.DevicePlanner(env, pp, "f32", Q, want_chain=True, want_path=True)
    pl.set_queries(sa, da)
    _launch(pl)
    first = _dev_out(pl, Q)
    _assert_equals_host(first, want, Q, "A")
    pl.set_queries(sb, db)
    _launch(pl)
    _assert_equals_host(_dev_out(pl, Q), api.plan_batch(env, sb, db, pp, "f32"), Q, "B")
    pl.set_queries(sa, da)
    _launch(pl)
    again = _dev_out(pl, Q)
    for a, b in zip(first, again):
        assert np.array_equal(a, b)


PARTIAL = {4096: (0, 1, 33, 4095), 65536: (1000, 32767, 32768, 65536)}


@pytest.mark.parametrize("group,want_path", [(0, False), (0, True), (32, False), (32, True), (1, False)])
def test_partial_batches_and_workspace_sizing(api, adev, cat, bench_queries, group, want_path):
    """a planner built for max_queries plans every n <= max_queries in the workspace auvrrt_plan_workspace_bytes_q
    sized: rows < n equal the host entry for those n queries, rows >= n keep their sentinel bytes, n = 0 launches
    nothing.  Group 0 switches kernels within one planner: one warp per tree below 32768 queries or with paths, one
    thread per tree from 32768 queries on."""
    env, _ = cat
    starts, seeds = bench_queries(0, 65536)
    pp = api.plan_params(32, max_traj_time=60.0, path_cap=48 if want_path else 0, group=group)
    lib = __import__("auvrrt")._lib.lib()
    sizes = {q: lib.auvrrt_plan_workspace_bytes_q(env.handle, C.byref(pp), 0, q) for q in (0, 4096, 32768, 65536)}
    print("group", group, "want_path", want_path, "workspace bytes by max_queries:", sizes)
    for cap, ns in PARTIAL.items():
        pl = adev.DevicePlanner(env, pp, "f32", cap, want_chain=True, want_path=want_path)
        assert pl.workspace.numel() <= sizes[0]
        for n in ns:
            pl.set_queries(starts[:n], seeds[:n])
            l0 = api.launch_count()
            _launch(pl)
            out = _dev_out(pl, n)
            _assert_sentinel_tail(out, n, (cap, n))
            if n == 0:
                assert api.launch_count() == l0
                continue
            want = api.plan_batch(env, starts[:n], seeds[:n], pp, "f32")
            _assert_equals_host(out, want, n, (cap, n))
            rec = want["records"]
            if n >= 1000:
                assert (rec["status"] == ST_OK).any() and (rec["status"] == ST_NO_PATH).any(), (cap, n)


def test_launch_runs_on_the_callers_stream(api, adev, cat, bench_queries):
    """on a side stream: ~50 ms of sleep, then the starts are written, then the launch.  Waiting on that stream alone,
    the result is the host entry's for the new starts; a launch on another stream would plan the stale ones"""
    env, _ = cat
    Q = 4096
    stale, seeds = bench_queries(0, Q)
    fresh = stale[::-1].copy()
    pp = api.plan_params(256)
    want = api.plan_batch(env, fresh, seeds, pp, "f32")
    pl = adev.DevicePlanner(env, pp, "f32", Q, want_chain=True)
    pl.set_queries(stale, seeds)
    fresh_dev = torch.from_numpy(fresh).to(device=pl.dev, dtype=pl.rdtype)
    for t in (pl.records, pl.chain):
        _fill(t)
    torch.cuda.synchronize()
    side = torch.cuda.Stream(device=pl.dev)
    with torch.cuda.stream(side):
        torch.cuda._sleep(100_000_000)
        pl.starts.copy_(fresh_dev)
        pl.launch(side)
    side.synchronize()
    rec = pl.records.to("cpu", non_blocking=False).numpy()
    chain = pl.chain.cpu().numpy().view(np.uint32)
    _assert_equals_host((rec, chain, None), want, Q)


@pytest.mark.parametrize("prec", ["f32", "f64"])
def test_seeds_with_the_high_bit_set(api, adev, cat, bench_queries, prec):
    """seeds travel as int64 bit patterns: 2^63 + k and 2^64 - 1 - k plan as the host entry's uint64 seeds"""
    env, _ = cat
    Q = 256
    starts, _ = bench_queries(0, Q)
    k = np.arange(Q // 2, dtype=np.uint64)
    seeds = np.concatenate([np.uint64(1 << 63) + k, np.uint64((1 << 64) - 1) - k])
    pp = api.plan_params(512)
    want = api.plan_batch(env, starts, seeds, pp, prec)
    pl = adev.DevicePlanner(env, pp, prec, Q, want_chain=True)
    pl.set_queries(starts, seeds)
    _launch(pl)
    _assert_equals_host(_dev_out(pl, Q), want, Q)
    assert len(np.unique(want["records"]["n_uniforms"])) > Q // 2        # distinct streams, not one seed repeated


@pytest.mark.parametrize("group", [32, 1])
def test_records_without_a_chain_buffer(api, adev, cat, bench_queries, group):
    """want_chain=False gives the chained records wherever depth <= chain_cap; with chain_cap = 8 the deeper plans are
    OVERFLOW with a chain and OK without one, and nothing else in their records differs"""
    env, _ = cat
    Q = 512
    starts, seeds = bench_queries(0, Q)
    for ccap in (96, 8):
        pp = api.plan_params(1024, chain_cap=ccap, group=group)
        pls = [adev.DevicePlanner(env, pp, "f32", Q, want_chain=w) for w in (True, False)]
        for pl in pls:
            pl.set_queries(starts, seeds)
            _launch(pl)
        rc, rn = (_records(pl.records.cpu().numpy()) for pl in pls)
        deep = rc["depth"] > ccap
        print("chain_cap", ccap, "group", group, "deeper plans:", int(deep.sum()), "of", Q)
        assert np.array_equal(rc[~deep].view(np.uint8), rn[~deep].view(np.uint8))
        if ccap == 8:
            assert deep.mean() > 0.5 and (~deep & (rc["status"] == ST_OK)).any()
            assert (rn["status"][deep] == ST_OK).all() and (rc["status"][deep] == ST_OVERFLOW).all()
            fixed = rc[deep].copy()
            fixed["status"] = ST_OK
            assert np.array_equal(fixed.view(np.uint8), rn[deep].view(np.uint8))
        else:
            assert not deep.any()


def test_bad_arguments_write_nothing(api, adev, cat, bench_queries):
    """through the raw ABI: a path buffer without a chain buffer, and a workspace one byte short, are AUVRRT_ERR_ARG,
    launch nothing and leave every output untouched"""
    import auvrrt
    env, _ = cat
    lib = auvrrt._lib.lib()
    Q = 64
    starts, seeds = bench_queries(0, Q)
    for group in (0, 32, 1):
        pp = api.plan_params(64, group=group, path_cap=0 if group == 1 else 32)
        pl = adev.DevicePlanner(env, pp, "f32", Q, want_chain=True, want_path=group != 1)
        pl.set_queries(starts, seeds)
        for t in (pl.records, pl.chain, pl.path):
            _fill(t)
        torch.cuda.synchronize()
        vp = adev._vp
        calls = {"too small": (pl.workspace.numel() - 1, pl.chain)}
        if pl.path is not None:
            calls["path without chain"] = (pl.workspace.numel(), None)
        for what, (wsb, chain) in calls.items():
            l0 = api.launch_count()
            rc = lib.auvrrt_plan_batch_dev(env.handle, vp(pl.starts), vp(pl.seeds), Q, C.byref(pp), 0, vp(pl.workspace), wsb,
                                           vp(pl.records), vp(chain), vp(pl.path), None, adev._stream_ptr())
            torch.cuda.synchronize()
            assert rc == ERR_ARG and api.launch_count() == l0, (group, what, rc)
            _assert_sentinel_tail(_dev_out(pl, Q), 0, (group, what))
        pl.launch()                      # the same call with good arguments runs
        torch.cuda.synchronize()
        assert (_records(pl.records.cpu().numpy())["n_nodes"] > 1).any()


# ------------------------------------------------------------------------------------ (B) auvrrt_materialize
def _mode_params(api, mode, group, I=512, **kw):
    if mode == 3:
        return api.plan_params(I, mode=3, v=1.0, max_traj_time=200.0, dubins_rho=1.0, dubins_eta=20.0, near_radius=15.0,
                               dubins_w=12, chain_cap=255, group=group, **kw)
    return api.plan_params(I, mode=mode, max_traj_time=200.0, chain_cap=96, group=group, **kw)


def _assert_paths_equal(path, n_path, want_path, want_n, cap, tag):
    assert np.array_equal(n_path, want_n), tag
    m = _path_mask(want_n, cap)
    assert np.array_equal(path[m], want_path[m]), tag


CASES = [(0, 32), (1, 32), (2, 32), (3, 32), (0, 16), (0, 8)]


@pytest.mark.parametrize("world", ["catalina", "coast", "offset"])
@pytest.mark.parametrize("prec", ["f32", "f64"])
@pytest.mark.parametrize("mode,group", CASES, ids=["mode%d-g%d" % c for c in CASES])
def test_materialize_equals_in_kernel_path(api, worlds, world, prec, mode, group):
    """materialize(chain, depth) is the path the planner wrote, bit for bit: n_path and every row"""
    env, _ = worlds(world)
    Q = 64
    starts = ew.free_starts(world, Q, 100 + mode)
    seeds = np.arange(Q) + 4000 + 100 * mode + group
    pp = _mode_params(api, mode, group, path_cap=2048)
    r = api.plan_batch(env, starts, seeds, pp, prec)
    rec = r["records"]
    ok = rec["status"] == ST_OK
    print(world, prec, mode, group, "status OK:", int(ok.sum()), "of", Q)
    assert ok.mean() >= 0.75
    path, n_path = api.materialize(env, starts[ok], seeds[ok], r["chain"][ok], rec["depth"][ok], pp, prec)
    if mode == 3 and prec == "f32":
        # the in-kernel writer starts every Dubins edge from the tree's node row, which the planner's own evaluation of
        # the edge (collision and cost tests inlined) produced; materialize carries the end state of its re-created
        # edge.  In fp32 the two compilations of the sampler differ in the last bits (measured on a B200), so the
        # rows agree to the fp32 build's tolerance and the waypoint counts exactly
        assert np.array_equal(n_path, rec["n_path"][ok])
        m = _path_mask(n_path, pp.path_cap)
        assert np.allclose(path[m], r["path"][ok][m], rtol=1e-5, atol=1e-3), np.abs(path[m] - r["path"][ok][m]).max()
        return
    _assert_paths_equal(path, n_path, r["path"][ok], rec["n_path"][ok], pp.path_cap, (world, prec, mode, group))


def test_materialize_thread_per_tree_chains_f64(api, cat):
    """fp64, reference-pinned in both planners: thread-per-tree chains (group 1) re-create the warp planner's in-kernel
    paths of the same queries bit for bit, and the records agree"""
    env, _ = cat
    Q = 256
    starts = ew.free_starts("catalina", Q, 11)
    seeds = np.arange(Q) + 777
    t = api.plan_batch(env, starts, seeds, api.plan_params(512, max_traj_time=200.0, group=1), "f64")
    w = api.plan_batch(env, starts, seeds, api.plan_params(512, max_traj_time=200.0, group=32, path_cap=2048), "f64")
    rt, rw = t["records"], w["records"]
    for k in ("status", "n_nodes", "depth", "best_iter"):
        assert np.array_equal(rt[k], rw[k]), k
    assert np.allclose(rt["cost"], rw["cost"], rtol=1e-12, atol=0)
    assert np.array_equal(t["chain"], w["chain"])
    ok = rt["status"] == ST_OK
    assert ok.mean() >= 0.75
    pp = api.plan_params(512, max_traj_time=200.0, group=1, path_cap=2048)
    path, n_path = api.materialize(env, starts[ok], seeds[ok], t["chain"][ok], rt["depth"][ok], pp, "f64")
    _assert_paths_equal(path, n_path, w["path"][ok], rw["n_path"][ok], 2048, "tpt f64")


def test_materialize_thread_per_tree_chains_f32(api, cat, bench_queries):
    """config 5's case: 40,000 queries with group 0 (the thread-per-tree kernel runs), 512 iterations.  Every path
    re-created with group 1 ends exactly at its record's leaf and runs forward in time; it is safe under the collide
    kernel and has the record's cost up to the fp32 build's flips.  Measured on a B200: all 39,796 leaves exact, 22
    paths unsafe under k_collide's fp32 test and 2 with the cost off by more than 2e-4 -- points at obstacle and cell
    boundaries where two fp32 evaluations disagree.  Re-created with the warp evaluator instead (what group 0 / 1 did
    before), 1,341 leaves were exact and 41 paths failed a check."""
    env, ow = cat
    Q = 40_000
    starts, seeds = bench_queries(0, Q)
    r = api.plan_batch(env, starts, seeds, api.plan_params(512), "f32")
    rec = r["records"]
    ok = np.flatnonzero(rec["status"] == ST_OK)
    assert len(ok) > Q // 4
    failed = {"leaf": 0, "time": 0, "safe": 0, "cost": 0}
    paths = []
    for d in np.unique(rec["depth"][ok]):
        ids = ok[rec["depth"][ok] == d]
        pp = api.plan_params(512, group=1, path_cap=34 * (int(d) + 1))
        rows, n_path = api.materialize(env, starts[ids], seeds[ids], r["chain"][ids], rec["depth"][ids], pp, "f32")
        assert (n_path <= pp.path_cap).all()
        for j, q in enumerate(ids):
            p = rows[j, :n_path[j]]
            paths.append((q, p))
            if not (p[-1, 4] == rec["t_leaf"][q] and p[-1, 5] == rec["path_length"][q]):
                failed["leaf"] += 1
            if not np.all(np.diff(p[:, 4]) >= 0):
                failed["time"] += 1
            want = orc.cost(p[::-1][:, [0, 1, 4]], p[-1, 4], ow, [-3, -3, -4])
            if not np.all(np.abs(rec["cost"][q] - want) <= 2e-4 * np.maximum(np.abs(want), 1.0)):
                failed["cost"] += 1
    safe = api.collide(env, [p[:, :2] for _, p in paths], "f32")
    failed["safe"] = int((safe != 1).sum())
    print("thread-per-tree fp32 paths checked:", len(paths), "of", Q, "queries; failures by check:", failed)
    assert failed["leaf"] == 0 and failed["time"] == 0, failed
    assert failed["safe"] <= 1e-3 * len(paths) and failed["cost"] <= 1e-3 * len(paths), failed


def test_materialize_rejects_overflowed_chains(api, cat):
    """a chain_cap = 8 plan: its OVERFLOW records (depth > 8) and a negative depth are AUVRRT_ERR_ARG; the other
    records of the same batch still re-create their in-kernel paths"""
    import auvrrt
    env, _ = cat
    Q = 128
    starts = ew.free_starts("catalina", Q, 5)
    seeds = np.arange(Q) + 50
    pp = api.plan_params(1024, max_traj_time=200.0, chain_cap=8, path_cap=512)
    r = api.plan_batch(env, starts, seeds, pp, "f32")
    rec = r["records"]
    over, ok = rec["status"] == ST_OVERFLOW, rec["status"] == ST_OK
    assert over.any() and ok.any() and (rec["depth"][over] > 8).all() and (rec["n_path"][over] == 0).all()
    for sel in (over, np.ones(Q, bool)):
        with pytest.raises(auvrrt._lib.AuvrrtError, match="chain_cap"):
            api.materialize(env, starts[sel], seeds[sel], r["chain"][sel], rec["depth"][sel], pp, "f32")
    neg = rec["depth"][ok].copy()
    neg[0] = -1
    with pytest.raises(auvrrt._lib.AuvrrtError):
        api.materialize(env, starts[ok], seeds[ok], r["chain"][ok], neg, pp, "f32")
    path, n_path = api.materialize(env, starts[ok], seeds[ok], r["chain"][ok], rec["depth"][ok], pp, "f32")
    _assert_paths_equal(path, n_path, r["path"][ok], rec["n_path"][ok], pp.path_cap, "chain_cap 8")


@pytest.mark.parametrize("prec", ["f32", "f64"])
def test_materialize_short_path_buffer(api, cat, prec):
    """path_cap below the path: the full n_path comes back and the rows written are the full path's prefix -- what the
    in-kernel writer reports as OVERFLOW for the same cap"""
    env, _ = cat
    Q = 32
    starts = ew.free_starts("catalina", Q, 9)
    seeds = np.arange(Q) + 90
    pp = api.plan_params(1024, path_cap=2048)
    full = api.plan_batch(env, starts, seeds, pp, prec)
    rec = full["records"]
    ok = rec["status"] == ST_OK
    assert ok.all()
    cap = int(np.min(rec["n_path"])) // 2
    short = api.plan_params(1024, path_cap=cap)
    path, n_path = api.materialize(env, starts, seeds, full["chain"], rec["depth"], short, prec)
    assert np.array_equal(n_path, rec["n_path"])
    assert np.array_equal(path, full["path"][:, :cap])
    k = api.plan_batch(env, starts, seeds, short, prec)
    assert (k["records"]["status"] == ST_OVERFLOW).all() and np.array_equal(k["records"]["n_path"], rec["n_path"])
    assert np.array_equal(k["path"], path)


@pytest.mark.parametrize("prec", ["f32", "f64"])
def test_materialize_no_path_record_is_its_start(api, cat, prec):
    """a NO_PATH record has depth 0: it materialises to the start row alone"""
    env, _ = cat
    Q = 16
    starts = ew.free_starts("catalina", Q, 13)
    starts[:, 2] = np.linspace(-3, 3, Q)
    starts[:, 3] = np.linspace(0, 40, Q)
    starts[:, 4] = np.linspace(0, 80, Q)
    pp = api.plan_params(4, path_cap=64)
    r = api.plan_batch(env, starts, np.arange(Q), pp, prec)
    rec = r["records"]
    assert (rec["status"] == ST_NO_PATH).all() and (rec["depth"] == 0).all()
    path, n_path = api.materialize(env, starts, np.arange(Q), r["chain"], rec["depth"], pp, prec)
    assert (n_path == 1).all()
    dt = np.float32 if prec == "f32" else np.float64
    want = np.column_stack([starts[:, :3], np.zeros(Q), starts[:, 3:5]]).astype(dt).astype(np.float64)
    assert np.array_equal(path[:, 0], want)
    assert not path[:, 1:].any()


# ------------------------------------------------------------------------------------ (C) edge and nearest-node _dev
SP5 = [2.0, 0.5, 30.0, 0.5, 2.0]


def _edge_inputs(n, seed, origin=(0.0, 0.0)):
    rs = np.random.RandomState(seed)
    par = np.stack([rs.uniform(-300, -100, n) + origin[0], rs.uniform(-60, 100, n) + origin[1], rs.uniform(-6, 6, n),
                    rs.uniform(0, 520, n), rs.uniform(0, 500, n)], 1)
    ang, dist = rs.uniform(-np.pi, np.pi, n), rs.uniform(2, 40, n)
    q0 = par[:, :3].copy()
    q1 = np.stack([q0[:, 0] + dist * np.cos(ang), q0[:, 1] + dist * np.sin(ang), rs.uniform(-np.pi, np.pi, n)], 1)
    return par, np.arange(n, dtype=np.uint64) * 3 + 11, q0, q1


def _check_edges(api, adev, env, n, prec, seed):
    dt = torch.float32 if prec == "f32" else torch.float64
    npdt = np.float32 if prec == "f32" else np.float64
    dev = torch.device("cuda", env.device)
    par, seeds, q0, q1 = _edge_inputs(n, seed)
    par, q0, q1 = (a.astype(npdt).astype(np.float64) for a in (par, q0, q1))
    P, S = torch.from_numpy(par).to(dev, dt), torch.from_numpy(seeds.view(np.int64)).to(dev)
    A, B = torch.from_numpy(q0).to(dev, dt), torch.from_numpy(q1).to(dev, dt)

    def z(*shape, dtype=dt):
        return torch.full(shape, 7, dtype=dtype, device=dev)
    side = torch.cuda.Stream(device=dev)
    u8, i32 = torch.uint8, torch.int32
    with torch.cuda.stream(side):
        arc = (z(n, dtype=u8), z(n, dtype=i32), z(n, 5))
        adev.edges_arc_dev(env, P, S, SP5, *arc, prec, stream=side)
        arc_nl = (z(n, dtype=u8), z(n, dtype=i32))
        adev.edges_arc_dev(env, P, S, SP5, *arc_nl, None, prec, stream=side)
        arcc = (z(n, dtype=u8), z(n, dtype=i32), z(n, 5), z(n, 3))
        adev.edges_arc_cost_dev(env, P, S, SP5, -4.0, *arcc, prec, stream=side)
        arcc_nl = (z(n, dtype=u8), z(n, dtype=i32), z(n, 3))
        adev.edges_arc_cost_dev(env, P, S, SP5, -4.0, arcc_nl[0], arcc_nl[1], None, arcc_nl[2], prec, stream=side)
        dub = (z(n, dtype=u8), z(n, dtype=u8), z(n))
        adev.edges_dubins_dev(env, A, B, 1.0, 20, *dub, prec, stream=side)
        dubc = (z(n, dtype=u8), z(n, dtype=u8), z(n), z(n, 3))
        adev.edges_dubins_cost_dev(env, A, B, 1.0, 20, 1.0, -4.0, *dubc, prec, stream=side)
    side.synchronize()

    def np_(ts):
        return [t.cpu().numpy().astype(np.float64) if t.is_floating_point() else t.cpu().numpy() for t in ts]
    for got, want in ((arc, api.edges_arc(env, par, seeds, SP5, prec)),
                      (arcc, api.edges_arc_cost(env, par, seeds, SP5, -4.0, prec)),
                      (dub, api.edges_dubins(env, q0, q1, 1.0, 20, prec)),
                      (dubc, api.edges_dubins_cost(env, q0, q1, 1.0, 20, 1.0, -4.0, prec))):
        for g, w in zip(np_(got), want):
            assert np.array_equal(g, w), (n, prec)
    # without a leaf buffer (bench config 4): the same booleans, counts and costs
    assert all(np.array_equal(a, b) for a, b in zip(np_(arc_nl), np_(arc[:2])))
    assert all(np.array_equal(a, b) for a, b in zip(np_(arcc_nl), np_((arcc[0], arcc[1], arcc[3]))))
    s = np_(arcc)[0]
    assert (s == 1).any() and (s == 0).any()


@pytest.mark.parametrize("world", ["catalina", "huge"])
@pytest.mark.parametrize("prec", ["f32", "f64"])
def test_edges_dev_equal_host_entries(api, adev, worlds, world, prec):
    """edges_arc(_cost)_dev and edges_dubins(_cost)_dev on a side stream equal the host entries bit for bit; on huge the
    launchers take the warp-per-edge fallback"""
    env, _ = worlds(world)
    _check_edges(api, adev, env, 20_000, prec, 3 if world == "catalina" else 4)


def test_edges_dev_batch_loop_f32(api, adev, worlds):
    """3.2M fp32 edges: the thread-per-edge kernel's 1024-thread shape and batch loop, through the _dev entries"""
    env, _ = worlds("catalina")
    _check_edges(api, adev, env, 3_200_000, "f32", 5)


@pytest.mark.parametrize("prec", ["f32", "f64"])
def test_nn_dev_equals_host_entry(api, adev, prec):
    """nn_dev on a side stream equals auvrrt_nn; a tree that is not 16-byte aligned is AUVRRT_ERR_ARG"""
    import auvrrt
    dt = torch.float32 if prec == "f32" else torch.float64
    dev = torch.device("cuda", 0)
    rs = np.random.RandomState(17)
    n, nq = 100_003, 37
    tree = rs.uniform(-500, 500, (n, 2)).astype(np.float32).astype(np.float64)
    qs = rs.uniform(-500, 500, (nq, 2)).astype(np.float32).astype(np.float64)
    tx, ty = (torch.from_numpy(np.ascontiguousarray(tree[:, i])).to(dev, dt) for i in (0, 1))
    qx, qy = (torch.from_numpy(np.ascontiguousarray(qs[:, i])).to(dev, dt) for i in (0, 1))
    idx = torch.full((nq,), -7, dtype=torch.int32, device=dev)
    scr = adev.nn_scratch(nq, dev)
    side = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(side):
        adev.nn_dev(tx, ty, qx, qy, idx, scr, prec, stream=side)
    side.synchronize()
    assert np.array_equal(idx.cpu().numpy(), api.nn(tree, qs, prec))
    with pytest.raises(auvrrt._lib.AuvrrtError, match="aligned"):
        adev.nn_dev(tx[1:], ty[1:], qx, qy, idx, scr, prec)
