"""GPU: the device end of a planning step -- each mission's best plan (auvrrt_plan_best_dev) and its path
(auvrrt_materialize_dev), and DevicePlanner.best_paths on top of them.

1. The selection equals a numpy reference on synthetic records: ragged, empty and all-failed missions, planted exact
   ties, -0.0 / +0.0, NaN and +inf costs, OVERFLOW and negative depths, offsets out of range; one mission of 2^20
   records (the split kernel) and 4096 missions of about 256 (a warp per mission).
2. materialize_dev equals the host entry api.materialize bit for bit, in every mode, precision and group, on the
   catalina / coast / offset worlds, through a pick list with -1, repeats and out-of-range picks, a short path_cap,
   and records whose depth cannot be re-created.
3. DevicePlanner.best_paths equals the host pipeline (records -> numpy argmin per mission -> api.materialize) with
   group 0 on both sides of 32768 queries, so both planners run; on the caller's stream.
4. refresh -> plan -> best -> path captured in one CUDA graph equals the eager sequence bit for bit, for two track sets.
"""
import os

import numpy as np
import pytest
import torch

import envelope_worlds as ew

pytestmark = pytest.mark.gpu

ST_OK, ST_NO_PATH, ST_OVERFLOW = 0, 1, 5


@pytest.fixture(scope="module")
def mods():
    import auvrrt
    from auvrrt import api
    from auvrrt import device as adev
    assert api.device_count() > 0 and torch.cuda.is_available()
    return api, adev


@pytest.fixture(scope="module")
def worlds(mods):
    api, _ = mods
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = api.Env(**ew.assert_flags(name))
        return cache[name]
    yield get
    for e in cache.values():
        e.close()


# ------------------------------------------------------------------------------------ references
def ref_best(rec, off):
    """numpy: per mission the first minimum of cost[0] over status OK, depth >= 0, cost not NaN (-0.0 == +0.0)"""
    Q = len(rec)
    c = rec["cost"][:, 0]
    elig = (rec["status"] == ST_OK) & (rec["depth"] >= 0) & ~np.isnan(c)
    cz = np.where(c == 0, 0.0, c)
    M = len(off) - 1
    best = np.full(M, -1, np.int64)
    cost = np.full(M, np.inf)
    for m in range(M):
        lo = min(max(int(off[m]), 0), Q)
        hi = min(max(int(off[m + 1]), lo), Q)
        idx = lo + np.flatnonzero(elig[lo:hi])
        if len(idx):
            j = idx[int(np.argmin(cz[idx]))]
            best[m], cost[m] = j, c[j]
    return best, cost


def synthetic_records(Q, rs):
    from auvrrt.api import RECORD_DTYPE
    rec = np.zeros(Q, RECORD_DTYPE)
    rec["status"] = np.where(rs.random_sample(Q) < 0.8, ST_OK, rs.choice([ST_NO_PATH, 2, 3, 4, ST_OVERFLOW], Q))
    rec["depth"] = rs.randint(0, 60, Q)
    over = rec["status"] == ST_OVERFLOW
    rec["depth"][over] = rs.randint(97, 300, over.sum())
    rec["depth"][rs.random_sample(Q) < 0.01] = -1                      # negative depths, status OK or not
    rec["depth"][rs.random_sample(Q) < 0.005] = -(1 << 30)
    # few distinct values so that exact ties are everywhere
    c = -np.round(rs.random_sample(Q) * 40.0, 1)
    r = rs.random_sample(Q)
    c[r < 0.02] = 0.0
    c[(r >= 0.02) & (r < 0.04)] = -0.0
    c[(r >= 0.04) & (r < 0.05)] = np.nan
    c[(r >= 0.05) & (r < 0.06)] = np.inf
    c[(r >= 0.06) & (r < 0.062)] = -np.inf
    rec["cost"][:, 0] = c
    rec["cost"][:, 1:] = rs.random_sample((Q, 3))
    rec["n_nodes"] = rs.randint(1, 1000, Q)
    return rec


def _dev_records(rec):
    return torch.from_numpy(np.ascontiguousarray(rec).view(np.uint8).reshape(len(rec), -1).copy()).cuda()


def _check_best(adev, rec, off, stream=None):
    d = _dev_records(rec)
    doff = torch.from_numpy(np.asarray(off, np.int64)).cuda()
    best, cost = adev.plan_best_dev(d, doff, stream=stream)
    torch.cuda.synchronize()
    wb, wc = ref_best(rec, off)
    gb, gc = best.cpu().numpy(), cost.cpu().numpy()
    assert np.array_equal(gb, wb), np.flatnonzero(gb != wb)[:10]
    assert np.array_equal(gc.view(np.int64), wc.view(np.int64))            # bit for bit: -0.0 stays -0.0
    return wb


# ------------------------------------------------------------------------------------ 1. selection
def test_select_one_mission_of_2_20_records(mods):
    _, adev = mods
    rs = np.random.RandomState(1)
    Q = 1 << 20
    rec = synthetic_records(Q, rs)
    assert _check_best(adev, rec, [0, Q])[0] >= 0
    # the minimum planted three times, in different CTAs' slices: the lowest index wins
    rec["cost"][np.isneginf(rec["cost"][:, 0]), 0] = 0.0
    far = [5, 700_000, 1_000_000]
    rec["status"][far], rec["depth"][far] = ST_OK, 3
    rec["cost"][far, 0] = -1000.0
    assert _check_best(adev, rec, [0, Q])[0] == 5
    rec["status"][5] = ST_NO_PATH
    assert _check_best(adev, rec, [0, Q])[0] == 700_000
    # -0.0 == +0.0: the first zero wins and its own sign comes back
    rec["status"][:], rec["depth"][:] = ST_OK, 1
    rec["cost"][:, 0] = 1.0
    rec["cost"][[1000, 2000], 0] = [-0.0, 0.0]
    assert _check_best(adev, rec, [0, Q])[0] == 1000
    rec["cost"][[1000, 2000], 0] = [0.0, -0.0]
    assert _check_best(adev, rec, [0, Q])[0] == 1000
    rec["cost"][500_000, 0] = -np.inf
    assert _check_best(adev, rec, [0, Q])[0] == 500_000
    # nothing eligible: all failed, all NaN; +inf alone is a plan
    rec["status"][:] = ST_NO_PATH
    assert _check_best(adev, rec, [0, Q])[0] == -1
    rec["status"][:] = ST_OK
    rec["cost"][:, 0] = np.nan
    assert _check_best(adev, rec, [0, Q])[0] == -1
    rec["cost"][123_456, 0] = np.inf
    assert _check_best(adev, rec, [0, Q])[0] == 123_456


def test_select_many_ragged_missions(mods):
    _, adev = mods
    rs = np.random.RandomState(2)
    M = 4096
    sizes = rs.randint(0, 513, M)
    sizes[rs.random_sample(M) < 0.05] = 0                                   # empty missions
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    Q = int(off[-1])
    rec = synthetic_records(Q, rs)
    for m in rs.choice(M, 200, replace=False):                              # all-failed missions
        rec["status"][off[m]:off[m + 1]] = ST_NO_PATH
    wb = _check_best(adev, rec, off)
    assert (wb == -1).sum() > 200 and (wb >= 0).sum() > 3000
    # 4096 x 256 exactly, and 4096 x 64
    for R in (256, 64):
        r2 = synthetic_records(M * R, rs)
        _check_best(adev, r2, np.arange(M + 1, dtype=np.int64) * R)


def test_select_clamps_bad_offsets(mods):
    _, adev = mods
    rs = np.random.RandomState(3)
    Q = 5000
    rec = synthetic_records(Q, rs)
    off = np.array([-50, 10, 4000, 300, 300, 4999, 1 << 40, -(1 << 40), 20, 6000, Q], np.int64)
    _check_best(adev, rec, off)
    _check_best(adev, rec, [0, 0])
    # a large Q with few, uneven missions takes the split kernel
    big = synthetic_records(1 << 18, rs)
    _check_best(adev, big, [0, 7, 100_000, 100_000, 200_000 + 13, 1 << 18])
    _check_best(adev, big, [-9, 1 << 19])


# ------------------------------------------------------------------------------------ 2. materialize_dev
def _mode_params(api, mode, group, I=512, **kw):
    if mode == 3:
        return api.plan_params(I, mode=3, v=1.0, max_traj_time=200.0, dubins_rho=1.0, dubins_eta=20.0, near_radius=15.0,
                               dubins_w=12, chain_cap=255, group=group, **kw)
    return api.plan_params(I, mode=mode, max_traj_time=200.0, chain_cap=96, group=group, **kw)


def _plan_dev(api, adev, env, starts, seeds, pp, prec):
    pl = adev.DevicePlanner(env, pp, prec, len(seeds), want_chain=True)
    pl.set_queries(starts, seeds)
    pl.launch()
    torch.cuda.synchronize()
    return pl


def _host_rows(api, env, starts, seeds, chain, rec, pick, pp, prec, cap):
    """api.materialize of the picked plans, one row per pick; (-1: n 0, invalid: n -1) as materialize_dev reports"""
    import copy
    M = len(pick)
    rows = np.zeros((M, cap, 6))
    n = np.zeros(M, np.int32)
    Q = len(seeds)
    ok = np.array([0 <= p < Q and 0 <= rec["depth"][p] <= pp.chain_cap for p in pick], bool)
    n[~ok] = [0 if p == -1 else -1 for p in np.asarray(pick)[~ok]]
    if ok.any():
        sel = np.asarray(pick)[ok]
        hp = copy.copy(pp)
        hp.path_cap = cap
        r, k = api.materialize(env, starts[sel], seeds[sel], chain[sel], rec["depth"][sel], hp, prec)
        rows[ok], n[ok] = r, k
    return rows, n, ok


MAT_CASES = [(0, 32), (1, 32), (2, 32), (3, 32), (0, 16), (0, 8), (0, 1), (1, 1), (2, 1)]


@pytest.mark.parametrize("world", ["catalina", "coast", "offset"])
@pytest.mark.parametrize("prec", ["f32", "f64"])
@pytest.mark.parametrize("mode,group", MAT_CASES, ids=["mode%d-g%d" % c for c in MAT_CASES])
def test_materialize_dev_equals_host_entry(mods, worlds, world, prec, mode, group):
    api, adev = mods
    from auvrrt.api import RECORD_DTYPE
    env = worlds(world)
    Q = 64
    starts = ew.free_starts(world, Q, 200 + mode)
    seeds = np.arange(Q) + 9000 + 100 * mode + group
    pp = _mode_params(api, mode, group)
    pl = _plan_dev(api, adev, env, starts, seeds, pp, prec)
    rec = pl.records.cpu().numpy().view(RECORD_DTYPE).reshape(-1)
    chain = pl.chain.cpu().numpy().view(np.uint32)
    ok = np.flatnonzero(rec["status"] == ST_OK)
    assert len(ok) >= Q // 2
    pick = np.concatenate([ok, ok[:5], [-1, Q, 1 << 40, -2, -1], ok[::-1][:7]]).astype(np.int64)
    rdt = torch.float32 if prec == "f32" else torch.float64
    for cap in (2048, 7):
        out = torch.full((len(pick), cap, 6), float("nan"), dtype=rdt, device="cuda")
        out_n = torch.full((len(pick),), -99, dtype=torch.int32, device="cuda")
        adev.materialize_dev(env, pl.starts, pl.seeds, pl.records, pl.chain, torch.from_numpy(pick).cuda(), pp, prec, cap,
                             out=out, out_n=out_n)
        torch.cuda.synchronize()
        got, gn = out.cpu().numpy().astype(np.float64), out_n.cpu().numpy()
        want, wn, _ = _host_rows(api, env, starts, seeds, chain, rec, pick, pp, prec, cap)
        assert np.array_equal(gn, wn), (cap, gn, wn)
        written = np.arange(cap)[None, :] < np.clip(wn, 0, cap)[:, None]
        assert np.array_equal(got[written], want[written]), cap
        assert np.isnan(got[~written]).all(), "rows past n_path (or of a -1 / 0 row) were written"
        assert (wn > cap).any() == (cap == 7)                               # the short cap cuts paths


@pytest.mark.parametrize("prec", ["f32", "f64"])
def test_materialize_dev_invalid_depths(mods, worlds, prec):
    """OVERFLOW records of a chain_cap = 8 plan, and records whose depth was made negative or too deep: n_path -1, no row,
    and the neighbouring rows are the host entry's"""
    api, adev = mods
    from auvrrt.api import RECORD_DTYPE
    env = worlds("catalina")
    Q = 128
    starts = ew.free_starts("catalina", Q, 5)
    seeds = np.arange(Q) + 50
    pp = api.plan_params(1024, max_traj_time=200.0, chain_cap=8, group=32)
    pl = _plan_dev(api, adev, env, starts, seeds, pp, prec)
    rec = pl.records.cpu().numpy().view(RECORD_DTYPE).reshape(-1).copy()
    over, ok = np.flatnonzero(rec["status"] == ST_OVERFLOW), np.flatnonzero(rec["status"] == ST_OK)
    assert len(over) and len(ok) > 4
    rec["depth"][ok[1]] = -1
    rec["depth"][ok[3]] = 9
    d = _dev_records(rec)
    pick = np.array([ok[0], ok[1], ok[2], over[0], ok[3], ok[4]], np.int64)
    out, out_n = adev.materialize_dev(env, pl.starts, pl.seeds, d, pl.chain, torch.from_numpy(pick).cuda(), pp, prec, 512)
    torch.cuda.synchronize()
    gn = out_n.cpu().numpy()
    assert list(gn[[1, 3, 4]]) == [-1, -1, -1]
    chain = pl.chain.cpu().numpy().view(np.uint32)
    want, wn, _ = _host_rows(api, env, starts, seeds, chain, rec, pick, pp, prec, 512)
    assert np.array_equal(gn, wn)
    got = out.cpu().numpy()
    for j in (0, 2, 5):
        assert np.array_equal(got[j, :wn[j]].astype(np.float64), want[j, :wn[j]])


def test_materialize_dev_rejections(mods, worlds):
    api, adev = mods
    env = worlds("catalina")
    Q = 8
    pp = api.plan_params(64, group=32)
    pl = _plan_dev(api, adev, env, ew.free_starts("catalina", Q, 1), np.arange(Q), pp, "f32")
    pick = torch.zeros(2, dtype=torch.int64, device="cuda")
    out = torch.full((2, 16, 6), 7.0, device="cuda")
    for g in (0, 4):
        bad = api.plan_params(64, group=g)
        with pytest.raises(api._lib.AuvrrtError, match="group"):
            adev.materialize_dev(env, pl.starts, pl.seeds, pl.records, pl.chain, pick, bad, "f32", 16, out=out)
    m3 = api.plan_params(64, mode=3, group=1)
    with pytest.raises(api._lib.AuvrrtError, match="mode 3"):
        adev.materialize_dev(env, pl.starts, pl.seeds, pl.records, pl.chain, pick, m3, "f32", 16, out=out)
    with pytest.raises(ValueError):
        adev.materialize_dev(env, pl.starts.double(), pl.seeds, pl.records, pl.chain, pick, pp, "f32", 16)
    with pytest.raises(ValueError):
        adev.materialize_dev(env, pl.starts, pl.seeds, pl.records, pl.chain, pick.int(), pp, "f32", 16)
    with pytest.raises(ValueError):
        adev.plan_best_dev(pl.records, torch.zeros(3, dtype=torch.int32, device="cuda"))
    torch.cuda.synchronize()
    assert (out == 7.0).all()


# ------------------------------------------------------------------------------------ 3. DevicePlanner.best_paths
def _host_pipeline(api, env, starts, seeds, pl, off, path_cap, prec):
    from auvrrt.api import RECORD_DTYPE
    rec = pl.records[:pl.n].cpu().numpy().view(RECORD_DTYPE).reshape(-1)
    chain = pl.chain[:pl.n].cpu().numpy().view(np.uint32)
    best, cost = ref_best(rec, off)
    import copy
    pp = copy.copy(pl.params)
    pp.group = api.plan_group(pl.params, pl.n, pl.path is not None)
    rows, n, _ = _host_rows(api, env, starts, seeds, chain, rec, best, pp, prec, path_cap)
    return best, cost, rows, n


@pytest.mark.parametrize("Q,R", [(4096, 64), (40960, 64)], ids=["warp", "thread-per-tree"])
def test_best_paths_equal_host_pipeline(mods, worlds, Q, R):
    api, adev = mods
    import bench
    env = worlds("catalina")
    starts, seeds = bench.make_queries(0, Q)
    pp = api.plan_params(256 if Q > 32768 else 1024, chain_cap=96)
    pl = adev.DevicePlanner(env, pp, "f32", Q, want_chain=True)
    pl.set_queries(starts, seeds)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    off = np.arange(Q // R + 1, dtype=np.int64) * R
    with torch.cuda.stream(s):
        doff = torch.from_numpy(off).cuda()
        pl.launch(s)
        r = pl.best_paths(doff, 1024, stream=s)
    s.synchronize()
    assert pl.group == (1 if Q >= 32768 else 32)
    best, cost, rows, n = _host_pipeline(api, env, starts, seeds, pl, off, 1024, "f32")
    assert np.array_equal(r["best"].cpu().numpy(), best)
    assert np.array_equal(r["cost"].cpu().numpy().view(np.int64), cost.view(np.int64))
    gn = r["n_path"].cpu().numpy()
    assert np.array_equal(gn, n) and (gn > 0).mean() > 0.5
    got = r["path"].cpu().numpy().astype(np.float64)
    m = np.arange(1024)[None, :] < np.clip(n, 0, 1024)[:, None]
    assert np.array_equal(got[m], rows[m])


# ------------------------------------------------------------------------------------ 4. one CUDA graph
def test_refresh_plan_best_path_in_one_graph(mods, catalina_map, golden_dir):
    api, adev = mods
    z = np.load(os.path.join(golden_dir, "occupancy.npz"))
    polys = [z["cell_xy"][z["cell_off"][i]:z["cell_off"][i + 1]] for i in range(len(z["cell_off"]) - 1)]
    bounds = np.asarray(z["bounds"], np.float64)
    T, S, P = 9, 32, 815
    bins = np.array([[b * 50.0, (b + 1) * 50.0] for b in range(T)])
    rs = np.random.RandomState(21)

    def tracks():
        return np.concatenate([np.stack([rs.uniform(-330, -80) + np.cumsum(rs.normal(0, 0.6, P)),
                                         rs.uniform(-60, 90) + np.cumsum(rs.normal(0, 0.6, P)),
                                         0.03 * 20 * np.arange(P)], 1) for _ in range(S)])
    sets = [torch.from_numpy(tracks()).cuda() for _ in range(2)]
    toff = torch.from_numpy(np.arange(S + 1, dtype=np.int64) * P).cuda()
    occ = adev.SharkOccupancy(polys, bounds, 10.0, 50.0, 50.0, T, S, S * P)
    env = api.Env.from_map(catalina_map, bins, None)
    Q, R = 512, 64
    starts = ew.free_starts("catalina", Q, 31)
    pp = api.plan_params(512, max_traj_time=200.0, chain_cap=96)
    pl = adev.DevicePlanner(env, pp, "f32", Q, want_chain=True)
    pl.set_queries(starts, np.arange(Q) + 70)
    trk = torch.empty_like(sets[0])
    doff = torch.from_numpy(np.arange(Q // R + 1, dtype=np.int64) * R).cuda()

    def step():
        occ.grid_dev(trk, toff, env=env)
        pl.launch()
        return pl.best_paths(doff, 512)

    def snap(r):
        return {k: v.cpu().numpy().copy() for k, v in r.items()}

    eager = []
    for t in sets:
        trk.copy_(t)
        eager.append(snap(step()))
        torch.cuda.synchronize()
    assert not np.array_equal(eager[0]["cost"], eager[1]["cost"])          # the tracks change the plans
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()                                                               # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = step()
    for t, want in zip(sets, eager):
        trk.copy_(t)
        g.replay()
        torch.cuda.synchronize()
        got = snap(out)
        for k in ("best", "n_path"):
            assert np.array_equal(got[k], want[k]), k
        assert np.array_equal(got["cost"].view(np.int64), want["cost"].view(np.int64))
        m = np.arange(512)[None, :] < np.clip(want["n_path"], 0, 512)[:, None]
        assert np.array_equal(got["path"][m], want["path"][m])
    occ.close()
