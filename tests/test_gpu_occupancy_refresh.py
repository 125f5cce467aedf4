"""Shark-occupancy grids from device-resident tracks, and a live world's probability table refreshed in place
(auvrrt_occ_* / auvrrt_env_set_probs* of include/auvrrt.h; auvrrt.device.SharkOccupancy).

GPU: the grids equal the golden grids and the oracle bit for bit, including for points on lattice lines, cell
corners, shared edges and the boundary's vertices (the candidate-cell index of the histogram); a refreshed world
plans and costs byte-for-byte like a world created from the same table; the refresh captures into a CUDA graph.
CPU: the occupancy kernels spill nothing."""
import os
import re
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from oracle import orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PP = os.path.join(ROOT, "auv-sim_b200", "path_planning")
CSRC = os.path.join(ROOT, "auv-sim_b200", "csrc")
# CATALINA_TRACK_MAP of path_planning/sharkOccupancyGrid.py (config 3's raw tracks in the map's frame)
TRACK_MAP = {"x0": 370.0, "y0": 4.0, "sx": 250.0 / 964.0, "sy": 150.0 / 496.0, "ox": -330.0, "oy": -60.0,
             "frame_dt": 0.03, "time_scale": 20.0}


# ------------------------------------------------------------------ fixtures

@pytest.fixture(scope="module")
def occ_golden(golden_dir):
    z = np.load(os.path.join(golden_dir, "occupancy.npz"))
    polys = [z["cell_xy"][z["cell_off"][i]:z["cell_off"][i + 1]] for i in range(len(z["cell_off"]) - 1)]
    cases = []
    for ci in range(int(z["n_cases"])):
        toff, trk = z["c%d_toff" % ci], z["c%d_trk" % ci]
        cases.append({"tracks": [trk[toff[i]:toff[i + 1]] for i in range(len(toff) - 1)],
                      "params": z["c%d_params" % ci], "grid": z["c%d_grid" % ci]})
    return polys, np.asarray(z["bounds"], np.float64), cases


@pytest.fixture(scope="module")
def raw_tracks(golden_dir):
    """config 3: data/sharkTrackingData.csv (32 sharks x 815 frames) as tracks_to_shark_dict maps it"""
    z = np.load(os.path.join(golden_dir, "shark_tracks_raw.npz"))
    m = TRACK_MAP
    x, y = z["x"].astype(np.float64), z["y"].astype(np.float64)
    t = np.arange(x.shape[1]) * m["frame_dt"] * m["time_scale"]
    return [np.stack([m["ox"] + (x[s] - m["x0"]) * m["sx"], m["oy"] + (y[s] - m["y0"]) * m["sy"], t], 1)
            for s in range(len(x))]


@pytest.fixture(scope="module")
def random_tracks():
    """the 32 x 815 random walks of tests/test_occupancy.py"""
    rs = np.random.RandomState(5)
    return [np.stack([rs.uniform(-330, -80) + np.cumsum(rs.normal(0, 0.6, 815)),
                      rs.uniform(-60, 90) + np.cumsum(rs.normal(0, 0.6, 815)), 0.03 * 30 * np.arange(1, 816)], 1)
            for _ in range(32)]


def _dev_tracks(tracks):
    import torch
    off = np.zeros(len(tracks) + 1, np.int64)
    off[1:] = np.cumsum([len(t) for t in tracks])
    flat = np.concatenate([np.asarray(t, np.float64).reshape(-1, 3) for t in tracks]) if off[-1] else np.zeros((0, 3))
    return torch.from_numpy(np.ascontiguousarray(flat)).cuda(), torch.from_numpy(off).cuda()


def _t_occ(bin_interval, tracks):
    """createBinList's T (auvrrt_occupancy_dims)"""
    longest = 0.0
    for t in tracks:
        if len(t) and t[-1][2] > longest:
            longest = t[-1][2]
    return int(np.floor(longest / bin_interval))


def _cell_table(grid, polys, bounds, cell_size):
    """keep_zero_cells=True's per-bin dicts as a table [T, C]: cell c at cellToIndex of its bounds"""
    rc = [(int((min(p[:, 1]) - bounds[1]) / cell_size), int((min(p[:, 0]) - bounds[0]) / cell_size))
          for p in (np.asarray(q, np.float64).reshape(-1, 2) for q in polys)]
    return np.ascontiguousarray(np.stack([[g[r, c] for r, c in rc] for g in grid]).reshape(len(grid), len(polys)))


def _grid_dev(polys, bounds, cs, bi, rg, tracks, n_bins):
    import torch
    from auvrrt import device as adev
    occ = adev.SharkOccupancy(polys, bounds, cs, bi, rg, n_bins, len(tracks), sum(len(t) for t in tracks))
    trk, off = _dev_tracks(tracks)
    out = torch.full(occ.grid_shape, -1.0, dtype=torch.float64, device="cuda")
    t_occ = torch.full((1,), -7, dtype=torch.int32, device="cuda")
    occ.grid_dev(trk, off, out=out, t_occ=t_occ)
    torch.cuda.synchronize()
    return out.cpu().numpy(), int(t_occ.item()), occ


def _bins(n, bi=50.0):
    return np.array([[b * bi, (b + 1) * bi] for b in range(n)], np.float64).reshape(-1, 2)


# ------------------------------------------------------------------ 1. bit-exact grids

@pytest.mark.gpu
def test_grid_dev_equals_golden_grids(occ_golden):
    from auvrrt import api
    polys, bounds, cases = occ_golden
    for c in cases:
        cs, bi, rg = c["params"]
        got, t_occ, _ = _grid_dev(polys, bounds, cs, bi, rg, c["tracks"], len(c["grid"]))
        assert got.shape == c["grid"].shape and np.array_equal(got, c["grid"])
        _, bins = api.occupancy_grid(polys, bounds, cs, bi, rg, c["tracks"])
        assert t_occ == len(bins) == _t_occ(bi, c["tracks"])


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["random", "config3"])
def test_grid_dev_equals_oracle(occ_golden, random_tracks, raw_tracks, which):
    polys, bounds, _ = occ_golden
    tracks = random_tracks if which == "random" else raw_tracks
    want = orc.occupancy(polys, bounds, 10.0, 50.0, 50.0, tracks)
    got, t_occ, _ = _grid_dev(polys, bounds, 10.0, 50.0, 50.0, tracks, len(want))
    assert t_occ == len(want) == {"random": 14, "config3": 9}[which]
    assert np.array_equal(got, want)
    # more bins than the tracks cover: the covered prefix is unchanged
    got2, t_occ2, _ = _grid_dev(polys, bounds, 10.0, 50.0, 50.0, tracks, len(want) + 2)
    assert t_occ2 == t_occ and np.array_equal(got2[:t_occ], want)


# ------------------------------------------------------------------ 2. the candidate-cell index is exact

def _edge_points(polys, bounds, extra, seed):
    """every vertex of every cell (cell corners, the ends of shared clipped edges, the boundary's vertices), every
    edge midpoint, points on the lattice lines x = minx + 10 i and y = miny + 10 j, the union box's corners and
    points just outside it, plus `extra`"""
    rs = np.random.RandomState(seed)
    v = np.concatenate([np.asarray(p, np.float64).reshape(-1, 2) for p in polys])
    mids = np.concatenate([0.5 * (np.asarray(p, np.float64) + np.roll(np.asarray(p, np.float64), -1, 0)) for p in polys])
    lo, hi = v.min(0), v.max(0)
    xs = bounds[0] + 10.0 * np.arange(int((hi[0] - bounds[0]) / 10) + 2)
    ys = bounds[1] + 10.0 * np.arange(int((hi[1] - bounds[1]) / 10) + 2)
    lat = np.concatenate([np.stack([np.repeat(xs, 6), rs.uniform(lo[1], hi[1], 6 * len(xs))], 1),
                          np.stack([rs.uniform(lo[0], hi[0], 6 * len(ys)), np.repeat(ys, 6)], 1),
                          np.stack(np.meshgrid(xs, ys), -1).reshape(-1, 2)])
    box = np.array([[lo[0], lo[1]], [hi[0], hi[1]], [lo[0], hi[1]], [hi[0], lo[1]],
                    [np.nextafter(lo[0], -np.inf), lo[1]], [np.nextafter(hi[0], np.inf), hi[1]],
                    [lo[0], np.nextafter(lo[1], -np.inf)], [hi[0], np.nextafter(hi[1], np.inf)]])
    return np.concatenate([v, mids, lat, box, np.asarray(extra, np.float64).reshape(-1, 2)])


def _as_tracks(pts, n_sharks, horizon, seed):
    """points dealt to n_sharks tracks with time stamps over [0, horizon], the last one of each track at horizon"""
    rs = np.random.RandomState(seed)
    pts = pts[rs.permutation(len(pts))]
    out = []
    for part in np.array_split(pts, n_sharks):
        t = np.sort(rs.uniform(0.0, horizon, len(part)))
        t[-1] = horizon
        out.append(np.column_stack([part, t]))
    return out


@pytest.mark.gpu
def test_index_exact_on_lattice_lines_corners_and_edges(occ_golden, catalina_map):
    polys, bounds, _ = occ_golden
    pts = _edge_points(polys, bounds, catalina_map["boundary"], 1)
    for n_sharks in (3, 17):
        tracks = _as_tracks(pts, n_sharks, 199.0, n_sharks)
        want = orc.occupancy(polys, bounds, 10.0, 50.0, 50.0, tracks)
        got, t_occ, _ = _grid_dev(polys, bounds, 10.0, 50.0, 50.0, tracks, len(want))
        assert t_occ == len(want) == 3 and np.array_equal(got, want)


@pytest.mark.gpu
def test_index_exact_on_non_lattice_clip():
    """cells of splitCell over the non-convex 40-vertex ring of the `coast` world: clipped edges at every angle"""
    import envelope_worlds as ew
    sys.path.insert(0, PP)
    for n in ("sharkOccupancyGrid", "_world", "motion_plan_state"):
        sys.modules.pop(n, None)
    try:
        import sharkOccupancyGrid as sog
        ring = ew.coast()[0]["boundary"]
        cells = sog.splitCell([tuple(p) for p in ring], 10)
    finally:
        sys.path.remove(PP)
    polys = [np.array(c.pts) for c in cells]
    bounds = np.array([ring[:, 0].min(), ring[:, 1].min(), ring[:, 0].max(), ring[:, 1].max()])
    rs = np.random.RandomState(2)
    extra = np.concatenate([ring, np.stack([rs.uniform(bounds[0], bounds[2], 4000), rs.uniform(bounds[1], bounds[3], 4000)], 1)])
    pts = _edge_points(polys, bounds, extra, 3)
    for cs_, rg in ((10.0, 50.0), (10.0, 25.0)):
        tracks = _as_tracks(pts, 8, 149.0, int(rg))
        want = orc.occupancy(polys, bounds, cs_, 50.0, rg, tracks)
        got, t_occ, _ = _grid_dev(polys, bounds, cs_, 50.0, rg, tracks, len(want))
        assert t_occ == len(want) == 2 and np.array_equal(got, want)


# ------------------------------------------------------------------ 3. refreshing a live world

def _plans(env, prec, group):
    from auvrrt import api
    Q = 48
    starts = np.tile([-200.0, 0.0, 0.0, 0.0, 0.0], (Q, 1))
    starts[:, 0] += np.linspace(-60, 60, Q)
    r = api.plan_batch(env, starts, np.arange(Q) + 11, api.plan_params(384, group=group, bin_interval=50.0), prec)
    return r["records"].tobytes(), r["chain"].tobytes()


def _costs(env, prec):
    from auvrrt import api
    rs = np.random.RandomState(9)
    paths = [np.column_stack([-300 + 200 * rs.random_sample(40), -40 + 120 * rs.random_sample(40), np.sort(rs.uniform(0, 450, 40))])
             for _ in range(64)]
    return api.cost(env, paths, np.full(64, 450.0), [-3.0, -3.0, -4.0], precision=prec).tobytes()


def _same_outputs(a, b):
    for prec in ("f64", "f32"):
        for group in (32, 1):
            assert _plans(a, prec, group) == _plans(b, prec, group), (prec, group)
        assert _costs(a, prec) == _costs(b, prec), prec


@pytest.mark.gpu
def test_refresh_world_equals_fresh_world(occ_golden, catalina_map, raw_tracks, shark_grid):
    import torch
    from auvrrt import api
    from auvrrt import device as adev
    polys, bounds, _ = occ_golden
    want = _cell_table(orc.occupancy(polys, bounds, 10.0, 50.0, 50.0, raw_tracks), polys, bounds, 10.0)
    T = _t_occ(50.0, raw_tracks)
    assert T == 9 and want.shape == (9, 986)
    occ = adev.SharkOccupancy(polys, bounds, 10.0, 50.0, 50.0, T, 32, 32 * 815)
    trk, off = _dev_tracks(raw_tracks)
    t_occ = torch.zeros(1, dtype=torch.int32, device="cuda")
    for start in (np.zeros((T, 986)), shark_grid[1][:T]):                # zeros, or the CSV grid's first rows
        env = api.Env.from_map(catalina_map, _bins(T), start)
        assert np.array_equal(env.probs("f64"), start)
        occ.grid_dev(trk, off, env=env, t_occ=t_occ)
        torch.cuda.synchronize()
        assert int(t_occ.item()) == T
        assert np.array_equal(env.probs("f64"), want)
        assert np.array_equal(env.probs("f32"), want.astype(np.float32).astype(np.float64))
        fresh = api.Env.from_map(catalina_map, _bins(T), want)
        _same_outputs(env, fresh)
    zero = api.Env.from_map(catalina_map, _bins(T), np.zeros((T, 986)))
    assert _costs(zero, "f64") != _costs(env, "f64")                        # the refreshed table is what the cost reads


@pytest.mark.gpu
def test_refresh_fewer_bins_than_tracks(occ_golden, catalina_map, raw_tracks):
    import torch
    from auvrrt import api
    from auvrrt import device as adev
    polys, bounds, _ = occ_golden
    want = _cell_table(orc.occupancy(polys, bounds, 10.0, 50.0, 50.0, raw_tracks), polys, bounds, 10.0)
    occ = adev.SharkOccupancy(polys, bounds, 10.0, 50.0, 50.0, 5, 32, 32 * 815)
    env = api.Env.from_map(catalina_map, _bins(5), None)
    trk, off = _dev_tracks(raw_tracks)
    t_occ = torch.zeros(1, dtype=torch.int32, device="cuda")
    occ.grid_dev(trk, off, env=env, t_occ=t_occ)
    torch.cuda.synchronize()
    assert int(t_occ.item()) == 9
    assert np.array_equal(env.probs("f64"), want[:5])
    _same_outputs(env, api.Env.from_map(catalina_map, _bins(5), want[:5]))


# ------------------------------------------------------------------ 4. asynchronous, allocation-free

@pytest.mark.gpu
def test_refresh_captures_into_cuda_graph(occ_golden, catalina_map, raw_tracks):
    import torch
    from auvrrt import api
    from auvrrt import device as adev
    polys, bounds, _ = occ_golden
    T = 9
    occ = adev.SharkOccupancy(polys, bounds, 10.0, 50.0, 50.0, T, 32, 32 * 815)
    env = api.Env.from_map(catalina_map, _bins(T), None)
    trk, off = _dev_tracks(raw_tracks)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        occ.grid_dev(trk, off, env=env)                                    # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        occ.grid_dev(trk, off, env=env)
    rs = np.random.RandomState(12)
    moved = [np.column_stack([t[:, 0] + rs.normal(0, 8.0, len(t)), t[:, 1] + rs.normal(0, 8.0, len(t)), t[:, 2]])
             for t in raw_tracks]
    new_trk, _ = _dev_tracks(moved)
    trk.copy_(new_trk)                                                      # new tracks, same tensor
    g.replay()
    torch.cuda.synchronize()
    want = _cell_table(orc.occupancy(polys, bounds, 10.0, 50.0, 50.0, moved), polys, bounds, 10.0)
    assert np.array_equal(env.probs("f64"), want)
    other = api.Env.from_map(catalina_map, _bins(T), None)
    occ.grid_dev(new_trk, off, env=other)                                   # the same refresh, not captured
    torch.cuda.synchronize()
    assert np.array_equal(other.probs("f64"), want)
    _same_outputs(env, other)


@pytest.mark.gpu
def test_refresh_launch_count(occ_golden, catalina_map, raw_tracks):
    import torch
    from auvrrt import api
    from auvrrt import device as adev
    polys, bounds, _ = occ_golden
    occ = adev.SharkOccupancy(polys, bounds, 10.0, 50.0, 50.0, 9, 32, 32 * 815)
    env = api.Env.from_map(catalina_map, _bins(9), None)
    trk, off = _dev_tracks(raw_tracks)
    out = torch.empty(occ.grid_shape, dtype=torch.float64, device="cuda")
    for kw, n in ((dict(env=env), 5), (dict(out=out), 4), (dict(out=out, env=env), 5)):
        l0 = api.launch_count()
        occ.grid_dev(trk, off, **kw)
        assert api.launch_count() - l0 == n, kw
    empty = torch.zeros((0, 3), dtype=torch.float64, device="cuda")
    l0 = api.launch_count()
    occ.grid_dev(empty, torch.zeros(33, dtype=torch.int64, device="cuda"), env=env)     # no points: no histogram
    assert api.launch_count() - l0 == 4
    torch.cuda.synchronize()


# ------------------------------------------------------------------ 5. rejections and the table entries

@pytest.mark.gpu
def test_rejections_leave_the_world_unchanged(occ_golden, catalina_map, raw_tracks, shark_grid):
    import torch
    from auvrrt import api
    from auvrrt import device as adev
    polys, bounds, _ = occ_golden
    occ = adev.SharkOccupancy(polys, bounds, 10.0, 50.0, 50.0, 9, 32, 32 * 815)
    trk, off = _dev_tracks(raw_tracks)
    start = shark_grid[1][:9]
    good = api.Env.from_map(catalina_map, _bins(9), start)
    bad_bins = _bins(9)
    bad_bins[4, 1] = np.nextafter(bad_bins[4, 1], 0)
    worlds = [api.Env.from_map(catalina_map, _bins(8), shark_grid[1][:8]),                     # T mismatch
              api.Env(catalina_map["circles"], catalina_map["boundary"], catalina_map["habitats"], _bins(9),
                      catalina_map["cells"][:985], start[:, :985]),                                # C mismatch
              api.Env.from_map(catalina_map, bad_bins, start),                                   # bins mismatch
              api.Env.from_map(catalina_map, _bins(9, 40.0), start)]                             # bin interval mismatch
    for w in worlds:
        before = w.probs("f64")
        with pytest.raises(api._lib.AuvrrtError, match="bin|cells"):
            occ.grid_dev(trk, off, env=w)
        torch.cuda.synchronize()
        assert np.array_equal(w.probs("f64"), before)
    many, many_off = _dev_tracks(raw_tracks + raw_tracks[:1])                                  # 33 sharks
    short = adev.SharkOccupancy(polys, bounds, 10.0, 50.0, 50.0, 9, 32, 32 * 815 - 1)
    for o, t, f in ((occ, many, many_off), (short, trk, off)):
        with pytest.raises(api._lib.AuvrrtError, match="sharks|points"):
            o.grid_dev(t, f, env=good)
    cpu = trk.cpu()
    for t, f in ((trk.float(), off), (cpu, off), (trk[:, :2].contiguous(), off), (trk.t().contiguous().t(), off),
                 (trk, off.int()), (trk, off.view(1, -1)), (trk.reshape(-1), off)):
        with pytest.raises(ValueError):
            occ.grid_dev(t, f, env=good)
    with pytest.raises(ValueError):
        occ.grid_dev(trk, off, out=torch.empty((9, 35, 55), dtype=torch.float64, device="cuda"), env=good)
    with pytest.raises(ValueError):
        occ.grid_dev(trk, off, t_occ=torch.empty(1, dtype=torch.int64, device="cuda"), env=good)
    with pytest.raises(ValueError):
        good.set_probs(start[:, :-1])
    with pytest.raises(ValueError):
        adev.env_set_probs_dev(good, torch.from_numpy(start).float().cuda())
    with pytest.raises(ValueError):
        adev.env_set_probs_dev(good, torch.from_numpy(start))
    torch.cuda.synchronize()
    assert np.array_equal(good.probs("f64"), start)
    assert np.array_equal(good.probs("f32"), start.astype(np.float32).astype(np.float64))


@pytest.mark.gpu
def test_set_probs_round_trip(catalina_map):
    import torch
    from auvrrt import api
    from auvrrt import device as adev
    rs = np.random.RandomState(3)
    env = api.Env.from_map(catalina_map, _bins(6), None)
    a = rs.random_sample((6, 986)) * 0.7
    env.set_probs(a)
    assert np.array_equal(env.probs("f64"), a) and np.array_equal(env.probs("f32"), a.astype(np.float32).astype(np.float64))
    _same_outputs(env, api.Env.from_map(catalina_map, _bins(6), a))
    b = torch.from_numpy(rs.random_sample((6, 986))).cuda()
    adev.env_set_probs_dev(env, b)
    torch.cuda.synchronize()
    assert np.array_equal(env.probs(), b.cpu().numpy())
    assert np.array_equal(env.probs("f32"), b.cpu().numpy().astype(np.float32).astype(np.float64))
    empty = api.Env.from_map(catalina_map, (), None)                       # T == 0: nothing to write
    empty.set_probs(np.zeros((0, 986)))
    assert empty.probs().shape == (0, 986)


# ------------------------------------------------------------------ 6. compile

def test_occupancy_kernels_spill_nothing():
    nvcc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    if not os.path.exists(nvcc):
        nvcc = "nvcc"
    with tempfile.TemporaryDirectory() as d:
        r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
                            "-diag-suppress", "128", "-Xptxas", "-v", "-c", "-o", os.path.join(d, "occupancy.o"),
                            os.path.join(CSRC, "occupancy.cu")], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout[-3000:]
    props = re.findall(r"Function properties for (\S+)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads",
                       r.stdout)
    names = {n for n, *_ in props}
    for k in ("k_occ_hist", "k_occ_norm", "k_occ_auv", "k_occ_avg", "k_occ_to_env"):
        assert any(k in n for n in names), k
    for n, _, st, ld in props:
        assert st == "0" and ld == "0", (n, st, ld)
