"""GPU: per-episode reset of the vectorised gym planner (auvrrt_gym_reset_dev, k_gym_reset_masked) and the
torch environment built on it (gym_rrt.envs.DeviceVecRRTEnv, next-step auto-reset).

A recycled slot must replay a fresh episode exactly: the masked reset and a full reset of a second batch feed the
same kernel the same inputs, so records, trees, counts and paths are compared array-equal, in both builds."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle.harness import GYM_MAIN_OBSTACLES  # noqa: E402

MAIN = (0, 0, 50, 50)


@pytest.fixture(scope="module")
def mods():
    import torch
    import auvrrt
    from auvrrt import device, gym
    assert auvrrt.api.device_count() > 0
    return torch, gym, device


def _episodes(Q, seed):
    rs = np.random.default_rng(seed)
    starts = np.column_stack([rs.uniform(5, 15, Q), rs.uniform(5, 15, Q), rs.uniform(-np.pi, np.pi, Q)])
    goals = np.column_stack([rs.uniform(35, 45, Q), rs.uniform(35, 45, Q)])
    return starts, goals


def _gym_dtype():
    from auvrrt.gym import GYM_RECORD_DTYPE
    return GYM_RECORD_DTYPE


def _recs(t):
    """uint8 [Q, 88] device records -> GYM_RECORD_DTYPE [Q]"""
    return np.frombuffer(t.cpu().numpy().tobytes(), dtype=_gym_dtype())


def _agent(rs, cnt, n_subcells, q_never=(), mix=True):
    """a random occupied sub-cell per episode, with empty cells and -1 mixed in; -1 for the episodes in q_never"""
    act = np.argmax((cnt > 0) * rs.random(cnt.shape), axis=1).astype(np.int32)
    if mix:
        empty = np.argmax((cnt == 0) * rs.random(cnt.shape), axis=1).astype(np.int32)
        pick = rs.random(len(act))
        act = np.where(pick < 0.1, empty, np.where(pick < 0.15, -1, act)).astype(np.int32)
    act[list(q_never)] = -1
    return act


def _dev_tensors(torch, dev, starts, goals, seeds):
    return (torch.from_numpy(np.ascontiguousarray(starts, np.float64)).to(dev),
            torch.from_numpy(np.ascontiguousarray(goals, np.float64)).to(dev),
            torch.from_numpy(np.asarray(seeds, np.uint64).view(np.int64).copy()).to(dev))


def _same_episode(a, qa, b, qb):
    ta, tb = a.tree(qa), b.tree(qb)
    for k in ta:
        assert np.array_equal(ta[k], tb[k]), (k, qa, qb)
    assert np.array_equal(a.counts(qa, 1), b.counts(qb, 1)), (qa, qb)
    assert np.array_equal(a.path(qa), b.path(qb)), (qa, qb)


@pytest.mark.parametrize("prec", ["f32", "f64"])
def test_recycled_slot_replays_fresh_episode(mods, prec):
    torch, gym, D = mods
    P = gym.F64 if prec == "f64" else gym.F32
    Q, k1, k2 = 512, 60, 60
    kw = dict(freq=10.0, node_cap=41, track_counts=True, precision=P)
    starts0, goals0 = _episodes(Q, 1)
    starts0[7::61] = [10.0, -120.0, 0.3]                    # off the grid: KeyError at __init__, status KEY_ERROR, n_occ = 0
    seeds0 = np.arange(Q, dtype=np.uint64) + 100
    never = np.arange(3, Q, 53)                             # never stepped before the masked reset
    A, C = (gym.GymBatch(MAIN, GYM_MAIN_OBSTACLES, Q, **kw) for _ in range(2))
    A.reset(starts0, goals0, seeds0)
    C.reset(starts0, goals0, seeds0)
    dev = torch.device("cuda", 0)
    d_act = torch.zeros(Q, dtype=torch.int32, device=dev)
    d_rec = torch.zeros((Q, 88), dtype=torch.uint8, device=dev)
    rs = np.random.default_rng(2)
    history = []

    def step_all(act, batches):
        d_act.copy_(torch.from_numpy(act))
        D.gym_step_dev(A, d_act, d_rec)
        out = [b.step(a) for b, a in batches]
        return _recs(d_rec), out

    for it in range(k1):
        act = _agent(rs, A.counts(), A.n_subcells, never)
        ra, (rc,) = step_all(act, [(C, act)])
        assert np.array_equal(ra, rc)
        history.append(act)
    st = ra["status"]
    done, over, keyerr = ra["done"] != 0, st == 5, (st == 3) & (ra["n_occupied"] == 0)
    assert done.any() and over.any() and keyerr.any(), (done.sum(), over.sum(), keyerr.sum())
    assert (ra["steps"][never] == 0).all()
    mask = rs.random(Q) < 0.25
    mask[never] = True
    mask[keyerr] = True
    mask[np.flatnonzero(done)[0]] = mask[np.flatnonzero(over)[0]] = True
    assert (~mask).sum() > 100 and (done & ~mask).any() and (over & ~mask).any()
    starts1, goals1 = _episodes(Q, 9)
    seeds1 = np.arange(Q, dtype=np.uint64) + 5000
    ds, dg, dd = _dev_tensors(torch, dev, np.where(mask[:, None], starts1, np.nan), np.where(mask[:, None], goals1, np.nan),
                              np.where(mask, seeds1, np.uint64(0)))      # rows outside the mask are not read: NaN there
    D.gym_reset_dev(A, torch.from_numpy(mask).to(dev), ds, dg, dd)
    # reference for the recycled slots: a full reset at time 0 with their new inputs, -1 until the reset
    B = gym.GymBatch(MAIN, GYM_MAIN_OBSTACLES, Q, **kw)
    B.reset(np.where(mask[:, None], starts1, starts0), np.where(mask[:, None], goals1, goals0), np.where(mask, seeds1, seeds0))
    for act in history:
        B.step(np.where(mask, -1, act).astype(np.int32))
    for it in range(k2):
        act = _agent(rs, A.counts(), A.n_subcells)
        ra, (rb, rc) = step_all(act, [(B, act), (C, act)])
        assert np.array_equal(ra[mask], rb[mask]), it
        assert np.array_equal(ra[~mask], rc[~mask]), it
    assert (ra["done"][mask] != 0).any() and (ra["status"][mask] == 5).any()
    for q in range(Q):
        _same_episode(A, q, B if mask[q] else C, q)
    for b in (A, B, C):
        b.close()


def _home(c, hsize):
    shift = 32 - int(hsize).bit_length() + 1
    return ((int(c) * 2654435761) & 0xFFFFFFFF) >> shift


def test_no_ghost_cells(mods):
    torch, gym, D = mods
    Q, cap = 256, 101
    hsize = 16
    while hsize < 2 * cap:
        hsize <<= 1
    kw = dict(freq=10.0, node_cap=cap, track_counts=True, precision=gym.F32)
    starts, goals = _episodes(Q, 4)
    A = gym.GymBatch(MAIN, GYM_MAIN_OBSTACLES, Q, **kw)
    A.reset(starts, goals, np.arange(Q) + 7)
    rs = np.random.default_rng(5)
    for it in range(90):
        A.step(_agent(rs, A.counts(), A.n_subcells, mix=False))
    old = [A.tree(q)["occupied"] for q in range(Q)]
    mask = np.zeros(Q, bool)
    mask[::2] = True
    # the clear must undo probe chains: some recycled episode held two cells with the same home slot
    collide = [q for q in np.flatnonzero(mask) if len({_home(c, hsize) for c in old[q]}) < len(old[q])]
    assert len(collide) > 10, len(collide)
    starts1, goals1 = _episodes(Q, 6)
    dev = torch.device("cuda", 0)
    ds, dg, dd = _dev_tensors(torch, dev, starts1, goals1, np.arange(Q) + 900)
    D.gym_reset_dev(A, torch.from_numpy(mask.astype(np.uint8)).to(dev), ds, dg, dd)
    fresh = [A.tree(q)["occupied"] for q in range(Q)]
    ghosts = {q: [c for c in old[q] if c not in set(fresh[q])] for q in np.flatnonzero(mask)}
    assert np.mean([len(g) > 5 for g in ghosts.values()]) > 0.5
    before = A.step(np.full(Q, -1, np.int32))
    for r in range(max(len(g) for g in ghosts.values())):
        act = np.full(Q, -1, np.int32)
        for q, g in ghosts.items():
            act[q] = g[r % len(g)] if g else -1
        rec = A.step(act)
        assert (rec["last_parent"][mask] == -1).all(), r
        assert np.array_equal(rec["n_uniforms"][mask], before["n_uniforms"][mask])
        assert (rec["n_nodes"][mask] == 1).all() and (rec["steps"][mask] == 0).all()
    cnt = A.counts()
    assert np.array_equal(cnt[mask].sum(1), np.ones(mask.sum()))
    # and the recycled episodes keep growing exactly like freshly created ones
    B = gym.GymBatch(MAIN, GYM_MAIN_OBSTACLES, Q, **kw)
    B.reset(starts1, goals1, np.arange(Q) + 900)
    for it in range(60):
        cnt = A.counts()
        act = _agent(rs, cnt, A.n_subcells, mix=False)
        ra, rb = A.step(act), B.step(act)
        assert np.array_equal(ra[mask], rb[mask]), it
    cnt = A.counts()
    assert np.array_equal(cnt.sum(1), ra["n_nodes"])      # main()'s world: every node has a sub-cell
    A.close(); B.close()


def test_golden_after_masked_reset(mods, gym_golden):
    """the unmodified reference's step-by-step episodes, replayed in a slot recycled through the masked path"""
    torch, gym, D = mods
    dev = torch.device("cuda", 0)
    eps = [ep for ep in gym_golden if ep.name.startswith("step")]
    assert len(eps) == 6
    for ep in eps:
        Q = 3
        b = gym.GymBatch(ep.boundary, ep.obstacles, Q, freq=ep.freq, cell_side_length=ep.cell_side,
                         subsections_in_cell=ep.subsections, node_cap=ep.max_step + 1, track_counts=True, precision=gym.F64)
        st, go = _episodes(Q, 3)
        b.reset(st, go, np.arange(Q) + 77)
        rs = np.random.default_rng(8)
        for it in range(40):
            b.step(_agent(rs, b.counts(), b.n_subcells))
        mask = np.array([0, 1, 0], np.uint8)
        ds, dg, dd = _dev_tensors(torch, dev, np.tile(ep.start, (Q, 1)), np.tile(ep.goal, (Q, 1)), np.full(Q, ep.seed, np.uint64))
        D.gym_reset_dev(b, torch.from_numpy(mask).to(dev), ds, dg, dd)
        acts = ep.flat(ep.actions)
        d_act = torch.full((Q,), -1, dtype=torch.int32, device=dev)
        d_rec = torch.zeros((Q, 88), dtype=torch.uint8, device=dev)
        s = 0
        for a in acts:
            d_act[1] = int(a)
            D.gym_step_dev(b, d_act, d_rec, full_candidates=True)
            r0 = _recs(d_rec)[1]
            assert r0["status"] == 0
            if r0["last_parent"] < 0:
                assert r0["steps"] == s
                continue
            assert r0["steps"] == s + 1
            assert r0["last_parent"] == ep.parent[s] and r0["last_nwp"] == ep.nwp[s], (ep.name, s)
            assert r0["last_accepted"] == ep.accepted[s] and r0["done"] == ep.done[s], (ep.name, s)
            assert r0["n_nodes"] == ep.n_nodes[s] and r0["n_occupied"] == ep.n_occupied[s]
            assert r0["last_uniforms"] == ep.n_uniforms[s]
            assert np.allclose(r0["cand"], ep.cand[s], rtol=1e-9, atol=1e-9), (ep.name, s)
            s += 1
        assert s == ep.steps
        t = b.tree(1)
        assert np.allclose(t["nodes"], ep.nodes, rtol=1e-9, atol=1e-9)
        assert np.array_equal(t["occupied"], ep.flat(ep.occupied))
        cnt = b.counts(1, 1)[0]
        nz = np.flatnonzero(cnt)
        assert np.array_equal(np.stack([nz, cnt[nz]], 1), ep.counts_nz)
        if ep.found:
            assert r0["done"] == 1 and r0["n_path"] == len(ep.path)
            assert np.allclose(b.path(1), ep.path, rtol=1e-9, atol=1e-9)
        b.close()


# ---- DeviceVecRRTEnv ----------------------------------------------------------------------------------------

def _env(Q, prec="f32", max_episode_steps=200, **kw):
    from gym_rrt.envs import DeviceVecRRTEnv
    return DeviceVecRRTEnv(MAIN, GYM_MAIN_OBSTACLES, Q, freq=10, precision=prec, max_episode_steps=max_episode_steps, **kw)


def _policy(torch, obs, gen):
    """a random occupied sub-cell: argmax of noise x (obs > 0); torch has no uint16 comparison, counts stay < 2^15"""
    noise = torch.rand(obs.shape, device=obs.device, generator=gen)
    return torch.argmax(noise * (obs.view(torch.int16) > 0), dim=1).to(torch.int32)


def test_env_terminal_observation_then_fresh_start(mods):
    torch, gym, D = mods
    Q = 256
    env = _env(Q)
    starts, goals = _episodes(Q, 12)
    seeds = np.arange(Q, dtype=np.uint64) + 31
    obs = env.reset(starts, goals, seeds)
    assert obs.dtype == torch.uint16 and obs.shape == (Q, env.n_actions)
    fresh = gym.GymBatch(MAIN, GYM_MAIN_OBSTACLES, Q, freq=10.0, node_cap=257, track_counts=True)
    fresh.reset(starts, goals, seeds)
    one_hot = fresh.counts()
    gen = torch.Generator(device="cuda").manual_seed(0)
    checked = 0
    pending = None
    for t in range(150):
        obs, rew, term, trunc, info = env.step(_policy(torch, obs, gen))
        if pending is not None:
            qs = pending
            assert info["reset"][qs].all() and (rew[qs] == 0).all()
            assert not term[qs].any() and not trunc[qs].any()
            q_np = qs.cpu().numpy()
            assert np.array_equal(obs.cpu().numpy()[q_np], one_hot[q_np])       # the start cell alone
            checked += len(q_np)
            pending = None
        if term.any():
            qs = torch.nonzero(term).flatten()
            rec = np.frombuffer(info["records"].cpu().numpy().tobytes(), _gym_dtype())
            o = obs.cpu().numpy()
            assert (rew[qs] == 300).all()
            for q in qs.cpu().numpy()[:4]:
                c = env.batch.tree(int(q))["cells"]
                assert np.array_equal(o[q], np.bincount(c[c >= 0], minlength=env.n_actions))
                assert o[q].sum() == rec["n_nodes"][q]
            pending = qs
    assert checked > 5, checked
    env.close(); fresh.close()


def test_env_truncates_on_the_last_step(mods):
    torch, gym, D = mods
    Q, T = 64, 7
    env = _env(Q, max_episode_steps=T)
    starts, goals = _episodes(Q, 13)
    env.reset(starts, goals, np.arange(Q))
    act = torch.full((Q,), -1, dtype=torch.int32, device="cuda")          # nothing grows: only the time limit ends it
    for call in range(1, 3 * (T + 1) + 1):
        obs, rew, term, trunc, info = env.step(act)
        k = call % (T + 1)                          # calls T, 2T + 1, ... end an episode; the call after each resets
        assert not term.any()
        assert bool(info["reset"].all()) == (k == 0) and not (k != 0 and info["reset"].any()), call
        assert bool(trunc.all()) == (k == T) and not (k != T and trunc.any()), call
        assert (rew == (0 if k == 0 else -1)).all()
    env.close()


@pytest.mark.parametrize("prec", ["f32", "f64"])
def test_env_second_episode_matches_host_batch(mods, prec):
    torch, gym, D = mods
    Q = 128
    env = _env(Q, prec, max_episode_steps=15, max_nodes=41)
    starts, goals = _episodes(Q, 14)
    seeds = np.arange(Q, dtype=np.uint64) + 3
    obs = env.reset(starts, goals, seeds)
    ref = gym.GymBatch(MAIN, GYM_MAIN_OBSTACLES, Q, freq=10.0, node_cap=41, track_counts=True,
                       precision=gym.F64 if prec == "f64" else gym.F32)
    ref.reset(starts, goals, seeds + np.uint64(Q))
    gen = torch.Generator(device="cuda").manual_seed(1)
    compared = 0
    for t in range(50):
        act = _policy(torch, obs, gen)
        obs, rew, term, trunc, info = env.step(act)
        in1 = ((env.episode == 1) & ~info["reset"]).cpu().numpy()
        rr = ref.step(np.where(in1, act.cpu().numpy(), -1).astype(np.int32))
        got = np.frombuffer(info["records"].cpu().numpy().tobytes(), _gym_dtype())
        assert np.array_equal(got[in1], rr[in1]), t
        compared += int(in1.sum())
    assert compared > 5 * Q
    env.close(); ref.close()


def test_env_deterministic_sync_free_two_launches(mods):
    torch, gym, D = mods
    from auvrrt import api
    Q = 512
    starts, goals = _episodes(Q, 15)
    envs = [_env(Q, max_episode_steps=30) for _ in range(2)]
    obs = [e.reset(starts, goals, np.arange(Q) + 11) for e in envs]
    gens = [torch.Generator(device="cuda").manual_seed(3) for _ in envs]
    outs = [[], []]
    n = 80
    torch.cuda.synchronize()
    l0 = api.launch_count()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for t in range(n):
            for i, e in enumerate(envs):
                o, rew, term, trunc, info = e.step(_policy(torch, obs[i], gens[i]))
                outs[i].append((o.view(torch.int16).clone(), rew, term, trunc, info["reset"], info["status"], info["records"].clone()))
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert api.launch_count() - l0 == 2 * 2 * n
    ended = 0
    for a, b in zip(*outs):
        for x, y in zip(a, b):
            assert torch.equal(x, y)
        ended += int(a[4].sum())
    assert ended > Q                                  # slots were recycled along the way
    for e in envs:
        e.close()


def test_errors(mods):
    torch, gym, D = mods
    from auvrrt._lib import AuvrrtError, lib
    Q = 8
    dev = torch.device("cuda", 0)
    b = gym.GymBatch(MAIN, GYM_MAIN_OBSTACLES, Q, freq=10.0, node_cap=17, track_counts=True)
    starts, goals = _episodes(Q, 16)
    ds, dg, dd = _dev_tensors(torch, dev, starts, goals, np.arange(Q))
    mask = torch.ones(Q, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    # a masked reset reads the previous tree: refused before any full reset
    assert lib().auvrrt_gym_reset_dev(b.handle, mask.data_ptr(), ds.data_ptr(), dg.data_ptr(), dd.data_ptr(), stream) == 1
    with pytest.raises(AuvrrtError):
        D.gym_reset_dev(b, mask, ds, dg, dd)
    D.gym_reset_dev(b, None, ds, dg, dd)
    D.gym_reset_dev(b, mask, ds, dg, dd)
    torch.cuda.synchronize()
    bad = [(mask.cpu(), ds, dg, dd), (mask.float(), ds, dg, dd), (mask[:4], ds, dg, dd), (mask, ds.float(), dg, dd),
           (mask, ds[:, :2], dg, dd), (mask, ds, dg.t().contiguous().t(), dd), (mask, ds, dg, dd.int()), (mask, ds, dg, dd[:-1]),
           (mask, ds.cpu(), dg, dd)]
    for args in bad:
        with pytest.raises(ValueError):
            D.gym_reset_dev(b, *args)
    rec = torch.zeros((Q, 88), dtype=torch.uint8, device=dev)
    act = torch.zeros(Q, dtype=torch.int32, device=dev)
    for a, r in [(act.long(), rec), (act.cpu(), rec), (act[:3], rec), (act, rec.view(-1)), (act, rec[:, :80]),
                 (act, rec.cpu())]:
        with pytest.raises(ValueError):
            D.gym_step_dev(b, a, r)
    nc = gym.GymBatch(MAIN, GYM_MAIN_OBSTACLES, Q, freq=10.0, node_cap=17)
    with pytest.raises(ValueError):
        D.gym_counts_tensor(nc)
    nc.close()
    view = D.gym_counts_tensor(b)
    assert view.dtype == torch.uint16 and view.shape == (Q, b.n_subcells) and view.device == dev
    assert np.array_equal(view.cpu().numpy(), b.counts())
    b.close()
    env = _env(Q)
    with pytest.raises(RuntimeError):
        env.step(act)
    env.reset(starts, goals, np.arange(Q))
    for a in (act.long(), act.cpu(), act[:3]):
        with pytest.raises(ValueError):
            env.step(a)
    env.close()
