"""GPU: next-step auto-reset (BatchedNavGym(auto_reset='next_step'), auto_reset =
NAVGYM_AUTORESET_NEXT_STEP).

The defining property: an environment that ends an episode returns its final observation, and the
following launch ignores its action and starts the next episode exactly as reset_envs(done) would
have.  So for the same per-episode actions every (env, episode, step) record of a next-step env is
the record of an auto_reset=False env that calls reset_envs(done) after every step; the next-step
env only lags by one launch per ended episode.  Also: one launch in detail (NaN actions of the
resetting environments, hits, outputs), the launch order, the pending flag after host-side
resets, the host-buffer paths, sharding, scripted pedestrians and rejected input."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
NB = 512
OUTPUTS = ('reward', 'done', 'is_success', 'is_crash', 'truncated', 'distance')
ROWS = ('obs', 'tail64', 'steps', 'episodes', 'map_id', 'noise_std')   # [B, ...] per-env buffers


@pytest.fixture(scope='module')
def world():
    """Two outdoor maps with spawn pools (for resample_map) and a bank of scripted pedestrians."""
    from nav_gym_b200 import maps, worlds
    from nav_gym_b200.batched_env import MapPool, filter_spawn_pool
    rng = np.random.RandomState(43)
    ms, pools = [], []
    for _ in range(2):
        m = maps.create_outdoor_map(10, 0.7, rng)
        pools.append(filter_spawn_pool(m, maps.spawn_pool(m, 4096, rng, min_goal_dist=1.5, max_goal_dist=6)))
        ms.append(m)
    mp = MapPool(ms, 'cuda:0', spawn_pools=pools)
    bank = worlds.scripted_pedestrians(ms[0], 1, 256, rng)[0]   # [256, 16] waypoint walkers
    return ms, mp, bank


def _bits(t):
    return t.view({torch.float64: torch.int64, torch.float32: torch.int32, torch.float16: torch.int16}[t.dtype]) \
        if t.is_floating_point() else t


def _env(world, B, auto_reset, seed=3, spawn_seed=None, **kw):
    """An env on the two-map pool with random start maps and spawns from the pools; two calls that
    differ only in auto_reset build the same env."""
    from nav_gym_b200.batched_env import BatchedNavGym
    _, mp, _ = world
    map_id = np.random.RandomState(seed).randint(0, 2, B).astype(np.int32)
    kw.setdefault('record_hits', True)
    e = BatchedNavGym(B, mp, map_id=map_id, seed=seed, auto_reset=auto_reset, **kw)
    e.reset_from_spawn_pool(np.random.RandomState(seed + 1 if spawn_seed is None else spawn_seed))
    return e


def _obstacles(env, seed):
    """Static explicit obstacles, the same for every launch: four discs per env within 3 m of its
    start and two short box segments, so that scans see them and crashes occur."""
    rng = np.random.RandomState(seed)
    B = env.B
    pos = env.state[:2].T.cpu().numpy()
    discs = np.zeros((B, 4, 3), np.float32)
    discs[..., :2] = pos[:, None, :] + rng.uniform(-3, 3, (B, 4, 2))
    discs[..., 2] = rng.uniform(0.1, 0.4, (B, 4))
    a = pos[:, None, :] + rng.uniform(-3, 3, (B, 2, 2))
    segs = np.concatenate([a, a + rng.uniform(-1, 1, (B, 2, 2))], axis=2).astype(np.float32)
    dev = lambda x, t: torch.from_numpy(np.ascontiguousarray(x)).to('cuda', t)
    return dict(discs=dev(discs, torch.float32), ndisc=dev(rng.randint(0, 5, B), torch.int32),
                segs=dev(segs, torch.float32), nseg=dev(rng.randint(0, 3, B), torch.int32))


def _policy(env):
    """Actions that depend only on (global env id, episode, step, state): head for the goal, plus a
    hashed perturbation.  Two envs in the same (episode, step, state) get the same action, whatever
    the launch index."""
    from nav_gym_b200 import _lib
    st = env.state
    bearing = torch.atan2(st[_lib.S_GY] - st[_lib.S_PY], st[_lib.S_GX] - st[_lib.S_PX]) - st[_lib.S_TH]
    err = torch.remainder(bearing + np.pi, 2 * np.pi) - np.pi
    gid = torch.arange(env.B, device=env.device, dtype=torch.int64) + int(env.args.env_offset)
    h = (gid * 2654435761 + env.episodes.long() * 40503 + env.steps.long() * 9973) % 1000003
    u1 = (h % 1024).double() / 1024.0
    u2 = ((h // 1024) % 1024).double() / 1024.0
    w = (1.5 * err + 0.8 * (u1 - 0.5)).clamp(-0.64, 0.64)
    v = 0.3 + 0.2 * u2
    return torch.stack([v, w], dim=1).float().contiguous()


def _goal_distance(env):
    """float32 of the float64 distance from pose to goal, computed as the step computes it."""
    from nav_gym_b200 import _lib
    st = env.state
    dx, dy = st[_lib.S_GX] - st[_lib.S_PX], st[_lib.S_GY] - st[_lib.S_PY]
    return torch.sqrt(dx * dx + dy * dy).float()


def _snap(env, names):
    out = {n: getattr(env, n).clone() for n in names}
    out['state'] = env.state.T.clone()
    return out


@pytest.mark.parametrize('B', [777, 6144])
@pytest.mark.parametrize('S', [1, 3])
@pytest.mark.parametrize('dtype', [torch.float32, torch.float16])
def test_next_step_records_equal_reset_envs_after_every_step(world, B, S, dtype):
    """Env A steps with auto_reset='next_step'; env B with auto_reset=False and reset_envs(done)
    after every step.  Every record of A, keyed by (env, episode, step), equals B's: the stepped
    ones B's step, the reset ones B's row after reset_envs.  Philox noise, static obstacles,
    max_episode_steps and resample_map on the two-map pool; 777 and 6144 environments run the COOP
    and the non-COOP instantiations on a 148-SM part."""
    T = 60
    kw = dict(num_scan_stack=S, obs_dtype=dtype, max_episode_steps=25, resample_map=True, max_disc=4, max_seg=2)
    a = _env(world, B, 'next_step', **kw)
    b = _env(world, B, False, **kw)
    geom = _obstacles(a, B + S)
    map0 = a.map_id.clone()
    step_names = ROWS + OUTPUTS + ('hits',)
    # B's records: launch t's step, and its rows after reset_envs(done)
    hist_step = {n: torch.empty((T,) + tuple(getattr(b, n).shape), dtype=getattr(b, n).dtype, device='cuda')
                 for n in step_names}
    hist_step['state'] = torch.empty(T, B, b.state.shape[0], dtype=torch.float64, device='cuda')
    hist_reset = {n: torch.empty_like(hist_step[n]) for n in ROWS + ('state',)}
    ar = torch.arange(B, device='cuda')
    lag = torch.zeros(B, dtype=torch.int64, device='cuda')   # A's reset launches so far, per env
    n_reset = n_crash = n_succ = n_trunc = 0
    for t in range(T):
        b.step(_policy(b), **geom)
        for n, v in _snap(b, step_names).items():
            hist_step[n][t] = v
        b.reset_envs(b.done)
        for n, v in _snap(b, ROWS).items():
            hist_reset[n][t] = v

        _, _, _, info = a.step(_policy(a), **geom)
        rst = info['autoreset']
        assert torch.equal(rst, a.steps == 0)
        lag += rst.long()
        idx = t - lag
        assert int(idx.min()) >= 0
        got = _snap(a, step_names)
        for n in ROWS + ('state',):
            want = torch.where(rst.view(-1, *[1] * (got[n].dim() - 1)), hist_reset[n][idx, ar], hist_step[n][idx, ar])
            assert torch.equal(_bits(got[n]), _bits(want)), (t, n)
        keep = ~rst
        for n in OUTPUTS + ('hits',):
            assert torch.equal(_bits(got[n][keep]), _bits(hist_step[n][idx, ar][keep])), (t, n)
        for n in OUTPUTS[:-1]:
            assert not bool(got[n][rst].any()), (t, n)
        assert torch.equal(_bits(a.distance[rst]), _bits(_goal_distance(a)[rst])), t
        n_reset += int(rst.sum())
        n_crash += int(a.is_crash.sum())
        n_succ += int(a.is_success.sum())
        n_trunc += int(a.truncated.sum())
    assert n_reset > 0 and n_crash > 0 and n_succ > 0 and n_trunc > 0, (n_reset, n_crash, n_succ, n_trunc)
    assert bool((a.map_id != map0).any())   # resample_map drew other maps


def test_one_launch_in_detail(world):
    """Three twins step identically until some episode ends.  Then A's next-step launch (NaN
    actions for the envs that reset) gives, bit for bit, what reset_envs(done) gives on twin B for
    the ended envs, with outputs 0, the goal distance of the new state and the reset scan's hits;
    and what a plain auto_reset=False step gives on twin C for the others."""
    B = 777
    kw = dict(max_episode_steps=12, resample_map=True, max_disc=4, max_seg=2)
    a, b, c = _env(world, B, 'next_step', **kw), _env(world, B, False, **kw), _env(world, B, False, **kw)
    geom = _obstacles(a, 5)
    for t in range(30):
        act = _policy(a)
        for e in (a, b, c):
            e.step(act, **geom)
        if bool(a.done.any()):
            break
    mask = a.done.bool().clone()
    assert bool(mask.any()) and not bool(mask.all())
    for e in (b, c):
        assert torch.equal(_bits(e.obs), _bits(a.obs)) and torch.equal(e.done, a.done)
    act = _policy(a)
    nan_act = act.clone()
    nan_act[mask] = float('nan')
    b.reset_envs(mask)
    c.step(act, **geom)
    _, _, _, info = a.step(nan_act, **geom)
    assert torch.equal(info['autoreset'], mask)
    keep = ~mask
    for n in ROWS:
        x = _bits(getattr(a, n))
        assert torch.equal(x[mask], _bits(getattr(b, n))[mask]), n
        assert torch.equal(x[keep], _bits(getattr(c, n))[keep]), n
    assert torch.equal(_bits(a.state[:, mask]), _bits(b.state[:, mask]))
    assert torch.equal(_bits(a.state[:, keep]), _bits(c.state[:, keep]))
    for n in OUTPUTS + ('hits',):
        assert torch.equal(_bits(getattr(a, n))[keep], _bits(getattr(c, n))[keep]), n
    for n in OUTPUTS[:-1]:
        assert not bool(getattr(a, n)[mask].any()), n
    assert torch.equal(_bits(a.distance[mask]), _bits(_goal_distance(a)[mask]))
    assert bool((a.steps[mask] == 0).all()) and bool(torch.isfinite(a.state[:, mask]).all())
    # hits of the reset scan: reset() records the first scan's hits from the pose in `state`
    b.reset()
    assert torch.equal(a.hits[mask], b.hits[mask])


def _launch_order(env):
    """The env ids of the next step's launch order (the current third of the schedule buffer)."""
    from nav_gym_b200 import _lib
    nbk, B = _lib.SCHED_BUCKETS, env.B
    s = env.sched.cpu().numpy()
    cur = env.args.sched_phase
    cnt = s[cur * nbk:(cur + 1) * nbk]
    lists = s[3 * nbk:].reshape(3, nbk, B)[cur]
    return np.concatenate([lists[k, :cnt[k]] for k in range(nbk)])


def test_launch_order_lists_every_environment_once(world):
    B = 777
    env = _env(world, B, 'next_step', max_episode_steps=6)
    resets = 0
    for t in range(20):
        _, _, _, info = env.step(_policy(env))
        resets += int(info['autoreset'].sum())
        assert np.array_equal(np.sort(_launch_order(env)), np.arange(B)), t
    assert resets > 0


def test_host_side_resets_clear_the_pending_flag(world):
    """reset_envs(done) and reset_from_spawn_pool() in next-step mode clear done for the envs they
    reset: the following step steps them (steps == 1) instead of starting another episode."""
    B = 777
    env = _env(world, B, 'next_step', max_episode_steps=6)
    for _ in range(6):
        env.step(_policy(env))
        if bool(env.done.any()):
            break
    mask = env.done.bool().clone()
    assert bool(mask.any())
    ep = env.episodes.clone()
    env.reset_envs(env.done)
    assert not bool(env.done.any())
    assert torch.equal(env.episodes, ep + mask.int())
    _, _, _, info = env.step(_policy(env))
    assert not bool(info['autoreset'].any())
    assert bool((env.steps[mask] == 1).all()) and torch.equal(env.episodes[mask], ep[mask] + 1)
    # a caller may set done to have the next step start new episodes; reset_from_spawn_pool clears it
    env.done.fill_(1)
    env.reset_from_spawn_pool(np.random.RandomState(9))
    assert not bool(env.done.any())
    ep = env.episodes.clone()
    env.step(_policy(env))
    assert bool((env.steps == 1).all()) and torch.equal(env.episodes, ep)
    env.done.zero_()
    env.done[:10] = 1
    _, _, _, info = env.step(_policy(env))
    assert info['autoreset'].nonzero().reshape(-1).tolist() == list(range(10))
    assert torch.equal(env.episodes[:10], ep[:10] + 1)


def _pinned(env):
    return (torch.empty(env.B, 2).pin_memory(), torch.empty(env.B, env.obs_dim, dtype=env.obs_dtype).pin_memory(),
            torch.empty(env.B).pin_memory(), torch.empty(env.B, dtype=torch.uint8).pin_memory())


@pytest.mark.parametrize('dtype', [torch.float32, torch.float16])
def test_step_host_matches_the_device_step(world, dtype):
    B = 1024
    a = _env(world, B, 'next_step', max_episode_steps=7, obs_dtype=dtype)
    b = _env(world, B, 'next_step', max_episode_steps=7, obs_dtype=dtype)
    act_h, obs_h, rew_h, done_h = _pinned(b)
    resets = 0
    for t in range(25):
        act = _policy(a)
        o, r, d, info = a.step(act)
        act_h.copy_(act)
        b.step_host(act_h, obs_h, rew_h, done_h)
        assert torch.equal(_bits(obs_h), _bits(o.cpu())) and torch.equal(rew_h, r.cpu()) and torch.equal(done_h, d.cpu()), t
        resets += int(info['autoreset'].sum())
    assert resets > 0
    assert torch.equal(_bits(b.state), _bits(a.state)) and torch.equal(b.episodes, a.episodes)


@pytest.mark.parametrize('groups', [2, 4])
def test_rollout_host_matches_the_device_step(world, groups):
    """navgym_host_rollout with the built-in action-bank policy over a next-step env."""
    from nav_gym_b200 import _lib
    B, K, rows_n = 1024, 37, 8
    g = torch.Generator(device='cuda')
    g.manual_seed(3)
    bank = torch.rand(rows_n, B, 2, device='cuda', generator=g) * torch.tensor([0.5, 1.28], device='cuda') \
        + torch.tensor([0, -0.64], device='cuda')
    a = _env(world, B, 'next_step', max_episode_steps=9)
    b = _env(world, B, 'next_step', max_episode_steps=9)
    for s in range(K):
        a.step(bank[s % rows_n])
    torch.cuda.synchronize()
    act_h = bank.cpu().pin_memory()
    cur, obs_h, rew_h, done_h = _pinned(b)
    b.host_groups(groups, cur, obs_h, rew_h, done_h)
    ab = _lib.ActionBank(C.c_void_p(act_h.data_ptr()), rows_n, B)
    b.rollout_host(K, C.cast(_lib.load().navgym_policy_action_bank, _lib.POLICY_FN), ab)
    assert torch.equal(_bits(obs_h), _bits(a.obs.cpu())) and torch.equal(rew_h, a.reward.cpu())
    assert torch.equal(done_h, a.done.cpu()) and torch.equal(_bits(b.state), _bits(a.state))
    assert torch.equal(b.steps, a.steps) and torch.equal(b.episodes, a.episodes)
    assert int(a.episodes.sum()) > 2 * B   # every env ended episodes and started new ones


def test_two_env_offset_shards_equal_the_single_batch(world):
    from nav_gym_b200.batched_env import BatchedNavGym
    _, mp, _ = world
    B, H = 1024, 512
    rng = np.random.RandomState(13)
    map_id = rng.randint(0, 2, B).astype(np.int32)
    rows = np.concatenate([mp.spawn_arrays[i][rng.randint(len(mp.spawn_arrays[i]), size=1)] for i in map_id])
    noise_std = rng.uniform(0, 0.05, B).astype(np.float32)
    kw = dict(seed=17, auto_reset='next_step', max_episode_steps=10, resample_map=True, record_hits=True)
    full = BatchedNavGym(B, mp, map_id=map_id, **kw)
    shards = [BatchedNavGym(H, mp, map_id=map_id[s * H:(s + 1) * H], env_offset=s * H, **kw) for s in range(2)]
    full.set_state(rows[:, 0:2], rows[:, 2:4], rows[:, 4], noise_std=noise_std)
    full.reset()
    for s, e in enumerate(shards):
        sl = slice(s * H, (s + 1) * H)
        e.set_state(rows[sl, 0:2], rows[sl, 2:4], rows[sl, 4], noise_std=noise_std[sl])
        e.reset()
    resets = 0
    for _ in range(40):
        act = _policy(full)
        _, _, _, info = full.step(act)
        resets += int(info['autoreset'].sum())
        for s, e in enumerate(shards):
            e.step(act[s * H:(s + 1) * H].contiguous())
    assert resets > 0
    for s, e in enumerate(shards):
        sl = slice(s * H, (s + 1) * H)
        assert torch.equal(_bits(full.obs[sl]), _bits(e.obs)), s
        assert torch.equal(_bits(full.state[:, sl]), _bits(e.state)), s
        for n in ('tail64', 'steps', 'episodes', 'map_id', 'noise_std', 'hits') + OUTPUTS:
            assert torch.equal(_bits(getattr(full, n)[sl]), _bits(getattr(e, n))), (s, n)


def test_reset_scan_sees_the_scripted_pedestrians_of_its_launch(world):
    """With scripted pedestrians the reset launch scans the new pose against the geometry emitted
    for that launch (the walkers advanced one step), as the oracle does."""
    from oracle import oracle as orc
    ms, _, bank = world
    B, P = 256, 4
    env = _env(world, B, 'next_step', max_episode_steps=5, scan_noise_std_range=(0.0, 0.0))
    rng = np.random.RandomState(7)
    rows = bank[rng.randint(len(bank), size=(B, P))].copy()
    pos = env.state[:2].T.cpu().numpy().astype(np.float32)
    rows[..., 0:2] = pos[:, None, :] + rng.uniform(-3, 3, (B, P, 2)).astype(np.float32)
    rows[..., 4:6] = rows[..., 0:2]
    env.attach_pedestrians(rows)
    env.reset()
    checked = 0
    for t in range(12):
        _, _, _, info = env.step(_policy(env))
        geo = [x.clone() for x in (env._pdiscs, env._pnd, env._psegs, env._pns)]
        torch.cuda.synchronize()
        for e in info['autoreset'].nonzero().reshape(-1).tolist()[:6]:
            st = env.state[:, e].cpu().numpy()
            mid = int(env.map_id[e])
            ob = orc.OracleBatch(ms, np.array([mid], np.int32), st[None, :2], st[None, 3:5], st[None, 2:3],
                                 max_disc=env.max_disc, max_seg=env.max_seg)
            ob.reset_obs(*[x[e][None].cpu().numpy() for x in geo])
            assert np.array_equal(ob.obs[0, :NB], env.obs[e, :NB].cpu().numpy()), (t, e)
            checked += 1
    assert checked >= 6


def test_bad_modes_are_rejected(world):
    from nav_gym_b200.batched_env import BatchedNavGym
    from nav_gym_b200.pedestrians import PedestrianSim
    _, mp, _ = world
    with pytest.raises(ValueError):
        BatchedNavGym(8, mp, auto_reset='bogus')
    assert BatchedNavGym(8, mp, auto_reset=2).args.auto_reset == 1   # a truthy non-string is same-step
    env = BatchedNavGym(8, mp, auto_reset='next_step')
    with pytest.raises(ValueError):
        PedestrianSim(env, 2)
    assert env.peds is None   # rejected before it attached anything
