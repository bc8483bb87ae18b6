"""GPU: the masked device reset (BatchedNavGym.reset_envs, PedestrianSim.reset_envs,
navgym_reset_envs).

The defining property: an auto_reset=False env that calls reset_envs(done) after every step is, bit
for bit, the auto_reset=True env of the same seed, spawns and actions -- while the caller gets to
read each ended episode's final observation in between.  Also: unmasked environments and the step
outputs are not touched, the result does not depend on how the masked set is split (calls, bool
mask or ids, env_offset shards), PedestrianSim follows the same rule, and malformed input is
rejected."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
NB = 512
PAD = -12345   # int16 sentinel written into the float16 padding halves before the first reset


@pytest.fixture(scope='module')
def world():
    """Two outdoor maps with spawn pools (for resample_map) and a bank of scripted pedestrians."""
    from nav_gym_b200 import maps, worlds
    from nav_gym_b200.batched_env import MapPool, filter_spawn_pool
    rng = np.random.RandomState(41)
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


OUTPUTS = ('reward', 'done', 'is_success', 'is_crash', 'truncated', 'distance')
STATE = ('state', 'tail64', 'steps', 'episodes', 'map_id', 'noise_std', 'hits')


def _same(a, b, tag, names=OUTPUTS + STATE, obs=True):
    if obs:
        assert torch.equal(_bits(a.obs), _bits(b.obs)), tag + ' obs'
    for name in names:
        x, y = getattr(a, name), getattr(b, name)
        if x is not None or y is not None:
            assert torch.equal(_bits(x), _bits(y)), tag + ' ' + name


def _env(world, B, auto_reset, S=1, dtype=torch.float32, seed=3, peds=True, spawn_seed=None, **kw):
    """An env on the two-map pool, random start maps, spawns from the pools, and (peds=True) four
    scripted pedestrians per env, half of them within 4 m of the robot so that scans see them and
    crashes occur.  Two calls with the same arguments but auto_reset build the same env."""
    from nav_gym_b200.batched_env import BatchedNavGym
    _, mp, bank = world
    map_id = np.random.RandomState(seed).randint(0, 2, B).astype(np.int32)
    e = BatchedNavGym(B, mp, map_id=map_id, seed=seed, auto_reset=auto_reset, num_scan_stack=S, record_hits=True,
                      obs_dtype=dtype, **kw)
    if dtype == torch.float16:
        _bits(e.obs[:, S * NB + 14:]).fill_(PAD)
    e.reset_from_spawn_pool(np.random.RandomState(seed + 1 if spawn_seed is None else spawn_seed))
    if peds:
        P = 4
        rng = np.random.RandomState(seed + 2)
        rows = bank[rng.randint(len(bank), size=(B, P))].copy()
        pos = e.state[:2].T.cpu().numpy().astype(np.float32)
        near = rng.rand(B, P) < 0.5
        rows[..., 0:2] = np.where(near[..., None], pos[:, None, :] + rng.uniform(-4, 4, (B, P, 2)).astype(np.float32),
                                  rows[..., 0:2])
        rows[..., 4:6] = rows[..., 0:2]
        e.attach_pedestrians(rows)
        e.reset()
    return e


def _seek(env, g, noise=0.3):
    """Actions that head for the goal (plus noise), so that episodes end in success inside a short run."""
    from nav_gym_b200 import _lib
    st = env.state
    bearing = torch.atan2(st[_lib.S_GY] - st[_lib.S_PY], st[_lib.S_GX] - st[_lib.S_PX]) - st[_lib.S_TH]
    err = torch.remainder(bearing + np.pi, 2 * np.pi) - np.pi
    w = (1.5 * err).float() + noise * torch.randn(env.B, device='cuda', generator=g)
    v = 0.3 + 0.2 * torch.rand(env.B, device='cuda', generator=g)
    return torch.stack([v, w.clamp(-0.64, 0.64)], dim=1).contiguous()


@pytest.mark.parametrize('B', [777, 6144])
@pytest.mark.parametrize('S', [1, 3])
@pytest.mark.parametrize('dtype', [torch.float32, torch.float16])
def test_reset_envs_after_every_step_equals_auto_reset(world, B, S, dtype):
    """60 steps with Philox noise, scripted pedestrians (legs + boxes), max_episode_steps and
    resample_map on the two-map pool: successes, crashes and truncations all end episodes.  777
    and 6144 environments run the COOP and the non-COOP instantiations on a 148-SM part."""
    kw = dict(S=S, dtype=dtype, max_episode_steps=30, resample_map=True)
    a = _env(world, B, True, **kw)
    b = _env(world, B, False, **kw)
    _same(a, b, 'reset')
    map0 = a.map_id.clone()
    g = torch.Generator(device='cuda')
    g.manual_seed(B + S)
    n_crash = n_succ = n_trunc = 0
    for t in range(60):
        act = _seek(a, g)
        a.step(act)
        b.step(act)
        _same(a, b, 'step %d' % t, OUTPUTS, obs=False)   # b's rows of ended episodes: final observations
        final = b.obs.clone()
        b.reset_envs(b.done)
        _same(a, b, 'step %d + reset_envs' % t)
        keep = b.done == 0
        assert torch.equal(_bits(final[keep]), _bits(b.obs[keep])), t   # only the ended rows were rewritten
        n_crash += int(a.is_crash.sum())
        n_succ += int(a.is_success.sum())
        n_trunc += int(a.truncated.sum())
    assert n_crash > 0 and n_succ > 0 and n_trunc > 0, (n_crash, n_succ, n_trunc)
    assert bool((a.map_id != map0).any())   # resample_map drew other maps


def _snapshot(env):
    names = ('obs',) + OUTPUTS + STATE + ('sched',)
    return {n: getattr(env, n).clone() for n in names if getattr(env, n) is not None}


def _launch_order(env):
    """The env ids of the next step's launch order (the current third of the schedule buffer)."""
    from nav_gym_b200 import _lib
    nbk, B = _lib.SCHED_BUCKETS, env.B
    s = env.sched.cpu().numpy()
    cur = env.args.sched_phase
    cnt = s[cur * nbk:(cur + 1) * nbk]
    lists = s[3 * nbk:].reshape(3, nbk, B)[cur]
    return np.concatenate([lists[k, :cnt[k]] for k in range(nbk)])


@pytest.mark.parametrize('auto_reset', [False, True])
def test_reset_envs_touches_only_the_masked_environments(world, auto_reset):
    B = 777
    env = _env(world, B, auto_reset, max_episode_steps=30)
    g = torch.Generator(device='cuda')
    g.manual_seed(5)
    for _ in range(7):
        env.step(_seek(env, g))
        if not auto_reset:
            env.reset_envs(env.done)
    rng = np.random.RandomState(7)
    mask = torch.from_numpy(rng.rand(B) < 0.3).cuda()
    assert bool((env.steps[mask] > 0).any())   # environments in mid-episode are among them
    before = _snapshot(env)
    n0 = env.lib.navgym_launch_count()
    env.reset_envs(mask)
    assert env.lib.navgym_launch_count() == n0 + 1
    after = _snapshot(env)
    keep = ~mask
    for n in OUTPUTS + ('hits', 'sched'):
        assert torch.equal(_bits(before[n]), _bits(after[n])), n
    for n in ('obs', 'tail64', 'steps', 'episodes', 'map_id', 'noise_std'):
        assert torch.equal(_bits(before[n][keep]), _bits(after[n][keep])), n
    assert torch.equal(_bits(before['state'][:, keep]), _bits(after['state'][:, keep]))
    assert torch.equal(after['episodes'][mask], before['episodes'][mask] + 1)
    assert bool((after['steps'][mask] == 0).all())
    # the next step's launch order lists every environment exactly once, as does the one after
    assert np.array_equal(np.sort(_launch_order(env)), np.arange(B))
    env.step(_seek(env, g))
    assert np.array_equal(np.sort(_launch_order(env)), np.arange(B))
    # an all-zero mask changes nothing
    before = _snapshot(env)
    env.reset_envs(torch.zeros(B, dtype=torch.bool, device='cuda'))
    env.reset_envs([])
    after = _snapshot(env)
    for n in before:
        assert torch.equal(_bits(before[n]), _bits(after[n])), n


def test_reset_envs_does_not_depend_on_how_the_mask_is_split(world):
    B = 777
    envs = [_env(world, B, False, max_episode_steps=30, resample_map=True) for _ in range(3)]
    g = torch.Generator(device='cuda')
    g.manual_seed(9)
    for _ in range(9):
        act = _seek(envs[0], g)
        for e in envs:
            e.step(act)
            e.reset_envs(e.done)
    _same(envs[0], envs[1], 'before')
    rng = np.random.RandomState(11)
    m = torch.from_numpy(rng.rand(B) < 0.4).cuda()
    part = torch.from_numpy(rng.rand(B) < 0.5).cuda()
    envs[0].reset_envs(m)
    envs[1].reset_envs(m & part)
    envs[1].reset_envs(m & ~part)
    envs[2].reset_envs(torch.nonzero(m).reshape(-1).tolist())
    _same(envs[0], envs[1], 'M vs M & A, M - A')
    _same(envs[0], envs[2], 'bool mask vs ids')
    envs[1].reset_envs(torch.nonzero(m).reshape(-1).to(torch.int32))   # device id tensor
    envs[2].reset_envs(m.to(torch.uint8))
    _same(envs[1], envs[2], 'int32 ids vs uint8 mask')


def test_two_env_offset_shards_equal_the_single_batch(world):
    from nav_gym_b200.batched_env import BatchedNavGym
    _, mp, _ = world
    B, H = 1024, 512
    rng = np.random.RandomState(13)
    map_id = rng.randint(0, 2, B).astype(np.int32)
    rows = np.concatenate([mp.spawn_arrays[i][rng.randint(len(mp.spawn_arrays[i]), size=1)] for i in map_id])
    noise_std = rng.uniform(0, 0.05, B).astype(np.float32)
    kw = dict(seed=17, auto_reset=False, max_episode_steps=20, resample_map=True, record_hits=True)
    full = BatchedNavGym(B, mp, map_id=map_id, **kw)
    shards = [BatchedNavGym(H, mp, map_id=map_id[s * H:(s + 1) * H], env_offset=s * H, **kw) for s in range(2)]
    full.set_state(rows[:, 0:2], rows[:, 2:4], rows[:, 4], noise_std=noise_std)
    full.reset()
    for s, e in enumerate(shards):
        sl = slice(s * H, (s + 1) * H)
        e.set_state(rows[sl, 0:2], rows[sl, 2:4], rows[sl, 4], noise_std=noise_std[sl])
        e.reset()
    g = torch.Generator(device='cuda')
    g.manual_seed(19)
    ended = 0
    for _ in range(40):
        act = _seek(full, g)
        full.step(act)
        ended += int(full.done.sum())
        full.reset_envs(full.done)
        for s, e in enumerate(shards):
            e.step(act[s * H:(s + 1) * H].contiguous())
            e.reset_envs(e.done)
    assert ended > 0
    for s, e in enumerate(shards):
        sl = slice(s * H, (s + 1) * H)
        assert torch.equal(_bits(full.obs[sl]), _bits(e.obs)), s
        assert torch.equal(_bits(full.state[:, sl]), _bits(e.state)), s
        for n in ('tail64', 'steps', 'episodes', 'map_id', 'noise_std', 'hits') + OUTPUTS:
            assert torch.equal(_bits(getattr(full, n)[sl]), _bits(getattr(e, n))), (s, n)


def test_pedestrian_sim_reset_envs_equals_auto_reset():
    """A PedestrianSim over an auto_reset=True env against one over an auto_reset=False env that
    calls sim.reset_envs(env.done) after every step: the robots and the pedestrians stay identical."""
    from nav_gym_b200 import maps
    from nav_gym_b200.batched_env import BatchedNavGym, MapPool, filter_spawn_pool
    from nav_gym_b200.pedestrians import HumanPolicy, PedestrianSim
    rng = np.random.RandomState(3)
    m = maps.create_indoor_map(3, 100, rng)
    pool = filter_spawn_pool(m, maps.spawn_pool(m, 2048, rng), 'cuda:0')
    mp = MapPool([m], 'cuda:0', spawn_pools=[pool])
    torch.manual_seed(0)
    policy = HumanPolicy()
    B, P = 64, 6
    pairs = []
    for auto_reset in (True, False):
        env = BatchedNavGym(B, mp, seed=0, auto_reset=auto_reset, max_episode_steps=8, record_hits=True)
        env.reset_from_spawn_pool(np.random.RandomState(0))
        pairs.append((env, PedestrianSim(env, P, policy=policy, seed=0)))
    (a, sa), (b, sb) = pairs
    g = torch.Generator(device='cuda')
    g.manual_seed(1)
    ended = 0
    for t in range(40):
        act = _seek(a, g)
        sa.step(act)
        sb.step(act)
        ended += int(b.done.sum())
        sb.reset_envs(b.done)
        _same(a, b, 'crowd step %d' % t)
        for k in ('pose', 'vel', 'v_pref', 'has_legs', 'goal_id', 'waypoint', 'prev_action', 'scan', 'dist_travelled'):
            assert torch.equal(_bits(getattr(sa, k)), _bits(getattr(sb, k))), (t, k)
    assert ended > 0
    with pytest.raises(ValueError):   # the sim has to respawn its pedestrians too
        b.reset_envs(b.done)


def test_malformed_masks_are_rejected(world):
    from nav_gym_b200 import _lib
    B = 64
    env = _env(world, B, False, peds=False)
    for bad in (torch.zeros(B - 1, dtype=torch.bool, device='cuda'),   # wrong length
                torch.zeros(B, dtype=torch.bool),                      # on the host
                torch.zeros(B, dtype=torch.float32, device='cuda'),    # not a mask, not ids
                torch.zeros(2, B, dtype=torch.uint8, device='cuda'),
                [0, B], [-1], [[0, 1]], [0.5]):
        with pytest.raises(ValueError):
            env.reset_envs(bad)
    lib = _lib.load()
    mask = torch.ones(B, dtype=torch.uint8, device='cuda')
    torch.cuda.synchronize()
    assert lib.navgym_reset_envs(C.byref(env.args), None, env._stream()) == 1   # cudaErrorInvalidValue
    for field, value in (('env_begin', -1), ('env_begin', B + 1), ('env_count', B + 1), ('obs_format', 7)):
        args = _lib.StepArgs.from_buffer_copy(env.args)
        setattr(args, field, value)
        assert lib.navgym_reset_envs(C.byref(args), C.c_void_p(mask.data_ptr()), env._stream()) == 1, (field, value)
    args = _lib.StepArgs.from_buffer_copy(env.args)
    args.env_begin, args.env_count = 40, 30
    assert lib.navgym_reset_envs(C.byref(args), C.c_void_p(mask.data_ptr()), env._stream()) == 1
    h = _env(world, B, False, dtype=torch.float16, peds=False)
    args = _lib.StepArgs.from_buffer_copy(h.args)
    args.obs_stride = NB + 15   # odd float16 stride
    assert lib.navgym_reset_envs(C.byref(args), C.c_void_p(mask.data_ptr()), h._stream()) == 1
    args.num_envs = 0
    assert lib.navgym_reset_envs(C.byref(args), None, h._stream()) == 0   # nothing to do
    # a sub-range launch resets exactly that range
    before = env.episodes.clone()
    args = _lib.StepArgs.from_buffer_copy(env.args)
    args.env_begin, args.env_count = 10, 20
    assert lib.navgym_reset_envs(C.byref(args), C.c_void_p(mask.data_ptr()), env._stream()) == 0
    d = (env.episodes - before).cpu().numpy()
    assert d[10:30].tolist() == [1] * 20 and not d[:10].any() and not d[30:].any()
    env.step(torch.zeros(B, 2, device='cuda'))
    torch.cuda.synchronize()
