"""GPU: float16 observation rows (BatchedNavGym(obs_dtype=torch.float16), NAVGYM_OBS_F16).

Every test runs a float16 env next to a float32 env of the same seed on the same MapPool and
checks the defining property bit for bit: the float16 env's scans are the float32 env's scans
rounded to float16, its tail (float32 in the row) is the float32 env's tail, and every other
output and every piece of state are identical.  Host-buffer paths, the HER kernel, export_env and
PedestrianSim are checked over float16 rows the same way, and malformed rows are rejected."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
NB = 512
PAD = -12345   # int16 sentinel written into the padding halves before reset()


@pytest.fixture(scope='module')
def world():
    from nav_gym_b200 import maps, worlds
    from nav_gym_b200.batched_env import MapPool, filter_spawn_pool
    rng = np.random.RandomState(40)
    m = maps.create_outdoor_map(10, 0.7, rng)
    pool = filter_spawn_pool(m, maps.spawn_pool(m, 4096, rng, min_goal_dist=1.5, max_goal_dist=6))
    mp = MapPool([m], 'cuda:0', spawn_pools=[pool])
    bank = worlds.scripted_pedestrians(m, 1, 256, rng)[0]   # [256, 16] waypoint walkers
    return m, mp, bank


def _bits(t):
    return t.view({torch.float64: torch.int64, torch.float32: torch.int32, torch.float16: torch.int16}[t.dtype]) \
        if t.is_floating_point() else t


STATE = ('reward', 'done', 'is_success', 'is_crash', 'truncated', 'distance', 'state', 'tail64', 'steps',
         'episodes', 'map_id', 'noise_std', 'hits')


def _same(a, b, tag, pad=True):
    """a: float32 env, b: float16 env -- the defining property, bitwise."""
    n = a.num_scan_stack * NB
    assert tuple(b.obs.shape) == (a.B, n + 16) and b.obs.dtype == torch.float16
    scans, tail = b.obs_parts()
    assert torch.equal(_bits(scans), _bits(a.obs[:, :n].half())), tag + ' scans'
    assert torch.equal(_bits(tail), _bits(a.obs[:, n:])), tag + ' tail'
    if pad:
        assert bool((_bits(b.obs[:, n + 14:]) == PAD).all()), tag + ' padding'
    for name in STATE:
        x, y = getattr(a, name), getattr(b, name)
        if x is not None or y is not None:
            assert torch.equal(_bits(x), _bits(y)), tag + ' ' + name


def _pair(world, B, S=1, auto_reset=True, peds=True, seed=3, **kw):
    """A float32 and a float16 env, same seed, same spawns, same scripted pedestrians (half of them
    within 4 m of the robot, so that scans see them and crashes occur)."""
    from nav_gym_b200.batched_env import BatchedNavGym
    m, mp, bank = world
    envs = []
    for dt in (torch.float32, torch.float16):
        e = BatchedNavGym(B, mp, seed=seed, auto_reset=auto_reset, num_scan_stack=S, record_hits=True,
                          obs_dtype=dt, **kw)
        if dt == torch.float16:
            _bits(e.obs[:, S * NB + 14:]).fill_(PAD)
        e.reset_from_spawn_pool(np.random.RandomState(seed + 1))
        envs.append(e)
    if peds:
        P = 4
        rng = np.random.RandomState(seed + 2)
        rows = bank[rng.randint(len(bank), size=(B, P))].copy()
        pos = envs[0].state[:2].T.cpu().numpy().astype(np.float32)
        near = rng.rand(B, P) < 0.5
        rows[..., 0:2] = np.where(near[..., None], pos[:, None, :] + rng.uniform(-4, 4, (B, P, 2)).astype(np.float32),
                                  rows[..., 0:2])
        rows[..., 4:6] = rows[..., 0:2]
        for e in envs:
            e.attach_pedestrians(rows)
            e.reset()
    return envs


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
@pytest.mark.parametrize('auto_reset', [True, False])
def test_step_and_reset_match_float32_env(world, B, S, auto_reset):
    """60 steps with Philox noise, scripted pedestrians (legs + boxes) and max_episode_steps:
    auto-reset passes, successes and truncations with auto_reset, crash re-scans without.  777
    and 6144 environments run the COOP and the non-COOP instantiations on a 148-SM part."""
    a, b = _pair(world, B, S, auto_reset=auto_reset, max_episode_steps=30)
    _same(a, b, 'reset')
    episodes0 = int(a.episodes.sum())
    g = torch.Generator(device='cuda')
    g.manual_seed(B + S)
    n_crash = n_succ = n_trunc = 0
    for t in range(60):
        act = _seek(a, g)
        a.step(act)
        b.step(act)
        _same(a, b, 'step %d' % t)
        n_crash += int(a.is_crash.sum())
        n_succ += int(a.is_success.sum())
        n_trunc += int(a.truncated.sum())
    assert n_crash > 0 and n_succ > 0 and n_trunc > 0, (n_crash, n_succ, n_trunc)
    if auto_reset:
        assert int(a.episodes.sum()) > episodes0   # episodes ended and restarted in the kernel


def _pinned_rows(env):
    return (torch.empty(env.B, 2).pin_memory(), torch.empty(env.B, env.obs_dim, dtype=env.obs_dtype).pin_memory(),
            torch.empty(env.B).pin_memory(), torch.empty(env.B, dtype=torch.uint8).pin_memory())


def test_step_host_rows_match_device_rows(world):
    """navgym_step_batch_host with 1 and 3 chunks writes the float16 device rows to pinned float16 rows."""
    from nav_gym_b200.batched_env import BatchedNavGym
    m, mp, _ = world
    B = 1000
    envs = [BatchedNavGym(B, mp, seed=9, auto_reset=True, max_episode_steps=20, obs_dtype=torch.float16) for _ in range(2)]
    for e in envs:
        e.reset_from_spawn_pool(np.random.RandomState(5))
    _, obs_h, rew_h, done_h = _pinned_rows(envs[1])
    g = torch.Generator(device='cuda')
    g.manual_seed(4)
    n_done = 0
    for t in range(30):
        act = _seek(envs[0], g)
        o, r, d, _ = envs[0].step(act)
        torch.cuda.synchronize()
        envs[1].step_host(act.cpu().pin_memory(), obs_h, rew_h, done_h, chunks=1 if t % 2 else 3)
        assert torch.equal(_bits(o.cpu()), _bits(obs_h)) and torch.equal(r.cpu(), rew_h) and torch.equal(d.cpu(), done_h), t
        n_done += int(d.sum())
    assert n_done > 0
    assert torch.equal(envs[0].state, envs[1].state) and torch.equal(envs[0].episodes, envs[1].episodes)


def test_async_host_groups_rows_match_device_rows(world):
    """host_groups + submit_host / wait_host, 2 groups in flight, on float16 rows."""
    from nav_gym_b200.batched_env import BatchedNavGym
    m, mp, _ = world
    B = 777
    envs = [BatchedNavGym(B, mp, seed=3, auto_reset=True, num_scan_stack=3, obs_dtype=torch.float16) for _ in range(2)]
    for e in envs:
        e.reset_from_spawn_pool(np.random.RandomState(7))
    act_h, obs_h, rew_h, done_h = _pinned_rows(envs[1])
    bounds = envs[1].host_groups(2, act_h, obs_h, rew_h, done_h)
    T = 12
    g = torch.Generator(device='cuda')
    g.manual_seed(6)
    want, acts = [], []
    for t in range(T):
        acts.append(_seek(envs[0], g).cpu())
        o, r, d, _ = envs[0].step(acts[-1].cuda())
        want.append((o.cpu().clone(), r.cpu().clone(), d.cpu().clone()))
    act_h.copy_(acts[0])
    for grp in range(2):
        envs[1].submit_host(grp)
    for t in range(T):
        for grp, (b0, b1) in enumerate(bounds):
            envs[1].wait_host(grp)
            assert torch.equal(_bits(obs_h[b0:b1]), _bits(want[t][0][b0:b1])), (t, grp)
            assert torch.equal(rew_h[b0:b1], want[t][1][b0:b1]) and torch.equal(done_h[b0:b1], want[t][2][b0:b1])
            if t + 1 < T:
                act_h[b0:b1].copy_(acts[t + 1][b0:b1])
                envs[1].submit_host(grp)


def test_rollout_in_c_rows_match_device_rows(world):
    """navgym_host_rollout with the action-bank policy on float16 rows."""
    from nav_gym_b200 import _lib
    from nav_gym_b200.batched_env import BatchedNavGym
    m, mp, _ = world
    B, K, rows_n = 1024, 37, 8
    g = torch.Generator(device='cuda')
    g.manual_seed(3)
    bank = torch.rand(rows_n, B, 2, device='cuda', generator=g) * torch.tensor([0.5, 1.28], device='cuda') \
        + torch.tensor([0, -0.64], device='cuda')
    a, b = [BatchedNavGym(B, mp, seed=21, auto_reset=True, max_episode_steps=9, obs_dtype=torch.float16) for _ in range(2)]
    for e in (a, b):
        e.reset_from_spawn_pool(np.random.RandomState(8))
    for s in range(K):
        a.step(bank[s % rows_n])
    torch.cuda.synchronize()
    act_h = bank.cpu().pin_memory()
    cur, obs_h, rew_h, done_h = _pinned_rows(b)
    b.host_groups(3, cur, obs_h, rew_h, done_h)
    ab = _lib.ActionBank(C.c_void_p(act_h.data_ptr()), rows_n, B)
    b.rollout_host(K, C.cast(_lib.load().navgym_policy_action_bank, _lib.POLICY_FN), ab)
    assert torch.equal(_bits(obs_h), _bits(a.obs.cpu())) and torch.equal(rew_h, a.reward.cpu())
    assert torch.equal(done_h, a.done.cpu()) and torch.equal(b.state, a.state)
    assert torch.equal(b.episodes, a.episodes) and int(a.episodes.sum()) > B
    # the pinned rows split like the device rows
    scans, tail = b.obs_parts(obs_h)
    assert scans.shape == (B, NB) and tail.shape == (B, 7) and tail.dtype == torch.float32
    assert torch.equal(_bits(tail), _bits(b.obs_parts()[1].cpu()))


def _her_rows(world, S, steps=24, B=777):
    """float16 rows (and goals) of a run with pedestrians next to the robots, and the float16 env
    that produced them.  A returned observation rarely shows the crash itself (the step rolls back
    and re-scans), so every 7th row gets its scans scaled down (a crash) and every 7th goal is put
    next to the row's pose (a success)."""
    a, b = _pair(world, B, S, auto_reset=False, seed=11)
    from nav_gym_b200 import _lib
    g = torch.Generator(device='cuda')
    g.manual_seed(12)
    rows, goals = [], []
    for t in range(steps):
        act = _seek(a, g)
        a.step(act)
        b.step(act)
        rows.append(b.obs.clone())
        goals.append(torch.stack([b.state[_lib.S_GX], b.state[_lib.S_GY]], 1).float())
    rows, goals = torch.cat(rows), torch.cat(goals)
    scans, tail = b.obs_parts(rows)
    scans[0::7] *= 0.02
    goals[1::7] = tail[1::7, 2:4] + 0.1
    return b, rows, goals


@pytest.mark.parametrize('S', [1, 3])
def test_her_on_float16_rows_equals_float32_rows(world, S):
    """compute_rewards on float16 rows (contiguous and a strided slice of a wider buffer) equals,
    bit for bit in every output, compute_rewards on float32 rows rebuilt from them; row counts
    below and above one full wave of CTAs (148 SMs x 4 CTAs x 8 warps = 4736 rows)."""
    env, rows, goals = _her_rows(world, S)
    n = S * NB
    N = rows.shape[0]
    assert N > 4736
    wide = torch.zeros(N, n + 40, dtype=torch.float16, device='cuda')
    wide[:, :n + 16] = rows
    strided = wide[:, :n + 16]
    assert strided.stride(0) == n + 40
    scans, tail = env.obs_parts(rows)
    rows32 = torch.cat([scans.float(), tail], 1)
    seen = dict(crash=0, success=0, discomfort=0)
    for cnt in (1000, N):
        want = env.compute_rewards(rows32[:cnt], goals[:cnt])
        for r16 in (rows[:cnt], strided[:cnt]):
            got = env.compute_rewards(r16, goals[:cnt])
            for k in want:
                assert torch.equal(_bits(got[k]), _bits(want[k])), (cnt, k)
        seen['crash'] += int(want['is_crash'].sum())
        seen['success'] += int(want['is_success'].sum())
        # discomfort: a scan under the discomfort threshold in a row that did not crash
        newest = rows32[:cnt, (S - 1) * NB:S * NB]
        disc = (newest < env.dthr).any(1) & ~want['is_crash'].bool()
        seen['discomfort'] += int(disc.sum())
    assert min(seen.values()) > 0, seen


def test_export_env_matches_float32_env(world):
    """export_env of a float16 env: the float32 env's export, scan columns rounded to float16."""
    a, b = _pair(world, 256, S=3, auto_reset=True)
    g = torch.Generator(device='cuda')
    g.manual_seed(2)
    for t in range(8):
        act = _seek(a, g)
        a.step(act)
        b.step(act)
    torch.cuda.synchronize()
    n = 3 * NB
    for i in (0, 17, 255):
        x, y = a.export_env(i), b.export_env(i)
        ox, oy = x.prev_obs['observation'], y.prev_obs['observation']
        assert np.array_equal(oy[:n], ox[:n].astype(np.float16).astype(np.float64)), i
        assert np.array_equal(oy[n:], ox[n:]), i
        for k in ('achieved_goal', 'desired_goal'):
            assert np.array_equal(x.prev_obs[k], y.prev_obs[k]), (i, k)
        for k in ('reward', 'done', 'is_success', 'is_crash', 'truncated', 'distance', 'episode', 'noise_std',
                  'steps_since_reset', 'num_scan_stack'):
            assert getattr(x, k) == getattr(y, k), (i, k)
        for k in ('px', 'py', 'theta', 'gx', 'gy', 'v', 'r'):
            assert getattr(x.robot, k) == getattr(y.robot, k), (i, k)
        assert [(h.px, h.py, h.theta) for h in x.humans] == [(h.px, h.py, h.theta) for h in y.humans], i


def test_pedestrian_sim_over_float16_env():
    """PedestrianSim (policy-driven pedestrians) never reads the robot's row: over a float16 env it
    gives the float32 sim's results, and the robot's outputs keep the defining property."""
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
    for dt in (torch.float32, torch.float16):
        env = BatchedNavGym(B, mp, seed=0, auto_reset=True, record_hits=True, obs_dtype=dt)
        if dt == torch.float16:
            _bits(env.obs[:, NB + 14:]).fill_(PAD)
        env.reset_from_spawn_pool(np.random.RandomState(0))
        pairs.append((env, PedestrianSim(env, P, policy=policy, seed=0)))
    (a, sa), (b, sb) = pairs
    g = torch.Generator(device='cuda')
    g.manual_seed(1)
    for t in range(10):
        act = _seek(a, g)
        sa.step(act)
        sb.step(act)
        _same(a, b, 'crowd step %d' % t)
        for k in ('pose', 'vel', 'scan', 'prev_action', 'waypoint', 'goal_id'):
            assert torch.equal(_bits(getattr(sa, k)), _bits(getattr(sb, k))), (t, k)


def test_malformed_float16_rows_are_rejected(world):
    from nav_gym_b200 import _lib
    from nav_gym_b200.batched_env import BatchedNavGym
    m, mp, _ = world
    B = 64
    with pytest.raises(ValueError):
        BatchedNavGym(B, mp, obs_dtype=torch.bfloat16)
    env = BatchedNavGym(B, mp, seed=1, auto_reset=True, obs_dtype=torch.float16)
    env.reset_from_spawn_pool(np.random.RandomState(1))
    goals = torch.zeros(8, 2, device='cuda')
    rows = env.obs[:8]
    env.compute_rewards(rows, goals)   # well-formed
    buf = torch.zeros(8, NB + 17, dtype=torch.float16, device='cuda')
    with pytest.raises(RuntimeError):            # odd stride
        env.compute_rewards(buf[:, :NB + 16], goals)
    with pytest.raises(RuntimeError):            # too short for 512 scans + a float32 tail
        env.compute_rewards(torch.zeros(8, NB + 12, dtype=torch.float16, device='cuda'), goals)
    flat = torch.zeros(8 * (NB + 16) + 2, dtype=torch.float16, device='cuda')
    with pytest.raises(RuntimeError):            # row base not 4-byte aligned
        env.compute_rewards(flat.as_strided((8, NB + 16), (NB + 16, 1), 1), goals)
    # through the argument block: unknown format, odd stride, too short a stride
    lib = _lib.load()
    act = torch.zeros(B, 2, device='cuda')
    env._geom(None, None, None, None, None, act)
    torch.cuda.synchronize()
    for field, value in (('obs_format', 7), ('obs_stride', NB + 15), ('obs_stride', NB + 12)):
        args = _lib.StepArgs.from_buffer_copy(env.args)
        setattr(args, field, value)
        assert lib.navgym_step_batch(C.byref(args), env._stream()) == 1, (field, value)   # cudaErrorInvalidValue
        assert lib.navgym_reset_obs_batch(C.byref(args), env._stream()) == 1, (field, value)
    h = _lib.HerArgs()
    h.count, h.obs_stride, h.num_scan_stack, h.obs_format = 8, NB + 16, 1, 5
    h.obs, h.goals, h.thr, h.dthr = C.c_void_p(rows.data_ptr()), C.c_void_p(goals.data_ptr()), \
        C.c_void_p(env.thr.data_ptr()), C.c_void_p(env.dthr.data_ptr())
    assert lib.navgym_compute_rewards(C.byref(h), env._stream()) == 1
    # float32 host rows handed to a float16 env
    act_h, _, rew_h, done_h = _pinned_rows(env)
    obs32 = torch.empty(B, NB + 7).pin_memory()
    with pytest.raises(AssertionError):
        env.step_host(act_h, obs32, rew_h, done_h)
    with pytest.raises(AssertionError):
        env.host_groups(2, act_h, obs32, rew_h, done_h)
    # misaligned pinned host rows through the C entry point
    big = torch.empty(B * (NB + 16) + 2, dtype=torch.float16).pin_memory()
    env._make_pipe(1)
    assert lib.navgym_step_batch_host(env._pipe[0], C.byref(env.args), env._stream(), C.c_void_p(act_h.data_ptr()),
                                      C.c_void_p(big.data_ptr() + 2), C.c_void_p(rew_h.data_ptr()),
                                      C.c_void_p(done_h.data_ptr())) == 1
    # the env still steps after all of the above
    env.step(act)
    torch.cuda.synchronize()
