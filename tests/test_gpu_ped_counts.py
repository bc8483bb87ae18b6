"""GPU: per-episode pedestrian counts (PedestrianSim(..., num_humans_range=(lo, hi))).

NavGym-v0 draws each episode's number of pedestrians uniformly from [5, 15].  With a range the sim
draws every episode's count on the device (navgym_peds_plan), at reset(), with each auto-reset and
with each reset_envs().  Checked here: a range (k, k) is the fixed count k bit for bit; the counts are
uniform, vary from episode to episode and do not depend on env_offset sharding; a respawned
environment adopts exactly the drawn count (slots beyond it untouched, including environments whose
slots straddle two CTAs of the planning kernel); the first scan of a new episode sees exactly the
new pedestrians; the masked reset equals auto-reset; bad arguments are rejected."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
NB = 512
STATE = ('pose', 'vel', 'v_pref', 'has_legs', 'dist_travelled', 'prev_action', 'goal_id', 'waypoint', 'goal_local',
         'scan')


@pytest.fixture(scope='module')
def outdoor():
    """Two outdoor maps with 30 boxes each and spawn pools of short episodes (resample_map;
    successes, crashes and truncations all happen within a few dozen steps)."""
    from nav_gym_b200 import maps
    from nav_gym_b200.batched_env import MapPool, filter_spawn_pool
    rng = np.random.RandomState(41)
    ms, pools = [], []
    for _ in range(2):
        m = maps.create_outdoor_map(30, 1.5, rng)
        pools.append(filter_spawn_pool(m, maps.spawn_pool(m, 4096, rng, min_goal_dist=1.5, max_goal_dist=6)))
        ms.append(m)
    return ms, MapPool(ms, 'cuda:0', spawn_pools=pools)


@pytest.fixture(scope='module')
def indoor():
    """One indoor map (the oracle's reset scan takes a single map)."""
    from nav_gym_b200 import maps
    from nav_gym_b200.batched_env import MapPool, filter_spawn_pool
    rng = np.random.RandomState(3)
    m = maps.create_indoor_map(3, 100, rng)
    pool = filter_spawn_pool(m, maps.spawn_pool(m, 2048, rng), 'cuda:0')
    return [m], MapPool([m], 'cuda:0', spawn_pools=[pool])


@pytest.fixture(scope='module')
def policy():
    from nav_gym_b200.pedestrians import HumanPolicy
    torch.manual_seed(0)
    return HumanPolicy()


def _env(world, B, auto_reset=True, seed=3, env_offset=0, map_id=None, **kw):
    from nav_gym_b200.batched_env import BatchedNavGym
    ms, mp = world
    if map_id is None:
        map_id = np.random.RandomState(seed).randint(0, len(ms), B).astype(np.int32)
    env = BatchedNavGym(B, mp, map_id=map_id, seed=seed, auto_reset=auto_reset, env_offset=env_offset,
                        record_hits=True, **kw)
    env.reset_from_spawn_pool(np.random.RandomState(seed + 1))
    return env


def _bits(t):
    return t.view({torch.float64: torch.int64, torch.float32: torch.int32}[t.dtype]) if t.is_floating_point() else t


def _actions(env, g, noise=0.3):
    """Half the environments head for their goal (successes), the other half drive at random
    (crashes)."""
    from nav_gym_b200 import _lib
    st = env.state
    bearing = torch.atan2(st[_lib.S_GY] - st[_lib.S_PY], st[_lib.S_GX] - st[_lib.S_PX]) - st[_lib.S_TH]
    err = torch.remainder(bearing + np.pi, 2 * np.pi) - np.pi
    w = (1.5 * err).float() + noise * torch.randn(env.B, device='cuda', generator=g)
    v = 0.3 + 0.2 * torch.rand(env.B, device='cuda', generator=g)
    rnd = torch.rand(env.B, 2, device='cuda', generator=g) * torch.tensor([0.5, 1.28], device='cuda') \
        - torch.tensor([0.0, 0.64], device='cuda')
    seek = torch.stack([v, w.clamp(-0.64, 0.64)], dim=1)
    half = (torch.arange(env.B, device='cuda') % 2 == 0)[:, None]
    return torch.where(half, seek, rnd).contiguous()


def test_a_range_of_one_value_is_the_fixed_count(outdoor, policy):
    """num_humans_range=(k, k) against nped=[k] * B: the count draw takes a Philox counter of its
    own, so every other draw and therefore the whole run is the same, bit for bit, through
    successes, crashes, truncations and resampled maps."""
    from nav_gym_b200.pedestrians import PedestrianSim
    B, P, k = 512, 8, 5
    kw = dict(max_episode_steps=30, resample_map=True)
    a = _env(outdoor, B, **kw)
    b = _env(outdoor, B, **kw)
    sa = PedestrianSim(a, P, nped=[k] * B, policy=policy, seed=5)
    sb = PedestrianSim(b, P, num_humans_range=(k, k), policy=policy, seed=5)
    map0 = a.map_id.clone()
    g = torch.Generator(device='cuda')
    g.manual_seed(2)
    n_succ = n_crash = n_trunc = 0
    for t in range(64):
        act = _actions(a, g)
        sa.step(act)
        sb.step(act)
        assert torch.equal(_bits(a.obs), _bits(b.obs)), t
        for name in ('reward', 'done', 'is_success', 'is_crash', 'truncated', 'state', 'map_id'):
            assert torch.equal(_bits(getattr(a, name)), _bits(getattr(b, name))), (t, name)
        for name in STATE:
            assert torch.equal(_bits(getattr(sa, name)), _bits(getattr(sb, name))), (t, name)
        assert torch.equal(a.nped, b.nped) and torch.equal(sb.cand_nped, b.nped), t
        n_succ += int(a.is_success.sum())
        n_crash += int(a.is_crash.sum())
        n_trunc += int(a.truncated.sum())
    assert b.nped.data_ptr() == sb.nped.data_ptr() and bool((b.nped == k).all())
    assert n_succ > 0 and n_crash > 0 and n_trunc > 0, (n_succ, n_crash, n_trunc)
    assert bool((a.map_id != map0).any())


def test_counts_are_uniform_vary_and_do_not_depend_on_sharding(outdoor, policy):
    """Counts collected through repeated reset_envs(all) and through auto-reset are uniform on
    lo..hi (chi-square), one environment's successive episodes do not all get the same count, and
    two env_offset shards of half the batch draw the full batch's counts."""
    from scipy import stats
    from nav_gym_b200.pedestrians import PedestrianSim
    B, H, P, lo, hi = 1024, 512, 15, 5, 15
    map_id = np.random.RandomState(7).randint(0, 2, B).astype(np.int32)
    env = _env(outdoor, B, map_id=map_id, max_episode_steps=4)
    sim = PedestrianSim(env, P, num_humans_range=(lo, hi), policy=policy, seed=9)
    shards = []
    for s in range(2):
        e = _env(outdoor, H, env_offset=s * H, map_id=map_id[s * H:(s + 1) * H], max_episode_steps=4)
        shards.append((e, PedestrianSim(e, P, num_humans_range=(lo, hi), policy=policy, seed=9)))

    def same_as_shards():
        for s, (e, ss) in enumerate(shards):
            sl = slice(s * H, (s + 1) * H)
            assert torch.equal(sim.nped[sl], ss.nped) and torch.equal(sim.cand_nped[sl], ss.cand_nped), s

    same_as_shards()
    per_env = [sim.nped.cpu().numpy()]
    everyone = torch.ones(B, dtype=torch.bool, device='cuda')
    for _ in range(11):   # every environment starts a new episode at every act()
        sim.reset_envs(everyone)
        sim.act()
        for s, (e, ss) in enumerate(shards):
            ss.reset_envs(torch.ones(H, dtype=torch.bool, device='cuda'))
            ss.act()
        same_as_shards()
        per_env.append(sim.nped.cpu().numpy())
    per_env = np.stack(per_env)                      # [12 episodes, B]
    assert all(len(set(per_env[:, e])) > 1 for e in range(B))
    # auto-reset: the count an ended episode's environment adopts at the next act()
    g = torch.Generator(device='cuda')
    g.manual_seed(4)
    auto = []
    for t in range(60):
        ended = env.done.bool().clone()
        sim.act()
        if t > 0:
            auto.append(sim.nped[ended].cpu().numpy())
        env.step(_actions(env, g))
        sim.observe()
    auto = np.concatenate(auto)
    assert len(auto) >= 8000, len(auto)
    counts = np.concatenate([per_env.reshape(-1), auto])
    assert len(counts) >= 20000 and counts.min() >= lo and counts.max() <= hi
    freq = np.bincount(counts - lo, minlength=hi - lo + 1)
    assert stats.chisquare(freq).pvalue > 1e-3, freq
    assert stats.chisquare(np.bincount(auto - lo, minlength=hi - lo + 1)).pvalue > 1e-3


def test_a_respawned_environment_adopts_the_drawn_count(outdoor, policy):
    """15 slots per environment (a planning CTA of 128 threads holds 8.53 environments, so many
    environments straddle two CTAs): after an episode ends, the next act() sets nped[e] to the
    cand_nped[e] read before it; exactly the slots below it are simulated (moved from the adopted
    pose, action written), the emitted geometry holds 2 leg discs or 4 box segments for each of
    them, and the slots at or beyond it keep their state bit for bit.  Growing and shrinking
    transitions both occur."""
    from nav_gym_b200.pedestrians import PedestrianSim, human_set_vel
    B, P, lo, hi = 256, 15, 5, 15
    env = _env(outdoor, B, max_episode_steps=6)
    sim = PedestrianSim(env, P, num_humans_range=(lo, hi), policy=policy, seed=11)
    straddle = np.array([(P * e) // 128 != (P * e + P - 1) // 128 for e in range(B)])
    g = torch.Generator(device='cuda')
    g.manual_seed(6)
    grow = shrink = straddled = 0
    slot = torch.arange(P, device='cuda')
    for t in range(40):
        ended = env.done.bool().clone()
        before = {k: getattr(sim, k).clone() for k in STATE}
        nped0, cand = sim.nped.clone(), sim.cand_nped.clone()
        cand_pose, cand_vp = sim.cand_pose.clone(), sim.cand_v_pref.clone()
        sim.act()
        want = torch.where(ended, cand, nped0)
        assert torch.equal(sim.nped, want), t
        live = slot[None, :] < sim.nped[:, None]              # [B, P]
        dead = ~live
        for k in STATE:
            assert torch.equal(_bits(getattr(sim, k)[dead]), _bits(before[k][dead])), (t, k)
        # the live slots were simulated: moved from the (adopted) pose with the clipped policy mean
        clipped = torch.stack([sim._mean[..., 0].clamp(0, 1), sim._mean[..., 1].clamp(-1, 1)], -1)
        assert torch.equal(sim.prev_action[live], clipped[live]), t
        pose0 = torch.where(ended[:, None, None], cand_pose, before['pose'])
        vp = torch.where(ended[:, None], cand_vp, before['v_pref'])
        assert torch.equal(sim.v_pref[live], vp[live]), t
        pose1, _ = human_set_vel(pose0, sim.prev_action.double() * vp[..., None], env.args.dt)
        assert torch.allclose(pose1[live], sim.pose[live], rtol=0, atol=1e-12), t
        # the geometry the robot's lidar sees: 2 leg discs per legged pedestrian, 4 segments otherwise
        legs = (sim.has_legs & live).sum(1)
        assert torch.equal(env._pnd.long(), 2 * legs) and torch.equal(env._pns.long(), 4 * (sim.nped.long() - legs)), t
        e_end = ended.cpu().numpy()
        n_new, n_old = sim.nped.cpu().numpy(), nped0.cpu().numpy()
        grow += int((e_end & (n_new > n_old)).sum())
        shrink += int((e_end & (n_new < n_old)).sum())
        straddled += int((e_end & straddle & (n_new != n_old)).sum())
        env.step(_actions(env, g))
        sim.observe()
        assert torch.equal(_bits(sim.scan[dead]), _bits(before['scan'][dead])), t
    assert grow > 20 and shrink > 20 and straddled > 10, (grow, shrink, straddled)


def test_the_first_scan_of_a_new_episode_sees_the_drawn_count(indoor, policy):
    """The robot's first observation after an auto-reset equals the oracle's reset scan of the new
    pose against the candidate geometry, and that geometry holds exactly cand_nped[e] pedestrians."""
    from oracle import oracle as orc
    from nav_gym_b200.pedestrians import PedestrianSim
    ms, mp = indoor
    m = ms[0]
    B, P, lo, hi = 256, 15, 5, 15
    env = _env(indoor, B, max_episode_steps=10)
    sim = PedestrianSim(env, P, num_humans_range=(lo, hi), policy=policy, seed=4)
    env.args.noise_lo = env.args.noise_hi = 0.0
    env.noise_std.zero_()
    dist = orc.edt(np.asarray(m['data']) >= 0.1)
    g = torch.Generator(device='cuda')
    g.manual_seed(1)
    slot = torch.arange(P, device='cuda')
    checked, counts = 0, set()
    for t in range(40):
        act = torch.rand(B, 2, device='cuda', generator=g) * torch.tensor([0.5, 1.28], device='cuda') \
            - torch.tensor([0.0, 0.64], device='cuda')
        sim.act()
        cn = sim.cand_nped.clone()
        cd, cnd = sim.cand_discs.clone(), sim.cand_nd.clone()
        cs, cns = sim.cand_segs.clone(), sim.cand_ns.clone()
        legs = (sim.cand_legs & (slot[None, :] < cn[:, None])).sum(1)
        assert torch.equal(cnd.long(), 2 * legs) and torch.equal(cns.long(), 4 * (cn.long() - legs)), t
        env.step(act)
        sim.observe()
        done = env.done.bool().cpu().numpy()
        if t < 1:
            continue   # (noise of the episodes that started before it was switched off)
        for e in np.where(done)[0][:3]:
            st = env.state[:, e].cpu().numpy()
            ob = orc.OracleBatch([m], np.zeros(1, np.int32), st[None, 0:2], st[None, 3:5], st[None, 2:3],
                                 max_disc=env.max_disc, max_seg=env.max_seg)
            ob.reset_obs(cd[e][None].cpu().numpy(), cnd[e][None].cpu().numpy(), cs[e][None].cpu().numpy(),
                         cns[e][None].cpu().numpy())
            assert np.array_equal(ob.obs[0, :NB], env.obs[e, :NB].cpu().numpy()), (t, e)
            counts.add(int(cn[e]))
            checked += 1
        if done.any():   # the next act() adopts exactly that count
            nd = torch.from_numpy(done).cuda()
            sim.act()
            assert torch.equal(sim.nped[nd], cn[nd]), t
            env.step(act)
            sim.observe()
    assert checked >= 6 and len(counts) >= 3, (checked, counts)


def test_masked_reset_equals_auto_reset_with_a_range(indoor, policy):
    """A sim over an auto_reset=False env calling sim.reset_envs(env.done) after every step against
    one over an auto_reset=True env, both drawing counts: every buffer, the counts included, is
    identical at every step."""
    from nav_gym_b200.pedestrians import PedestrianSim
    B, P = 64, 7
    pairs = []
    for auto_reset in (True, False):
        env = _env(indoor, B, auto_reset=auto_reset, seed=0, max_episode_steps=8)
        pairs.append((env, PedestrianSim(env, P, num_humans_range=(1, 7), policy=policy, seed=0)))
    (a, sa), (b, sb) = pairs
    g = torch.Generator(device='cuda')
    g.manual_seed(1)
    ended = 0
    for t in range(40):
        act = _actions(a, g)
        sa.step(act)
        sb.step(act)
        ended += int(b.done.sum())
        sb.reset_envs(b.done)
        assert torch.equal(_bits(a.obs), _bits(b.obs)), t
        for name in ('reward', 'done', 'is_success', 'is_crash', 'truncated', 'distance', 'state', 'tail64',
                     'steps', 'episodes', 'map_id', 'noise_std', 'hits'):
            assert torch.equal(_bits(getattr(a, name)), _bits(getattr(b, name))), (t, name)
        for name in STATE + ('nped', 'cand_nped', 'cand_pose', 'cand_discs', 'cand_nd', 'cand_segs', 'cand_ns'):
            assert torch.equal(_bits(getattr(sa, name)), _bits(getattr(sb, name))), (t, name)
        assert torch.equal(a._pnd, b._pnd) and torch.equal(a._pns, b._pns), t
    assert ended > 0
    assert len(set(sa.nped.cpu().tolist())) > 1


def test_export_env_lists_the_current_count(indoor, policy):
    from nav_gym_b200.pedestrians import PedestrianSim
    env = _env(indoor, 16)
    sim = PedestrianSim(env, 9, num_humans_range=(0, 9), policy=policy, seed=2)
    n = sim.nped.cpu().numpy()
    for i in range(16):
        assert len(env.export_env(i).humans) == n[i]
    assert len(set(n.tolist())) > 1


def test_bad_ranges_are_rejected_before_anything_is_attached(indoor, policy):
    from nav_gym_b200.pedestrians import PedestrianSim
    env = _env(indoor, 8)
    for kw in (dict(num_humans_range=(-1, 3)), dict(num_humans_range=(4, 3)), dict(num_humans_range=(2, 7)),
               dict(num_humans_range=(2, 5), nped=[3] * 8)):
        with pytest.raises(ValueError):
            PedestrianSim(env, 6, policy=policy, **kw)
        assert env.peds is None and getattr(env, 'crowd', None) is None, kw
