"""The host-buffer pipe against the device-resident step: a rejected submit or rollout leaves the
pipe's launch order as it was, and step_host under a PedestrianSim scans what env.step scans."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _pinned(*shape, dtype=torch.float32):
    return torch.empty(*shape, dtype=dtype).pin_memory()


def test_rejected_submit_and_rollout_leave_the_pipe_as_it_was():
    """An argument block with 200 + 200 obstacle slots (of 256) is rejected by the submit and by
    the rollout before anything is enqueued; the longest-first launch order of every group stays
    in step, so the groups keep giving the device-resident step's results bit for bit."""
    from nav_gym_b200 import _lib, maps
    from nav_gym_b200.batched_env import BatchedNavGym, MapPool, filter_spawn_pool
    lib = _lib.load()
    rng = np.random.RandomState(6)
    m = maps.create_outdoor_map(10, 0.7, rng)
    pool = filter_spawn_pool(m, maps.spawn_pool(m, 2048, rng, min_goal_dist=4, max_goal_dist=15))
    mp = MapPool([m], 'cuda:0', spawn_pools=[pool])
    B, T, K, rows_n = 1024, 12, 9, 4
    envs = [BatchedNavGym(B, mp, seed=3, auto_reset=True, longest_first=True) for _ in range(2)]
    for e in envs:
        e.reset_from_spawn_pool(np.random.RandomState(7))
    a, b = envs
    act_h, obs_h, rew_h, done_h = _pinned(B, 2), _pinned(B, 519), _pinned(B), _pinned(B, dtype=torch.uint8)
    bounds = b.host_groups(2, act_h, obs_h, rew_h, done_h)
    bad = _lib.StepArgs.from_buffer_copy(b.args)
    discs = torch.zeros(B, 200, 3, device='cuda')
    segs = torch.zeros(B, 200, 4, device='cuda')
    bad.max_disc = bad.max_seg = 200
    bad.discs, bad.segs = C.c_void_p(discs.data_ptr()), C.c_void_p(segs.data_ptr())
    pipe, p = b._pipe[0], b._host_ptrs

    acts = torch.from_numpy(rng.uniform([0.2, -0.64], [0.5, 0.64], (T, B, 2)).astype(np.float32))
    want = []
    for t in range(T):
        o, r, d, _ = a.step(acts[t].cuda())
        want.append((o.cpu().clone(), r.cpu().clone(), d.cpu().clone()))
    act_h.copy_(acts[0])
    for g in range(2):
        n = lib.navgym_launch_count()
        assert lib.navgym_step_batch_host_submit(pipe, C.byref(bad), g, *p) == 1   # cudaErrorInvalidValue
        assert lib.navgym_launch_count() == n
        b.submit_host(g)
    for t in range(T):
        for g, (b0, b1) in enumerate(bounds):
            b.wait_host(g)
            assert torch.equal(obs_h[b0:b1], want[t][0][b0:b1]), (t, g)
            assert torch.equal(rew_h[b0:b1], want[t][1][b0:b1]) and torch.equal(done_h[b0:b1], want[t][2][b0:b1]), (t, g)
            if t + 1 < T:
                act_h[b0:b1].copy_(acts[t + 1][b0:b1])
                if t == T // 2:
                    assert lib.navgym_step_batch_host_submit(pipe, C.byref(bad), g, *p) == 1
                b.submit_host(g)

    # the same through the rollout driver, with the action-bank policy
    gen = torch.Generator(device='cuda')
    gen.manual_seed(5)
    bank = torch.rand(rows_n, B, 2, device='cuda', generator=gen) * torch.tensor([0.5, 1.28], device='cuda') \
        + torch.tensor([0, -0.64], device='cuda')
    for s in range(K):
        a.step(bank[s % rows_n])
    torch.cuda.synchronize()
    bank_h = bank.cpu().pin_memory()
    ab = _lib.ActionBank(C.c_void_p(bank_h.data_ptr()), rows_n, B)
    policy = C.cast(lib.navgym_policy_action_bank, _lib.POLICY_FN)
    n = lib.navgym_launch_count()
    assert lib.navgym_host_rollout(pipe, C.byref(bad), K, C.cast(policy, C.c_void_p),
                                   C.cast(C.pointer(ab), C.c_void_p), *p) == 1
    assert lib.navgym_launch_count() == n
    b.rollout_host(K, policy, ab)
    assert torch.equal(obs_h, a.obs.cpu()) and torch.equal(rew_h, a.reward.cpu()) and torch.equal(done_h, a.done.cpu())
    assert torch.equal(b.state, a.state) and torch.equal(b.episodes, a.episodes)


def test_step_host_under_a_pedestrian_sim_equals_step():
    """A PedestrianSim moves its pedestrians itself: step_host only emits their geometry, as
    env.step does, so the robot scans the same pedestrians and both sims stay in step."""
    from nav_gym_b200 import _lib, maps
    from nav_gym_b200.batched_env import BatchedNavGym, MapPool, filter_spawn_pool
    from nav_gym_b200.pedestrians import HumanPolicy, PedestrianSim
    rng = np.random.RandomState(3)
    m = maps.create_indoor_map(3, 100, rng)
    pool = filter_spawn_pool(m, maps.spawn_pool(m, 2048, rng), 'cuda:0')
    mp = MapPool([m], 'cuda:0', spawn_pools=[pool])
    torch.manual_seed(0)
    policy = HumanPolicy()
    B, P = 64, 10
    twins = []
    for _ in range(2):
        env = BatchedNavGym(B, mp, seed=0, auto_reset=True)
        env.reset_from_spawn_pool(np.random.RandomState(0))
        twins.append((env, PedestrianSim(env, P, policy=policy, seed=0)))
    (env_a, sim_a), (env_b, sim_b) = twins
    robot = torch.stack([env_a.state[_lib.S_PX], env_a.state[_lib.S_PY]], dim=1)
    near = (sim_a.pose[..., :2] - robot[:, None, :]).norm(dim=2) < 10.0
    assert int(near.sum()) > B // 4, 'pedestrians within lidar range'
    obs_h, rew_h, done_h = _pinned(B, 519), _pinned(B), _pinned(B, dtype=torch.uint8)
    for t in range(8):
        act = torch.from_numpy(rng.uniform([0.2, -0.64], [0.5, 0.64], (B, 2)).astype(np.float32))
        sim_a.act()
        o, r, d, _ = env_a.step(act.cuda())
        sim_a.observe()
        sim_b.act()
        env_b.step_host(act.pin_memory(), obs_h, rew_h, done_h)
        sim_b.observe()
        torch.cuda.synchronize()
        assert torch.equal(obs_h, o.cpu()) and torch.equal(rew_h, r.cpu()) and torch.equal(done_h, d.cpu()), t
        assert torch.equal(sim_a.pose, sim_b.pose), t
