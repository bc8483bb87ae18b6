"""Soak: many steps of the robot batch and of the policy-driven crowd; checks that nothing
drifts into NaN / out-of-range values and that episode statistics stay sane."""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch
from nav_gym_b200.batched_env import BatchedNavGym, MapPool, filter_spawn_pool
from nav_gym_b200.pedestrians import PedestrianSim
from bench import build_world
m, pool = build_world(0, 65536)
pool = filter_spawn_pool(m, pool, 'cuda:0')
mp = MapPool([m], 'cuda:0', spawn_pools=[pool])
g = torch.Generator(device='cuda'); g.manual_seed(0)
def acts(B): return torch.rand(B, 2, device='cuda', generator=g) * torch.tensor([0.5, 1.28], device='cuda') + torch.tensor([0, -0.64], device='cuda')

B = 4096
env = BatchedNavGym(B, mp, seed=1, auto_reset=True, max_episode_steps=500)
env.reset_from_spawn_pool(np.random.RandomState(1))
n_steps = int(sys.argv[1]) if len(sys.argv) > 1 else 20000
done = succ = crash = trunc = 0
t0 = time.time()
for t in range(n_steps):
    env.step(acts(B))
    if t % 500 == 499:
        torch.cuda.synchronize()
        assert torch.isfinite(env.obs).all() and torch.isfinite(env.state).all() and torch.isfinite(env.reward).all()
        assert float(env.obs[:, :512].max()) < 25.3 and float(env.obs[:, :512].min()) > -0.3   # 25 m + noise
        assert int(env.steps.max()) <= 500
    done += int(env.done.sum()); succ += int(env.is_success.sum()); crash += int(env.is_crash.sum()); trunc += int(env.truncated.sum())
torch.cuda.synchronize()
print('robot batch: %d steps x %d envs in %.1f s; episodes ended %d (success %d, crash %d, truncated %d)' % (n_steps, B, time.time() - t0, done, succ, crash, trunc))

B, P = 1024, 8
env = BatchedNavGym(B, mp, seed=2, auto_reset=True)
env.reset_from_spawn_pool(np.random.RandomState(2))
sim = PedestrianSim(env, P, seed=2)
t0 = time.time()
eps = 0
for t in range(n_steps // 10):
    sim.step(acts(B))
    eps += int(env.done.sum())
    if t % 200 == 199:
        torch.cuda.synchronize()
        assert torch.isfinite(sim.pose).all() and torch.isfinite(sim.scan).all() and torch.isfinite(env.obs).all()
        assert float(sim.scan.max()) <= 6.0 and float(sim.scan.min()) >= 0.0
        sp = (sim.vel.norm(dim=-1) / sim.v_pref.clamp(min=1e-9))
        assert float(sp.max()) <= 1.0 + 1e-6                       # never faster than the preferred speed
torch.cuda.synchronize()
print('crowd: %d steps x %d envs x %d pedestrians in %.1f s; robot episodes ended %d; pedestrians within the map: %.3f' % (
    n_steps // 10, B, P, time.time() - t0, eps,
    float(((sim.pose[..., 0] > 0) & (sim.pose[..., 0] < 50) & (sim.pose[..., 1] > 0) & (sim.pose[..., 1] < 50)).float().mean())))
