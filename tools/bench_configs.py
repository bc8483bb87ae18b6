"""Throughput of the policy-driven crowd (SURVEY 8f row 2): C2's world with the reference's
pedestrians (PedestrianSim).  The BASELINE configurations c3 / c4 / c5 are measured by bench.py
itself (its `configs` block).  Device-resident numbers (CUDA events, no L2 flush), one JSON line."""
import json, os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch
from nav_gym_b200 import maps, _lib
from nav_gym_b200.batched_env import BatchedNavGym, MapPool, filter_spawn_pool


def random_policy(B, dev, seed=0):
    g = torch.Generator(device=dev); g.manual_seed(seed)
    bank = torch.rand(32, B, 2, device=dev, generator=g) * torch.tensor([0.5, 1.28], device=dev) + torch.tensor([0, -0.64], device=dev)
    it = [0]
    def f(obs):
        it[0] += 1
        return bank[it[0] % 32]
    return f


def crowd(dev, steps, warmup, B=4096, P=10):
    """C2's world with the reference's policy-driven pedestrians (PedestrianSim): P pedestrians per
    env, each with its own 512-beam scan and a CNN policy forward per step (random-init weights)."""
    from bench import build_world
    from nav_gym_b200.pedestrians import PedestrianSim
    m, pool = build_world(0)
    mp = MapPool([m], dev, spawn_pools=[pool])
    env = BatchedNavGym(B, mp, device=dev, seed=8, auto_reset=True)
    env.reset_from_spawn_pool(np.random.RandomState(4))
    sim = PedestrianSim(env, P, seed=8)
    pol = random_policy(B, dev)

    def phase(fn, n):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n
    for _ in range(warmup):
        sim.step(pol(None))
    ms = phase(lambda: sim.step(pol(None)), steps)
    parts = dict(act=phase(sim.act, 20), robot_step=phase(lambda: env.step(pol(None)), 20), observe=phase(sim.observe, 20))
    return dict(config='crowd', envs=B, pedestrians=P, ms_per_step=ms, env_steps_per_s=B / ms * 1e3,
                pedestrian_steps_per_s=B * P / ms * 1e3, pedestrian_rays_per_s=B * P * 512 / ms * 1e3,
                ms_parts=parts)


if __name__ == '__main__':
    dev = torch.device('cuda:0')
    which = sys.argv[1:] or ['crowd']
    for w in which:
        print(json.dumps(globals()[w](dev, 100, 20)))
