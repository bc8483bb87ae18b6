"""Crowd step time with per-episode pedestrian counts: PedestrianSim(num_humans_range=(5, 15)),
NavGym-v0's num_humans law, against a fixed count of the same mean (nped = 10), both over
max_ped = 15 slots, on the C2 world with auto-reset.  The two arms are built once and timed in
alternation (CUDA events, no L2 flush); mean_nped is the mean live count over an untimed window of
the same length after each timed one.  One JSON line.

    python tools/ped_counts_bench.py [--envs 4096] [--steps 200] [--warmup 50] [--rounds 3]"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from nav_gym_b200.batched_env import BatchedNavGym, MapPool  # noqa: E402
from nav_gym_b200.pedestrians import HumanPolicy, PedestrianSim  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--envs', type=int, default=4096)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=50)
    ap.add_argument('--rounds', type=int, default=3)
    args = ap.parse_args()
    from bench import _bank, build_world
    dev = torch.device('cuda:0')
    B, P = args.envs, 15
    m, pool = build_world(0)
    mp = MapPool([m], dev, spawn_pools=[pool])
    torch.manual_seed(0)
    policy = HumanPolicy()
    arms = {}
    for name, kw in (('fixed_10', dict(nped=[10] * B)), ('range_5_15', dict(num_humans_range=(5, 15)))):
        env = BatchedNavGym(B, mp, device=dev, seed=8, auto_reset=True)
        env.reset_from_spawn_pool(np.random.RandomState(4))
        arms[name] = (env, PedestrianSim(env, P, policy=policy, seed=8, **kw))
    bank = _bank(torch, dev, 32, B, 66)
    for env, sim in arms.values():
        for i in range(args.warmup):
            sim.step(bank[i % 32])
    out = {name: dict(ms_per_step=[], mean_nped=[]) for name in arms}
    for _ in range(args.rounds):
        for name, (env, sim) in arms.items():
            live = torch.zeros((), dtype=torch.float64, device=dev)
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(args.steps):
                sim.step(bank[i % 32])
            e1.record()
            torch.cuda.synchronize(dev)
            for i in range(args.steps):   # the live counts over an untimed window of the same length
                sim.step(bank[i % 32])
                live += sim.nped.double().mean()
            out[name]['ms_per_step'].append(e0.elapsed_time(e1) / args.steps)
            out[name]['mean_nped'].append(float(live) / args.steps)
    print(json.dumps(dict(device=torch.cuda.get_device_name(dev), envs=B, max_ped=P, steps=args.steps,
                          warmup=args.warmup, arms=out)))


if __name__ == '__main__':
    main()
