"""Cost of the masked device reset (BatchedNavGym.reset_envs) and of next-step auto-reset on the
C2 world, one command.

  python tools/reset_envs_bench.py --out DIR [--steps K] [--warmup W] [--reps R]

Three arms, alternated (auto, masked, next, auto, masked, next, ...), R times each, at 4096 and
32 768 envs with bench.py's action law (a seeded bank of uniform actions):
  auto     BatchedNavGym(auto_reset=True): env.step
  masked   BatchedNavGym(auto_reset=False): env.step, then env.reset_envs(env.done)
  next     BatchedNavGym(auto_reset='next_step'): env.step
ms per step = CUDA events around the step (and, in the masked arm, the reset), L2 flushed
(256 MiB memset) before every timed step, as bench.py does.  Then reset_envs alone at mask
fractions 0, 1 %, 10 % and 100 % (random masks, fixed seed), same timing and flush.  The card's
name, power limit and max SM clock are read in the same run.  Writes DIR/reset_envs_bench.json
and prints its summary as one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

SIZES = (4096, 32768)
FRACTIONS = (0.0, 0.01, 0.1, 1.0)


def card():
    try:
        out = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.max.sm',
                              '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=30).stdout
        name, power, clk = [x.strip() for x in out.strip().split('\n')[0].split(',')]
        return {'name': name, 'power_limit_w': float(power), 'sm_max_mhz': float(clk)}
    except Exception as e:   # the torch name below still identifies the card
        return {'nvidia_smi_error': repr(e)}


def timed(torch, fn, K, W, flush):
    """W untimed + K timed calls of fn(i), CUDA events around each, L2 flushed before each."""
    for i in range(W):
        fn(i)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    torch.cuda.synchronize()
    for i in range(K):
        flush.zero_()
        ev[i][0].record()
        fn(W + i)
        ev[i][1].record()
    torch.cuda.synchronize()
    return np.array([s.elapsed_time(e) for s, e in ev])


ARMS = {'auto': True, 'masked': False, 'next': 'next_step'}   # arm -> auto_reset


def run_arm(torch, arm, mp, banks, args, flush):
    from nav_gym_b200.batched_env import BatchedNavGym
    masked = arm == 'masked'
    out = {}
    for B in SIZES:
        env = BatchedNavGym(B, mp, device='cuda:0', seed=1234, auto_reset=ARMS[arm])
        env.reset_from_spawn_pool(np.random.RandomState(100))
        bank = banks[B]
        n_bank = bank.shape[0]

        def step(i):
            env.step(bank[i % n_bank])
            if masked:
                env.reset_envs(env.done)

        ms = timed(torch, step, args.steps, args.warmup, flush)
        ended = []   # episodes ending per step, over 100 untimed steps more
        for i in range(100):
            step(i)
            ended.append(env.done.sum())
        done_frac = float(torch.stack(ended).float().mean()) / B
        out['step_%d' % B] = {'ms_mean': float(ms.mean()), 'ms_median': float(np.median(ms)),
                              'env_steps_per_s': B / float(ms.mean()) * 1e3, 'done_fraction_per_step': done_frac}
        del env
    torch.cuda.empty_cache()
    return out


def reset_only(torch, mp, args, flush):
    from nav_gym_b200.batched_env import BatchedNavGym
    out = {}
    for B in SIZES:
        env = BatchedNavGym(B, mp, device='cuda:0', seed=1234, auto_reset=False)
        env.reset_from_spawn_pool(np.random.RandomState(100))
        g = torch.Generator(device='cuda:0')
        g.manual_seed(5)
        for f in FRACTIONS:
            mask = torch.rand(B, device='cuda:0', generator=g) < f
            ms = timed(torch, lambda i: env.reset_envs(mask), args.steps, args.warmup, flush)
            out['reset_%d_frac_%g' % (B, f)] = {'ms_mean': float(ms.mean()), 'ms_median': float(np.median(ms)),
                                                'masked_envs': int(mask.sum())}
        del env
    torch.cuda.empty_cache()
    return out


def summarize(reps):
    """{metric path: {min, median, max}} over the repetitions of one arm."""
    flat = {}
    for r in reps:
        for leg, d in r.items():
            for k, v in d.items():
                if isinstance(v, float):
                    flat.setdefault(leg + '.' + k, []).append(v)
    return {k: {'min': min(v), 'median': float(np.median(v)), 'max': max(v)} for k, v in flat.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True, help='output directory')
    ap.add_argument('--steps', type=int, default=500)
    ap.add_argument('--warmup', type=int, default=50)
    ap.add_argument('--reps', type=int, default=3)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('reset_envs_bench.py needs a CUDA device')
    import bench
    from nav_gym_b200 import worlds
    from nav_gym_b200.batched_env import MapPool
    dev = torch.device('cuda:0')
    torch.cuda.set_device(dev)
    info = card()
    info['torch_name'] = torch.cuda.get_device_name(dev)
    m, pool = worlds.load_bench_world()
    mp = MapPool([m], dev, spawn_pools=[pool])
    banks = {B: bench._bank(torch, dev, 64, B, 7) for B in SIZES}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    reps = {k: [] for k in ARMS}
    for r in range(args.reps):
        for key in ARMS:
            reps[key].append(run_arm(torch, key, mp, banks, args, flush))
    summ = {k: summarize(v) for k, v in reps.items()}
    alone = summarize([reset_only(torch, mp, args, flush) for _ in range(args.reps)])
    med = lambda k, p: summ[k][p]['median']
    result = {
        'card': info, 'world': 'C2 (worlds.load_bench_world)', 'steps': args.steps, 'warmup': args.warmup,
        'reps_per_arm': args.reps, 'order': 'auto, masked, next alternating; then reset_envs alone',
        'summary': summ, 'reset_envs_alone': alone,
        'masked_minus_auto_ms_median': {B: med('masked', 'step_%d.ms_mean' % B) - med('auto', 'step_%d.ms_mean' % B)
                                        for B in SIZES},
        'next_minus_auto_ms_median': {B: med('next', 'step_%d.ms_mean' % B) - med('auto', 'step_%d.ms_mean' % B)
                                      for B in SIZES},
        'reps': reps,
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, 'reset_envs_bench.json'), 'w') as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: result[k] for k in ('card', 'summary', 'reset_envs_alone', 'masked_minus_auto_ms_median',
                                                   'next_minus_auto_ms_median')}))


if __name__ == '__main__':
    main()
