"""float32 vs float16 observation rows (BatchedNavGym(obs_dtype=...)) on the C2 world, one command.

  python tools/obs_half_bench.py --out DIR [--steps K] [--warmup W] [--reps R]

The two arms alternate (f32, f16, f32, f16, ...), R times each, and every repetition measures:
  device_step    ms per lockstep step at 4096 and 32 768 envs, CUDA events around env.step, L2
                 flushed (256 MiB memset) before every timed step, as bench.py does
  kernel_only    ms per step at 4096 envs, CUDA events around K back-to-back steps, no flush:
                 the device bound of the host rollout below
  host_rollout   env-steps/s at 4096 envs through navgym_host_rollout (pinned action bank in,
                 pinned rows / reward / done out), env groups calibrated among 4 / 2 / 1 on a
                 200-step trial as bench.py does
  copy_only      env-steps/s of the same D2H row bytes with no stepping (4 chunks on 4 streams):
                 the PCIe / host-memory ceiling of host_rollout for that row width
  her            compute_rewards on 2^20 rows (S = 1), L2 flushed before every call: ms, rows/s,
                 and GB/s of the algorithmic bytes (2095 per float32 row, 1075 per float16 row)
The card's name, power limit and max SM clock are read in the same run.  Writes
DIR/obs_half_bench.json and prints its summary as one JSON line.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

HBM_DATASHEET_GBS = 7700.0   # NVIDIA HGX B200 data sheet, per GPU
HER_BYTES = {'f32': 2076 + 8 + 11, 'f16': 1056 + 8 + 11}


def card():
    try:
        out = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.max.sm',
                              '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=30).stdout
        name, power, clk = [x.strip() for x in out.strip().split('\n')[0].split(',')]
        return {'name': name, 'power_limit_w': float(power), 'sm_max_mhz': float(clk)}
    except Exception as e:   # the torch name below still identifies the card
        return {'nvidia_smi_error': repr(e)}


def run_arm(torch, dt, mp, bank_dev, act_h, args, flush):
    import bench
    from nav_gym_b200 import _lib
    from nav_gym_b200.batched_env import BatchedNavGym
    dev = torch.device('cuda:0')
    K, W = args.steps, args.warmup
    n_bank = bank_dev[4096].shape[0]
    out = {}
    # ---- device step, L2 flushed
    for B in (4096, 32768):
        env = BatchedNavGym(B, mp, device=dev, seed=1234, auto_reset=True, obs_dtype=dt)
        env.reset_from_spawn_pool(np.random.RandomState(100))
        bank = bank_dev[B]
        ms, _ = bench.device_leg(torch, env, lambda i: bank[i % n_bank], K, W, flush=flush)
        out['device_step_%d' % B] = {'ms_mean': float(ms.mean()), 'ms_median': float(np.median(ms)),
                                     'env_steps_per_s': B / float(ms.mean()) * 1e3}
        del env
    # ---- host rollout at 4096 envs
    B = 4096
    env = BatchedNavGym(B, mp, device=dev, seed=1234, auto_reset=True, obs_dtype=dt)
    env.reset_from_spawn_pool(np.random.RandomState(100))
    bank = bank_dev[B]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(W):
        env.step(bank[i % n_bank])
    e0.record()
    for i in range(K):
        env.step(bank[i % n_bank])
    e1.record()
    torch.cuda.synchronize(dev)
    out['kernel_only_4096'] = {'ms_per_step': e0.elapsed_time(e1) / K}
    out['kernel_only_4096']['env_steps_per_s'] = B / out['kernel_only_4096']['ms_per_step'] * 1e3
    lib = _lib.load()
    cur = torch.empty(B, 2, dtype=torch.float32).pin_memory()
    obs_h = torch.empty(B, env.obs_dim, dtype=dt).pin_memory()
    rew_h = torch.empty(B, dtype=torch.float32).pin_memory()
    done_h = torch.empty(B, dtype=torch.uint8).pin_memory()
    ab = _lib.ActionBank(C.c_void_p(act_h.data_ptr()), n_bank, B)
    policy = C.cast(lib.navgym_policy_action_bank, _lib.POLICY_FN)
    trial = {}
    for ng in (4, 2, 1):
        env.host_groups(ng, cur, obs_h, rew_h, done_h)
        env.rollout_host(max(W, 8), policy, ab)
        torch.cuda.synchronize(dev)
        t = time.perf_counter()
        env.rollout_host(200, policy, ab)
        torch.cuda.synchronize(dev)
        trial[ng] = B * 200 / (time.perf_counter() - t)
    ng = max(trial, key=trial.get)
    env.host_groups(ng, cur, obs_h, rew_h, done_h)
    env.rollout_host(max(W, 8), policy, ab)
    torch.cuda.synchronize(dev)
    t = time.perf_counter()
    env.rollout_host(K, policy, ab)
    torch.cuda.synchronize(dev)
    out['host_rollout_4096'] = {'env_steps_per_s': B * K / (time.perf_counter() - t), 'groups': ng,
                                'groups_trial_env_steps_per_s': {str(k): v for k, v in trial.items()},
                                'row_bytes': env.obs_dim * env.obs.element_size()}
    # ---- copy only: the same row bytes D2H, no stepping
    bounds = [(B * g // 4, B * (g + 1) // 4) for g in range(4)]
    streams = [torch.cuda.Stream(device=dev) for _ in bounds]
    torch.cuda.synchronize(dev)
    t = time.perf_counter()
    for i in range(K):
        for s_, (b0, b1) in zip(streams, bounds):
            with torch.cuda.stream(s_):
                obs_h[b0:b1].copy_(env.obs[b0:b1], non_blocking=True)
    torch.cuda.synchronize(dev)
    out['copy_only_4096'] = {'env_steps_per_s': B * K / (time.perf_counter() - t)}
    her_env = env
    # ---- HER on 2^20 rows: the same values in either format (float32 rows rounded for f16)
    N = 1 << 20
    g = torch.Generator(device=dev)
    g.manual_seed(11)
    rows32 = torch.rand(N, 519, device=dev, generator=g) * 10.0 + 1.5
    rows32[:, 512:516] = torch.rand(N, 4, device=dev, generator=g) * 50.0
    goals = torch.rand(N, 2, device=dev, generator=g) * 50.0
    if dt == torch.float16:
        rows = torch.zeros(N, 512 + 16, dtype=torch.float16, device=dev)
        scans, tail = her_env.obs_parts(rows)
        scans.copy_(rows32[:, :512])
        tail.copy_(rows32[:, 512:])
        del rows32
    else:
        rows = rows32
    ts = []
    for i in range(13):
        flush.zero_()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        res = her_env.compute_rewards(rows, goals)
        a1.record()
        torch.cuda.synchronize(dev)
        if i >= 3:
            ts.append(a0.elapsed_time(a1))
    ms = float(np.mean(ts))
    key = 'f16' if dt == torch.float16 else 'f32'
    gbs = N * HER_BYTES[key] / (ms * 1e-3) / 1e9
    out['her'] = {'rows': N, 'ms': ms, 'rows_per_s': N / ms * 1e3, 'algorithmic_bytes_per_row': HER_BYTES[key],
                  'GBps': gbs, 'frac_of_datasheet_hbm': gbs / HBM_DATASHEET_GBS,
                  'crash_frac': float(res['is_crash'].float().mean())}
    del env, her_env, rows, goals
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
        raise SystemExit('obs_half_bench.py needs a CUDA device')
    import bench
    from nav_gym_b200 import worlds
    from nav_gym_b200.batched_env import MapPool
    dev = torch.device('cuda:0')
    torch.cuda.set_device(dev)
    info = card()
    info['torch_name'] = torch.cuda.get_device_name(dev)
    m, pool = worlds.load_bench_world()
    mp = MapPool([m], dev, spawn_pools=[pool])
    n_bank = 64
    bank_dev = {B: bench._bank(torch, dev, n_bank, B, 7) for B in (4096, 32768)}
    act_h = bank_dev[4096].cpu().pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    reps = {'f32': [], 'f16': []}
    for r in range(args.reps):
        for key, dt in (('f32', torch.float32), ('f16', torch.float16)):
            reps[key].append(run_arm(torch, dt, mp, bank_dev, act_h, args, flush))
    summ = {k: summarize(v) for k, v in reps.items()}
    med = lambda k, p: summ[k][p]['median']
    result = {
        'card': info, 'world': 'C2 (worlds.load_bench_world)', 'steps': args.steps, 'warmup': args.warmup,
        'reps_per_arm': args.reps, 'order': 'f32, f16 alternating',
        'summary': summ,
        'ratios_f16_over_f32_median': {
            'host_rollout_4096': med('f16', 'host_rollout_4096.env_steps_per_s') / med('f32', 'host_rollout_4096.env_steps_per_s'),
            'copy_only_4096': med('f16', 'copy_only_4096.env_steps_per_s') / med('f32', 'copy_only_4096.env_steps_per_s'),
            'device_step_4096_ms': med('f16', 'device_step_4096.ms_mean') / med('f32', 'device_step_4096.ms_mean'),
            'device_step_32768_ms': med('f16', 'device_step_32768.ms_mean') / med('f32', 'device_step_32768.ms_mean'),
            'her_ms': med('f16', 'her.ms') / med('f32', 'her.ms'),
        },
        'hbm_reference': 'NVIDIA HGX B200 data sheet, 7.7 TB/s per GPU (not a measured peak)',
        'reps': reps,
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, 'obs_half_bench.json'), 'w') as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: result[k] for k in ('card', 'ratios_f16_over_f32_median', 'summary')}))


if __name__ == '__main__':
    main()
