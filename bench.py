#!/usr/bin/env python
"""bench.py — NavGym-v0 hot-path throughput on B200 (contract: see the task statement).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference]

A "step" is one lockstep NavGymEnv.step over the whole batch (kinematics -> lidar raycast ->
collision / goal checks -> reward + observation assembly, reference env.py:591-728).  The headline
workload is BASELINE.json configs[1] (C2): 4096 batched NavGym-v0 envs per GPU on one static indoor
map -- the reference's own create_indoor_map(3, 100) under np.random.seed(0), loaded from the
committed fixture tests/golden/bench_world.npz -- no pedestrians, default 512-beam lidar,
per-episode scan noise, random actions, device-side auto-reset from a 65 536-tuple spawn pool.
N>1 (torchrun) shards environments: 4096 per GPU, no collective on the step path (weak scaling).

Prints ONE JSON line (rank 0).  `value` = env-steps/s with inputs resident in HBM; `e2e` = the
same through the host-buffer C ABI (pinned actions in, obs/reward/done out, copies timed): the
better of the C rollout with rotating env groups and the blocking chunked call, both kept.
`configs` holds the other BASELINE configurations, device-resident: c3 (16 384 envs, 2000^2
outdoor map, 20 pedestrians; N=1), c4 (8192 envs per GPU = 65 536 / 8, 8 indoor + 8 outdoor
maps, 5..15 pedestrians, map re-drawn at reset; every N -- at N=8 this IS configs[3]), c5
(32 768 envs + on-device MLP policy, rollout loop; N=1), crowd (policy-driven pedestrians; N=1)
and her (the HER batch kernel with its HBM roofline; N=1).
`--impl reference` times the CPU restatement of the reference's path (oracle/, OpenMP over all
host cores) on the same world with the same 4096 environments per step.
`--dump-outputs DIR` writes what the last timed step of the headline leg returned to its caller
(obs, reward, done and the info fields) as DIR/<name>.npy in float32; inputs are seeded, so two
builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the tree it runs from untouched

ENVS_PER_GPU = 4096
NB = 512
OBS_DIM = NB + 7
METRIC = "env-steps/sec"
BYTES_PER_ENV_STEP = 2197  # SURVEY §8d: obs 2076 + reward 4 + done 1 + info 12 + action 8 + state 96
WORKLOAD = ("NavGym-v0 x%d envs/GPU, static indoor map 1000x1000 @0.05m (reference "
            "create_indoor_map(3, 100), np.random.seed(0); tests/golden/bench_world.npz), no "
            "pedestrians, 512-beam 360deg/25m lidar, scan noise U[0,0.05], random actions, "
            "auto-reset from a 65536-tuple spawn pool")
ACTION_LO, ACTION_HI = (0.0, -0.64), (0.5, 0.64)


def measured_peak():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
        except Exception:
            pass
    return 6650.0, 'fallback (B200_PROFILING.md)'


def build_world(seed=0, pool_n=None):
    """The bench world (both arms): the committed fixture, pure numpy, no CUDA library.  (`seed`
    is kept for the tools/ and oracle/analysis/ scripts written against round 1's generator.)"""
    from nav_gym_b200.worlds import load_bench_world
    m, pool = load_bench_world()
    return m, (pool if pool_n is None else pool[:pool_n])


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits',
                 '-lms', '50'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def wait_first(self, timeout=3.0):
        t_wait = time.time()
        while self.proc is not None and not self.rows and time.time() - t_wait < timeout:
            time.sleep(0.05)

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        rows = [r for (t, r) in self.rows if t0 - 0.05 <= t <= t1 + 0.15] or [r for (_, r) in self.rows]
        for r in rows:
            f = [x.strip() for x in r.split(',')]
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except Exception:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------ CPU arm
def cpu_reference_run(steps, warmup, B_cpu=ENVS_PER_GPU, seed=0):
    """The reference's per-step path restated on the CPU (oracle/navgym_oracle.c, OpenMP over
    all host cores; the reference itself is Python + absent native deps and cannot run on the
    GPU box).  Same world (the fixture), same action law, same B_cpu environments per step as
    the native arm.  Nothing of nav_gym_b200's CUDA library is loaded by this leg."""
    from oracle import oracle as orc
    orc.use_all_cores()
    m, pool = build_world()
    rng = np.random.RandomState(seed + 1)
    rows = pool[rng.randint(len(pool), size=B_cpu)]
    o = orc.OracleBatch([m], np.zeros(B_cpu, np.int32), rows[:, 0:2], rows[:, 2:4], rows[:, 4],
                        params=dict(t_stop=502.0))
    sigma = rng.uniform(0, 0.05, B_cpu).astype(np.float32)
    o.reset_obs(want_hits=False)
    unit = rng.standard_normal((4, B_cpu, 2, NB)).astype(np.float32)   # pre-drawn unit normals

    def one(i):
        act = rng.uniform(ACTION_LO, ACTION_HI, (B_cpu, 2)).astype(np.float32)
        noise = unit[i % len(unit)] * sigma[:, None, None]
        t = time.perf_counter()
        o.step(act, noise=noise, want_hits=False)
        dt = time.perf_counter() - t
        d = np.where(o.done)[0]
        if len(d):  # host-side respawn from the pool (the device does this in-kernel)
            r = pool[rng.randint(len(pool), size=len(d))]
            for col, src in ((orc.S_PX, 0), (orc.S_PY, 1), (orc.S_GX, 2), (orc.S_GY, 3), (orc.S_TH, 4),
                             (orc.S_PPX, 0), (orc.S_PPY, 1)):
                o.state[col, d] = r[:, src]
            o.state[orc.S_PV, d] = 0
            o.state[orc.S_PW, d] = 0
            o.steps[d] = 0
            sigma[d] = rng.uniform(0, 0.05, len(d)).astype(np.float32)
        return dt
    for i in range(warmup):
        one(i)
    tot = sum(one(i) for i in range(steps))
    return dict(value=B_cpu * steps / tot, ms_per_step=1e3 * tot / steps, cores=orc.num_threads(),
                B=B_cpu)


def cpu_baseline_block(sample_steps=60):
    r = cpu_reference_run(sample_steps, 3)
    return {"value": r['value'], "unit": METRIC, "cores": r['cores'], "kind": "port",
            "rays_per_s": r['value'] * NB,
            "sample": "%d envs x %d steps of the same world/action law, C restatement "
                      "(oracle/navgym_oracle.c) with OpenMP over %d threads; noise pre-drawn; the "
                      "reference itself is one env per Python process with pip natives absent on "
                      "this box (its own Python loop, timed in the build container: "
                      "tools/ref_python_baseline.py, BASELINE.md section 5: 372 env-steps/s with 1 "
                      "pedestrian, 58 with 5-15, one core)" % (r['B'], sample_steps, r['cores'])}


# ------------------------------------------------------------------------------ GPU legs
def _bank(torch, dev, n, B, seed):
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    lo = torch.tensor(ACTION_LO, device=dev)
    hi = torch.tensor(ACTION_HI, device=dev)
    return lo + (hi - lo) * torch.rand(n, B, 2, device=dev, generator=g)


def device_leg(torch, env, policy, K, W, flush=None, barrier=None):
    """W untimed + K timed lockstep steps, per-step CUDA events around env.step only.  Returns
    the per-step milliseconds (numpy) and the launch count."""
    from nav_gym_b200 import _lib
    lib = _lib.load()
    for i in range(W):
        env.step(policy(i))
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    if barrier:
        barrier()
    else:
        torch.cuda.synchronize(env.device)
    l0 = lib.navgym_launch_count()
    for i in range(K):
        if flush is not None:
            flush.zero_()
        act = policy(W + i)
        ev[i][0].record()
        env.step(act)
        ev[i][1].record()
    if barrier:
        barrier()
    else:
        torch.cuda.synchronize(env.device)
    return np.array([s.elapsed_time(e) for s, e in ev]), int(lib.navgym_launch_count() - l0)


DUMP_BYTES = 60 << 20   # --dump-outputs budget, all files together


def step_outputs(env):
    """Host copies, as float32, of what env.step returned: the env's own buffers (obs, reward,
    done, info), which the next step overwrites.  Flags and step counts are exact in float32."""
    out = {'obs': env.obs, 'reward': env.reward, 'done': env.done, 'is_success': env.is_success,
           'is_crash': env.is_crash, 'distance': env.distance, 'episode_step': env.steps,
           'truncated': env.truncated}
    return {k: v.float().cpu().numpy() for k, v in out.items()}


def dump_outputs(out_dir, arrays):
    """arrays: {name: [B, ...]} -> out_dir/<name>.npy.  Beyond DUMP_BYTES in all, every array keeps
    the same environments: a fixed, seeded sample of rows in ascending order."""
    B = len(arrays['obs'])
    row_bytes = sum(a[:1].nbytes for a in arrays.values())
    rows = np.arange(B)
    if B * row_bytes > DUMP_BYTES:
        rows = np.sort(np.random.RandomState(0).choice(B, DUMP_BYTES // row_bytes, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), np.ascontiguousarray(a[rows]))


def gather_block(B, ms, gathers_per_env_step, source):
    g = B * gathers_per_env_step / (ms * 1e-3) / 1e9
    return {"bound": "l2-gather", "achieved": g, "peak": GATHER_PEAK_G, "unit": "G gathers/s",
            "frac": g / GATHER_PEAK_G, "gathers_per_env_step": gathers_per_env_step,
            "gathers_source": source,
            "peak_source": "tools/gather_peak.cu on B200, 4 MB table, 64 warps/SM (profiles/r1_gather_peak.txt)"}


def config_c3(torch, dev, steps, warmup):
    from nav_gym_b200 import worlds
    from nav_gym_b200.batched_env import BatchedNavGym
    B, P = 16384, 20
    m, mp, peds = worlds.c3_world(dev, B, P)
    out = {"envs": B, "map": "outdoor 2000x2000 cells (100 m), 250 boxes", "pedestrians_per_env": P,
           "steps": steps, "warmup": warmup, "l2": "not flushed (16 MB EDT + 34 MB of rows per step > L2 share)"}
    bank = _bank(torch, dev, 32, B, 33)
    for mode, trunk in (('legs_boxes', False), ('trunk_discs', True)):
        env = BatchedNavGym(B, mp, device=dev, seed=5, auto_reset=True)
        env.reset_from_spawn_pool(np.random.RandomState(1))
        env.attach_pedestrians(peds, trunk_mode=trunk)
        env.reset()
        ms_, _ = device_leg(torch, env, lambda i: bank[i % 32], steps, warmup)
        ms = float(ms_.mean())
        out[mode] = {"ms_per_step": ms, "env_steps_per_s": B / ms * 1e3, "rays_per_s": B * NB / ms * 1e3,
                     "roofline_gather": gather_block(B, ms, GATHERS_C3, "oracle/analysis/config_gathers.py")}
        del env
    return out


def config_c4(torch, dev, steps, warmup, rank, world, barrier):
    from nav_gym_b200 import worlds
    from nav_gym_b200.batched_env import BatchedNavGym
    B = 8192
    ms_maps, mp, map_id, peds, nped = worlds.c4_world(dev, B, shard=rank)
    env = BatchedNavGym(B, mp, device=dev, map_id=map_id, seed=6, env_offset=rank * B, auto_reset=True,
                        resample_map=True)
    env.reset_from_spawn_pool(np.random.RandomState(2 + rank))
    env.attach_pedestrians(peds, nped=nped)
    env.reset()
    bank = _bank(torch, dev, 32, B, 44 + rank)
    ms_, _ = device_leg(torch, env, lambda i: bank[i % 32], steps, warmup, barrier=barrier)
    return {"envs_per_gpu": B, "global_envs": B * world, "maps": "8 indoor (cw 3-4, it 80-150) + 8 outdoor (10 boxes, w 0.3-1.0)",
            "pedestrians_per_env": "5..15 scripted (legs + boxes)", "resample_map": True,
            "steps": steps, "warmup": warmup}, float(ms_.sum())


def config_c5(torch, dev, steps, warmup, world_mp):
    """PPO-style rollout loop: 32 768 envs, a torch MLP policy (519-256-256-2, bf16) consuming
    `obs` in place on the device, actions fed straight back -- steps/s including the policy."""
    from nav_gym_b200.batched_env import BatchedNavGym
    B = 32768
    env = BatchedNavGym(B, world_mp, device=dev, seed=7, auto_reset=True)
    env.reset_from_spawn_pool(np.random.RandomState(3))
    torch.manual_seed(0)
    # the 519 observation columns are handed over as rows of 520 bf16 (one zero column): a 519-wide
    # bf16 row is 1038 bytes, which no tensor-core GEMM can load with aligned vectors
    net = torch.nn.Sequential(torch.nn.Linear(520, 256), torch.nn.Tanh(), torch.nn.Linear(256, 256),
                              torch.nn.Tanh(), torch.nn.Linear(256, 2)).to(dev).to(torch.bfloat16)
    lo = torch.tensor(ACTION_LO, device=dev)
    hi = torch.tensor(ACTION_HI, device=dev)
    scale = torch.ones(519, device=dev)
    scale[:512] = 1.0 / 25.0
    x = torch.zeros(B, 520, device=dev, dtype=torch.bfloat16)

    @torch.no_grad()
    def policy(i):
        torch.mul(env.obs, scale, out=x[:, :519])      # scale + cast in one pass over the rows
        return lo + (hi - lo) * torch.sigmoid(net(x).float())
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(warmup):
        env.step(policy(i))
    torch.cuda.synchronize(dev)
    e0.record()
    for i in range(steps):
        env.step(policy(i))
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    bank = _bank(torch, dev, 32, B, 55)
    ms_env, _ = device_leg(torch, env, lambda i: bank[i % 32], steps, warmup)
    ms_env = float(ms_env.mean())
    return {"envs": B, "policy": "torch MLP 519-256-256-2 bf16 on device (input rows zero-padded to 520 columns), obs consumed in place",
            "steps": steps, "warmup": warmup, "ms_per_step": ms, "env_steps_per_s": B / ms * 1e3,
            "ms_per_step_env_only": ms_env,
            "roofline_gather": gather_block(B, ms_env, GATHERS_PER_ENV_STEP, "as C2 (same world)")}


def config_her(torch, dev, env):
    """SURVEY 8f row 3: compute_rewards / compute_terminals / compute_info for stored observations
    (the reference's HER relabelling entry points, env.py:491-589) as one streaming kernel over
    2^20 rows.  HBM-bound: 2095 algorithmic bytes per row (2076 row + 8 goal in, 11 out)."""
    N, per_row = 1 << 20, 2095
    g = torch.Generator(device=dev)
    g.manual_seed(11)
    obs = torch.rand(N, OBS_DIM, device=dev, generator=g) * 10.0 + 1.5   # mostly clear of the thresholds
    obs[:, NB:NB + 4] = torch.rand(N, 4, device=dev, generator=g) * 50.0
    goals = torch.rand(N, 2, device=dev, generator=g) * 50.0
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ts = []
    for i in range(13):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = env.compute_rewards(obs, goals)
        e1.record()
        torch.cuda.synchronize(dev)
        if i >= 3:
            ts.append(e0.elapsed_time(e1))
    ms = float(np.mean(ts))
    peak, src = measured_peak()
    gbs = N * per_row / (ms * 1e-3) / 1e9
    return {"rows": N, "ms": ms, "rows_per_s": N / ms * 1e3, "l2": "flushed before every call",
            "crash_frac": float(out['is_crash'].float().mean()),
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                         "peak_source": src, "kernel": "her_kernel", "algorithmic_bytes_per_row": per_row}}


def config_crowd(torch, dev, steps, warmup, world_mp):
    """SURVEY 8f row 2: the C2 world with the reference's policy-driven pedestrians on the device
    (PedestrianSim: 10 per environment, each with its own 512-beam scan and a CNN policy forward
    per step through the library's tcgen05 kernels; random-init weights, human_policy.pth is not
    distributed).  One step = pedestrians act -> robots step -> pedestrians observe."""
    from nav_gym_b200.batched_env import BatchedNavGym
    from nav_gym_b200.pedestrians import PedestrianSim
    B, P = 4096, 10
    env = BatchedNavGym(B, world_mp, device=dev, seed=8, auto_reset=True)
    env.reset_from_spawn_pool(np.random.RandomState(4))
    sim = PedestrianSim(env, P, seed=8)
    bank = _bank(torch, dev, 32, B, 66)

    def timed(fn, n):
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / n
    for i in range(warmup):
        sim.step(bank[i % 32])
    ms = timed(lambda i: sim.step(bank[i % 32]), steps)
    n = B * P
    scan, goal, speed = sim.scan.reshape(n, -1), sim.goal_local.reshape(n, 2), sim.prev_action.reshape(n, 2)
    ms_policy = timed(lambda i: sim.native.mean(scan, goal, speed, out=sim._mean), 20)
    # f16x3: three f16 products per contraction -- act_fc1, conv2 (K 96), conv1 (as M128 x N96 x K16), act_fc2 (K 256)
    flop = 2.0 * n * 3 * (4096 * 256 + 128 * 32 * 96 + 128 * 96 * 16 + 256 * 128)
    tf = flop / (ms_policy * 1e-3) / 1e12
    peak_tf = None
    try:
        peak_tf = float(json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json'))).get('bf16_tflops'))
    except Exception:
        pass
    out = {"envs": B, "pedestrians_per_env": P, "policy": "HumanPolicy (human_policy.py:19-71), random-init, precision f16x3 (float32-grade)",
           "steps": steps, "warmup": warmup, "ms_per_step": ms, "env_steps_per_s": B / ms * 1e3,
           "pedestrian_steps_per_s": n / ms * 1e3, "pedestrian_rays_per_s": n * NB / ms * 1e3,
           "ms_policy_forward": ms_policy,
           "ms_parts": {"act": timed(lambda i: sim.act(), 20), "robot_step": timed(lambda i: env.step(bank[i % 32]), 20),
                        "observe": timed(lambda i: sim.observe(), 20)},
           "roofline_policy": {"bound": "tensor", "achieved": tf, "peak": peak_tf, "unit": "TFLOP/s",
                               "frac": (tf / peak_tf) if peak_tf else None,
                               "note": "tensor-core flop of the three launches' MMAs (conv1, conv2, act_fc1, act_fc2: three f16 products each) "
                                       "over the whole policy forward (operand conversion and epilogues on the CUDA cores included in the time)"}}
    return out


# ------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=2000)    # SURVEY §8d C2: 2000 timed steps
    ap.add_argument('--warmup', type=int, default=200)   # after 200 warm-up steps
    ap.add_argument('--impl', default='native', choices=['native', 'reference'])
    ap.add_argument('--envs', type=int, default=ENVS_PER_GPU, help='environments per GPU')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-flush', action='store_true')
    ap.add_argument('--no-configs', action='store_true', help='skip the c3 / c4 / c5 block')
    ap.add_argument('--no-e2e', action='store_true', help='skip the host-buffer legs (profiling runs)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help="write the last timed step's outputs (rank 0's environments) as DIR/<name>.npy")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != 'native':
        ap.error('--dump-outputs writes the outputs of the native arm')
    a.warmup = max(a.warmup, 3)
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))

    if a.impl == 'reference':
        # launchers such as torchrun export OMP_NUM_THREADS=1; the CPU arm uses every host core
        # (set before libgomp is first loaded: it reads its environment once)
        ncpu = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
        os.environ['OMP_NUM_THREADS'] = str(ncpu)
        os.environ['OMP_PROC_BIND'] = 'false'
        os.environ['OMP_WAIT_POLICY'] = 'active'
        if rank != 0:
            return
        K, W = min(a.steps, 400), min(a.warmup, 10)
        r = cpu_reference_run(K, W, B_cpu=a.envs)
        line = {"impl": "reference", "metric": METRIC, "value": r['value'], "unit": "env-steps/s",
                "n_gpus": a.gpus, "steps": K, "warmup": W,
                "ms_per_step": r['ms_per_step'], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32 scan / f64 pose", "data": "synthetic",
                "rays_per_s": r['value'] * NB,
                "config": {"workload": WORKLOAD % a.envs, "envs_per_step": r['B'],
                           "note": "CPU arm steps one GPU's share (%d envs) per step on all host cores, whatever --gpus" % r['B']},
                "cpu_baseline": {"value": r['value'], "unit": "env-steps/s", "cores": r['cores'],
                                 "kind": "port",
                                 "sample": "%d envs per step (the native arm's per-GPU batch), oracle C restatement + OpenMP" % r['B']},
                "e2e": {"value": r['value'], "unit": "env-steps/s", "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit('bench.py --impl native needs a CUDA device (no CPU fallback)')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        # NCCL prints its version banner on stdout when the first communicator comes up; stdout
        # is for the one JSON line, so file descriptor 1 points at stderr meanwhile
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group('nccl', device_id=dev)
            dist.barrier()
            torch.cuda.synchronize(dev)
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    from nav_gym_b200 import _lib
    from nav_gym_b200.batched_env import BatchedNavGym, MapPool
    import ctypes as C

    B = a.envs
    m, pool = build_world()
    mp = MapPool([m], dev, spawn_pools=[pool])
    env = BatchedNavGym(B, mp, device=dev, seed=1234, env_offset=rank * B, auto_reset=True)
    env.reset_from_spawn_pool(np.random.RandomState(100 + rank))
    K, W = a.steps, a.warmup
    n_bank = min(max(K, 8), 64)
    bank = _bank(torch, dev, n_bank, B, 7 + rank)
    flush = None if a.no_flush else torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    lib = _lib.load()

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    # ---- device-resident leg (the headline `value`) ------------------------------------
    sampler = ClockSampler(local) if rank == 0 else None
    for i in range(W):
        env.step(bank[i % n_bank])
    if sampler is not None:  # nvidia-smi needs a moment to deliver its first sample
        sampler.wait_first()
    t0 = time.time()
    step_ms, launches = device_leg(torch, env, lambda i: bank[i % n_bank], K, 0, flush=flush, barrier=barrier)
    t1 = time.time()
    total_ms = float(step_ms.sum())
    crash_frac = float(env.is_crash.float().mean().item())
    done_frac = float(env.done.float().mean().item())
    outputs = step_outputs(env) if a.dump_outputs and rank == 0 else None   # before the e2e legs step env

    # ---- end-to-end legs: HOST buffers, copies inside the timed region ----------------------
    # (a) rollout: the env groups rotate in C (navgym_host_rollout): per group H2D actions ->
    #     step -> D2H rows; a group's next actions (the policy: next row of a pinned action bank)
    #     are written only after its previous results landed; while the host serves group A,
    #     groups B.. are stepping, so PCIe hides behind the raycast.
    # (b) synchronous call: navgym_step_batch_host, one blocking call per step.
    # (c) the same D2H bytes with no simulation at all: this box's ceiling for the copy pattern.
    e2e = None
    if not a.no_e2e:
        Ke = K
        act_h = torch.empty(n_bank, B, 2, dtype=torch.float32).pin_memory()
        act_h.copy_(bank.cpu())
        obs_h = torch.empty(B, NB + 7, dtype=torch.float32).pin_memory()
        rew_h = torch.empty(B, dtype=torch.float32).pin_memory()
        done_h = torch.empty(B, dtype=torch.uint8).pin_memory()
        for i in range(min(30, max(W, 5))):
            env.step_host(act_h[i % n_bank], obs_h, rew_h, done_h)
        barrier()
        l0 = lib.navgym_launch_count()
        t_s = time.perf_counter()
        for i in range(Ke):
            env.step_host(act_h[i % n_bank], obs_h, rew_h, done_h)
        barrier()
        e2e_sync_ms = (time.perf_counter() - t_s) * 1e3
        sync_launches = int(lib.navgym_launch_count() - l0)

        # Group count: more groups hide more of the kernel behind the copies, but every group adds
        # submissions and smaller DMA chunks; which wins depends on how many GPUs share the host's
        # PCIe / memory system (8 GPUs: the copies are the bottleneck, fewer groups win).  The
        # candidates are timed on a short rollout (max over ranks, so every rank picks the same),
        # then the timed run uses the winner.  NAVGYM_HOST_GROUPS pins it.
        cur = torch.empty(B, 2, dtype=torch.float32).pin_memory()
        ab = _lib.ActionBank(C.c_void_p(act_h.data_ptr()), n_bank, B)
        policy = C.cast(lib.navgym_policy_action_bank, _lib.POLICY_FN)
        pinned = os.environ.get('NAVGYM_HOST_GROUPS')
        cands = [int(pinned)] if pinned else [4, 2, 1]
        trial = {}
        for ng in cands:
            bounds = env.host_groups(ng, cur, obs_h, rew_h, done_h)
            env.rollout_host(min(60, max(W, 8)), policy, ab)
            if len(cands) > 1:
                barrier()
                t_s = time.perf_counter()
                env.rollout_host(200, policy, ab)
                barrier()
                tt = torch.tensor([time.perf_counter() - t_s], dtype=torch.float64, device=dev)
                if world > 1:
                    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                trial[ng] = float(tt)
        n_groups = min(trial, key=trial.get) if trial else cands[0]
        if n_groups != cands[-1]:
            bounds = env.host_groups(n_groups, cur, obs_h, rew_h, done_h)
            env.rollout_host(min(60, max(W, 8)), policy, ab)
        barrier()
        l0 = lib.navgym_launch_count()
        t_s = time.perf_counter()
        env.rollout_host(Ke, policy, ab)
        barrier()
        e2e_ms = (time.perf_counter() - t_s) * 1e3
        e2e_launches = int(lib.navgym_launch_count() - l0)
        copy_bounds = [(B * g // 4, B * (g + 1) // 4) for g in range(4)]   # the copy-only leg keeps 4 chunks

        streams = [torch.cuda.Stream(device=dev) for _ in copy_bounds]
        torch.cuda.synchronize(dev)
        barrier()  # all ranks copy at the same time, as in the e2e legs
        t_s = time.perf_counter()
        for i in range(Ke):
            for s_, (b0, b1) in zip(streams, copy_bounds):
                with torch.cuda.stream(s_):
                    obs_h[b0:b1].copy_(env.obs[b0:b1], non_blocking=True)
        torch.cuda.synchronize(dev)
        barrier()
        copy_only_ms = (time.perf_counter() - t_s) * 1e3
        e2e = [e2e_ms, e2e_sync_ms, copy_only_ms]

    # ---- the other BASELINE configurations ----------------------------------------------
    cfg, c4_ms, c4_meta = {}, 0.0, None
    if not a.no_configs:
        ks, kw = max(min(K, 200), 40), 20
        c4_meta, c4_ms = config_c4(torch, dev, ks, kw, rank, world, barrier)
        if world == 1:
            cfg['c3'] = config_c3(torch, dev, ks, kw)
            cfg['c5'] = config_c5(torch, dev, ks, kw, mp)
            cfg['crowd'] = config_crowd(torch, dev, ks, kw, mp)
            cfg['her'] = config_her(torch, dev, env)

    t = torch.tensor([total_ms] + (e2e or [0.0, 0.0, 0.0]) + [c4_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms, e2e_sync_ms, copy_only_ms, c4_ms = [float(v) for v in t]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    clocks = sampler.stop(t0, t1) if sampler else None

    peak, peak_src = measured_peak()
    kernel_ms = float(step_ms.mean())
    achieved = B * BYTES_PER_ENV_STEP / (kernel_ms * 1e-3) / 1e9
    value = world * B * K / (total_ms * 1e-3)
    if c4_meta is not None:
        ms = c4_ms / c4_meta['steps']
        c4_meta.update({"ms_per_step": ms, "env_steps_per_s": world * 8192 / ms * 1e3,
                        "rays_per_s": world * 8192 * NB / ms * 1e3, "timing": "CUDA events, max over ranks",
                        "roofline_gather": gather_block(8192, ms, GATHERS_C4, "oracle/analysis/config_gathers.py")})
        cfg['c4'] = c4_meta
    line = {
        "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K,
        "warmup": W, "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32 scan / f64 pose", "data": "synthetic",
        "rays_per_s": value * NB,
        "config": {"workload": WORKLOAD % B, "envs_per_gpu": B, "global_envs": world * B,
                   "parallelism": "env-shard x%d, no step-path collective" % world,
                   "l2": "flushed between timed steps (256 MiB memset)" if flush is not None else "not flushed",
                   "crash_frac_last_step": crash_frac, "done_frac_last_step": done_frac},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": TRAFFIC_BYTES_PER_LAUNCH,
                     "peak_source": peak_src, "kernel": "step_kernel<false>",
                     "algorithmic_bytes_per_launch": B * BYTES_PER_ENV_STEP,
                     "kernel_ms": kernel_ms,
                     "note": "latency/issue-bound gather kernel: see DESIGN.md roofline section"},
        # second ceiling (SURVEY 8d ii): every march sample is one dependent 4-byte gather from the
        # L2-resident EDT; the peak is the dependent-random-gather rate tools/gather_peak.cu measured
        # on this pool's B200 at the kernel's launch shape (profiles/r1_gather_peak.txt)
        "roofline_gather": gather_block(B, kernel_ms, GATHERS_PER_ENV_STEP, "oracle/analysis/config_gathers.py"),
        "gpu_launches": launches,
        "clocks": clocks,
    }
    if K < 200:
        line["short_run"] = True
        line["short_run_note"] = ("%d timed steps = %.1f ms of device time: a smoke-sized run; the SURVEY 8d C2 "
                                  "protocol is 2000 steps after 200 warm-up (the default)" % (K, total_ms))
    if e2e is not None:
        # two public host-buffer APIs were timed over the same Ke steps (max over ranks): the C
        # rollout with rotating env groups and the blocking call (two chunked launches per step whose
        # copies overlap the next chunk's raycast).  The rollout wins wherever a GPU has the host to
        # itself; with 8 GPUs sharing one host memory system the blocking call's fewer, larger DMA
        # transfers can win.  `value` is the better one, named in `api`; both are kept.
        rollout_v = world * B * Ke / (e2e_ms * 1e-3)
        sync_v = world * B * Ke / (e2e_sync_ms * 1e-3)
        use_sync = sync_v > rollout_v
        rollout_api = ("BatchedNavGym.rollout_host (C ABI navgym_host_rollout): pinned host actions in, pinned "
                       "host obs/reward/done out, %d env groups rotated in C; a group's next actions are "
                       "written by the policy callback only after its previous results landed") % n_groups
        sync_api = ("BatchedNavGym.step_host (C ABI navgym_step_batch_host), one blocking call per step: pinned host "
                    "actions in, pinned host obs/reward/done out, two chunked launches whose copies overlap")
        line["e2e"] = {
            "value": max(rollout_v, sync_v), "unit": "env-steps/s",
            "h2d_bytes_per_step": B * 2 * 4, "d2h_bytes_per_step": B * ((NB + 7) * 4 + 4 + 1),
            "steps": Ke, "timing": "host wall clock, max over ranks",
            "gpu_launches": sync_launches if use_sync else e2e_launches,
            "api": sync_api if use_sync else rollout_api,
            "groups": n_groups,
            "groups_trial_env_steps_per_s": {str(k): world * B * 200 / v for k, v in trial.items()},
            "rollout_value": rollout_v, "rollout_api": rollout_api,
            "sync_value": sync_v, "sync_api": sync_api,
            "copy_only_value": world * B * Ke / (copy_only_ms * 1e-3),
            "frac_of_copy_only": copy_only_ms / min(e2e_ms, e2e_sync_ms),
            "copy_only_note": "every rank's observation rows copied D2H in the same chunks, all ranks at once, with no stepping: the PCIe / host-memory ceiling of the e2e figure on this box at this N"}
    if cfg:
        line["configs"] = cfg
    if not a.no_cpu_baseline and world == 1:
        line["cpu_baseline"] = cpu_baseline_block()
    if outputs is not None:
        dump_outputs(a.dump_outputs, outputs)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# dram__bytes_read.sum + dram__bytes_write.sum of step_kernel<false> per launch, from the
# `ncu --set full` capture summarised in profiles/ (None until measured).
TRAFFIC_BYTES_PER_LAUNCH = 3759616  # dram read + write of one launch, profiles/r2_step_kernel_ncu_full_summary.txt (final capture of round 2; round 1: 3193600)
# EDT gathers per env-step = march samples of the 512 beams (the t = 0 sample shared per scan) x
# scans per step, counted by the CPU checker on the same worlds: oracle/analysis/config_gathers.py
GATHERS_PER_ENV_STEP = 3415   # C2 / C5 world: 3382 per scan x 1.01
GATHERS_C3 = 4997             # 2000^2 outdoor: 4948 per scan x 1.01
GATHERS_C4 = 3575             # 16-map pool mean: 3540 per scan x 1.01
GATHER_PEAK_G = 700.0  # profiles/r1_gather_peak.txt

if __name__ == '__main__':
    main()
