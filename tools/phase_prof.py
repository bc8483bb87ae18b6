"""Per-phase cycle accounting of the fused step kernel (debug build with -DNAVGYM_PROFILE).
Build here:   python tools/phase_prof.py build
Run on GPU:   python tools/phase_prof.py run"""
import ctypes as C, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, 'tools', '_prof', 'libnavgym_b200_prof.so')
if sys.argv[1] == 'build':
    from nav_gym_b200 import _lib
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    r = subprocess.run([_lib._nvcc()] + _lib.NVCC_FLAGS + ['-DNAVGYM_PROFILE', '-Xptxas', '-v', '-o', OUT, _lib.SRC], capture_output=True, text=True)
    if r.returncode:
        sys.exit(r.stderr)
    lines = r.stderr.splitlines()
    for i, l in enumerate(lines):   # step_kernel<MODE_STEP, COOP, FMT>: stack / spills, registers / smem
        if 'Function properties for _Z11step_kernelILi0E' in l: print(l.split()[-1] + ':', lines[i+1].strip() + ';', lines[i+2].split(':', 1)[1].strip())
    print('built', OUT)
else:
    os.environ['NAVGYM_LIB'] = OUT
    import numpy as np, torch
    from nav_gym_b200 import _lib
    from nav_gym_b200.batched_env import BatchedNavGym, MapPool, filter_spawn_pool
    from bench import build_world
    B = 4096
    m, pool = build_world(0, 16384)
    npool = int(os.environ.get('NAVGYM_POOL_N', '0'))
    if npool: pool = pool[:npool]
    mp = MapPool([m], 'cuda:0', spawn_pools=[pool])
    env = BatchedNavGym(B, mp, seed=1, auto_reset=True)
    env.reset_from_spawn_pool(np.random.RandomState(1))
    bank = torch.rand(16, B, 2, device='cuda') * torch.tensor([0.5, 1.28], device='cuda') + torch.tensor([0, -0.64], device='cuda')
    if npool: bank = bank * 0
    for i in range(40): env.step(bank[i % 16])
    torch.cuda.synchronize()
    lib = _lib.load()
    buf = (C.c_ulonglong * 16)()
    lib.navgym_debug_read_prof(buf, 1)
    n = 20
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n): env.step(bank[i % 16])
    e1.record(); torch.cuda.synchronize()
    lib.navgym_debug_read_prof(buf, 1)
    names = ['prologue(kinematics)', 'pass setup', 'beam dirs(sincos)', 'march', 'obstacles', 'clip+noise+obs', 'reward/branch', 'epilogue']
    tot = sum(buf[:8])
    print('ms/step %.3f' % (e0.elapsed_time(e1) / n))
    for i, nm in enumerate(names):
        print('%-22s %8.0f cycles/CTA  %5.1f%%' % (nm, buf[i] / (n * B), 100.0 * buf[i] / tot))
    print('total %.0f cycles/CTA' % (tot / (n * B)))
    tl = env.tail64.cpu().numpy()
    t0 = tl[:, 0].min(); st = (tl[:, 0] - t0) / 1e3; en = (tl[:, 1] - t0) / 1e3; dur = en - st
    print('kernel span %.1f us; CTA duration us: mean %.1f p50 %.1f p90 %.1f p99 %.1f max %.1f' % (en.max(), dur.mean(), np.percentile(dur, 50), np.percentile(dur, 90), np.percentile(dur, 99), dur.max()))
    print('CTA start us: p50 %.1f p90 %.1f max %.1f ; last 5 to end: ' % (np.percentile(st, 50), np.percentile(st, 90), st.max()), [(round(st[i], 1), round(en[i], 1), int(tl[i, 3])) for i in np.argsort(en)[-5:]])
    ts = np.linspace(0, en.max(), 23)[1:-1]
    print('resident CTAs over time:', [int(((st <= t) & (en > t)).sum()) for t in ts])
    dn = env.done.cpu().numpy().astype(bool)
    print('episode-ending envs: %d of %d; start us p50 %.1f p90 %.1f max %.1f; duration us mean %.1f max %.1f; end us p50 %.1f max %.1f' % (
        dn.sum(), B, np.percentile(st[dn], 50), np.percentile(st[dn], 90), st[dn].max(), dur[dn].mean(), dur[dn].max(), np.percentile(en[dn], 50), en[dn].max()))
    print('others: duration us mean %.1f p99 %.1f max %.1f; end us max %.1f' % (dur[~dn].mean(), np.percentile(dur[~dn], 99), dur[~dn].max(), en[~dn].max()))
    late = np.argsort(en)[-40:]
    print('last 40 CTAs to end: %d episode-ending; their starts us: %s' % (dn[late].sum(), np.round(np.sort(st[late]), 1).tolist()))
    sm = tl[:, 2].astype(int)
    busy = np.array([en[sm == i].max() for i in np.unique(sm)])
    print('per-SM finish time us: min %.1f mean %.1f max %.1f' % (busy.min(), busy.mean(), busy.max()))
    wk = np.floor(tl[:, 4] / (4096.0 * 16777216.0)); cb = np.floor((tl[:, 4] - wk * 4096.0 * 16777216.0) / 4096.0); tl[:, 4] = tl[:, 4] - wk * 4096.0 * 16777216.0 - cb * 4096.0
    al, ia, rb = tl[:, 4], tl[:, 5], tl[:, 6]
    print('regime B: cycles per CTA mean %.0f (max warp); rounds %.1f; walk iterations %.1f; cycles/round %.0f; walk its/round %.1f' % (cb.mean(), rb.mean(), wk.mean(), cb.sum() / max(rb.sum(), 1), wk.sum() / max(rb.sum(), 1)))
    print('survivors per env: mean %.0f p99 %.0f max %.0f; regime A iterations (max over warps): mean %.1f p99 %.0f max %.0f; regime B rounds: mean %.1f p99 %.0f max %.0f' % (
        al.mean(), np.percentile(al, 99), al.max(), ia.mean(), np.percentile(ia, 99), ia.max(), rb.mean(), np.percentile(rb, 99), rb.max()))
    one = ~dn
    print('corr(duration, survivors) %.3f  corr(duration, A iters) %.3f  corr(duration, A+B) %.3f' % (
        np.corrcoef(dur[one], al[one])[0, 1], np.corrcoef(dur[one], ia[one])[0, 1], np.corrcoef(dur[one], (ia + rb)[one])[0, 1]))
    for i in np.argsort(dur)[-8:]:
        print('  slow env %5d: start %.1f dur %.1f us  survivors %d  A iters %d  B rounds %d  done %d' % (i, st[i], dur[i], al[i], ia[i], rb[i], dn[i]))
    cyc = dur[one] * 1.965e3
    print('one-scan envs: cycles per (A iter + B round): mean %.0f' % (cyc.sum() / max((ia + rb)[one].sum(), 1)))
    if os.environ.get('NAVGYM_DUMP'):
        np.save(os.environ['NAVGYM_DUMP'], np.column_stack([tl, dn.astype(np.float64), env.is_crash.cpu().numpy()]))
