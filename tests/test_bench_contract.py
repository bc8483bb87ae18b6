"""bench.py's output contract: one JSON line on stdout with the keys the driver reads.  The CPU
(reference) arm runs anywhere; the native arm needs a GPU."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better',
             'scaling', 'vs_baseline', 'dtype', 'data', 'config', 'e2e', 'gpu_launches'}


DUMP_NAMES = {'obs', 'reward', 'done', 'is_success', 'is_crash', 'distance', 'episode_step', 'truncated'}


def _run(args, env=None, ok=True):
    e = dict(os.environ)
    e.update(env or {})
    p = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + args, cwd=ROOT, env=e,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=900)
    assert (p.returncode == 0) == ok, p.stderr.decode()[-2000:]
    return p.stdout.decode()


def _load_dump(d):
    import numpy as np
    names = sorted(os.listdir(d))
    assert {n[:-4] for n in names} == DUMP_NAMES and all(n.endswith('.npy') for n in names)
    assert sum(os.path.getsize(os.path.join(d, n)) for n in names) <= 64 << 20
    return {n[:-4]: np.load(os.path.join(d, n)) for n in names}


def test_reference_arm_prints_one_json_line():
    out = _run(['--impl', 'reference', '--steps', '3', '--warmup', '3', '--envs', '64'])
    lines = [l for l in out.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert BASE_KEYS <= set(d) and d['impl'] == 'reference'
    assert d['metric'] == 'env-steps/sec' and d['unit'] == 'env-steps/s' and d['higher_is_better'] is True
    assert d['value'] > 0 and d['gpu_launches'] == 0
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1
    assert d['e2e']['value'] == d['value'] and d['e2e']['h2d_bytes_per_step'] == 0
    assert 'workload' in d['config']


def test_reference_arm_other_ranks_are_silent():
    out = _run(['--impl', 'reference', '--gpus', '2', '--steps', '3', '--warmup', '3', '--envs', '64'],
               env={'RANK': '1', 'WORLD_SIZE': '2', 'LOCAL_RANK': '1'})
    assert out.strip() == ''


def test_dump_outputs_is_for_the_native_arm(tmp_path):
    _run(['--impl', 'reference', '--steps', '3', '--envs', '64', '--dump-outputs', str(tmp_path / 'd')], ok=False)
    assert not (tmp_path / 'd').exists()


def test_dump_outputs_keeps_a_fixed_sample_of_large_batches(tmp_path):
    """Beyond the size budget every file keeps the same seeded rows; below it, all rows."""
    import numpy as np
    import bench
    B = 40000   # 40000 rows x 2104 bytes = 84 MB
    rng = np.random.RandomState(1)
    arrays = {n: rng.rand(B).astype(np.float32) for n in DUMP_NAMES - {'obs'}}
    arrays['obs'] = np.repeat(np.arange(B, dtype=np.float32)[:, None], 519, axis=1)
    for sub in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / sub), arrays)
    a, b = _load_dump(str(tmp_path / 'a')), _load_dump(str(tmp_path / 'b'))
    rows = a['obs'][:, 0].astype(np.int64)
    assert 20000 < len(rows) < B and (np.diff(rows) > 0).all() and (a['obs'] == rows[:, None]).all()
    for n in DUMP_NAMES:
        assert a[n].dtype == np.float32 and np.array_equal(a[n], b[n])
        if n != 'obs':
            assert np.array_equal(a[n], arrays[n][rows])
    small = {n: v[:100] for n, v in arrays.items()}
    bench.dump_outputs(str(tmp_path / 'c'), small)
    c = _load_dump(str(tmp_path / 'c'))
    assert all(np.array_equal(c[n], small[n]) for n in DUMP_NAMES)


@pytest.mark.gpu
def test_native_arm_dumps_the_same_outputs_for_the_same_arguments(tmp_path):
    """--dump-outputs: the last timed step's obs / reward / done / info as float32 files; seeded
    inputs, so two runs with the same arguments write identical arrays."""
    import json as _json
    import numpy as np
    dumps = []
    for sub in ('a', 'b'):
        out = _run(['--steps', '25', '--warmup', '3', '--envs', '512', '--no-configs', '--no-e2e',
                    '--no-cpu-baseline', '--dump-outputs', str(tmp_path / sub)])
        assert _json.loads(out)['steps'] == 25
        dumps.append(_load_dump(str(tmp_path / sub)))
    a, b = dumps
    assert a['obs'].shape == (512, 519) and all(a[n].shape == (512,) for n in DUMP_NAMES - {'obs'})
    for n in DUMP_NAMES:
        assert a[n].dtype == np.float32 and np.array_equal(a[n], b[n]), n
    assert np.isfinite(a['obs']).all() and a['episode_step'].max() >= 1 and set(np.unique(a['done'])) <= {0.0, 1.0}


@pytest.mark.gpu
def test_native_arm_prints_one_json_line():
    out = _run(['--steps', '20', '--warmup', '3', '--envs', '512', '--no-configs'])
    lines = [l for l in out.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert BASE_KEYS <= set(d) and 'impl' not in d
    assert d['n_gpus'] == 1 and d['steps'] == 20 and d['gpu_launches'] >= 20
    r = d['roofline']
    assert r['bound'] == 'hbm' and r['unit'] == 'GB/s' and abs(r['frac'] - r['achieved'] / r['peak']) < 1e-9
    assert d['cpu_baseline']['value'] > 0 and d['cpu_baseline']['kind'] == 'port'
    e = d['e2e']
    assert e['value'] > 0 and e['h2d_bytes_per_step'] == 512 * 8 and e['d2h_bytes_per_step'] == 512 * (519 * 4 + 5)
    assert d['clocks']['sm_mhz'] > 0 and d.get('short_run') is True
