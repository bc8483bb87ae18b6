"""CPU: the C-ABI library builds for sm_100a, loads, and exports every symbol that
include/navgym_b200.h declares.  No compute calls (there is no GPU here)."""
import ctypes as C
import os
import re

import pytest

from nav_gym_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def lib():
    _lib.build()
    return _lib.load()


def _declared():
    src = open(os.path.join(ROOT, 'include', 'navgym_b200.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(navgym_[a-z0-9_]+)\s*\(', src)))


def test_every_declared_symbol_is_exported(lib):
    names = _declared()
    assert len(names) >= 15
    for n in names:
        assert hasattr(lib, n), n
    assert sorted(_lib.EXPORTS) == names


def test_struct_layout_matches(lib):
    assert lib.navgym_sizeof_step_args() == C.sizeof(_lib.StepArgs)
    assert lib.navgym_sizeof_map() == C.sizeof(_lib.MapT)
    assert lib.navgym_abi_version() == 1


def test_no_cpu_fallback(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    with pytest.raises(RuntimeError):
        _lib.require_device()
    from nav_gym_b200.batched_env import BatchedNavGym
    import numpy as np
    m = dict(data=np.zeros((8, 8), np.int8), origin=(0, 0), resolution=0.05, width=8, height=8)
    with pytest.raises(RuntimeError):
        BatchedNavGym(1, [m])


def test_sass_is_sm100a(lib):
    import subprocess
    # the cuobjdump of the toolkit whose nvcc built the library, found the same way (PATH or
    # /usr/local/cuda/bin)
    nvcc = _lib._nvcc()
    assert nvcc is not None
    cuobjdump = os.path.join(os.path.dirname(nvcc), 'cuobjdump')
    out = subprocess.run([cuobjdump, '-lelf', _lib.SO], capture_output=True, text=True, check=True).stdout
    assert 'sm_100a' in out


def test_plain_c_client_links_and_runs(lib, tmp_path):
    """include/navgym_b200.h is valid C99 and a C program linked against the shared library
    sees the same ABI (struct sizes, no-op empty batch, host helper) -- the view a cgo / JNI /
    FFI host has of the boundary."""
    import shutil
    import subprocess
    from nav_gym_b200 import _lib
    gcc = shutil.which('gcc')
    if gcc is None:
        pytest.skip('no gcc')
    here = os.path.dirname(os.path.abspath(__file__))
    exe = str(tmp_path / 'abi_client')
    subprocess.check_call([gcc, '-std=c99', '-Wall', '-Wextra', '-pedantic', '-Werror',
                           '-I', os.path.dirname(_lib.HDR), os.path.join(here, 'abi_client.c'),
                           '-o', exe, '-L', os.path.dirname(_lib.SO), '-lnavgym_b200',
                           '-Wl,-rpath,' + os.path.dirname(_lib.SO)])
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0, (out.returncode, out.stdout, out.stderr)
    assert 'abi ok' in out.stdout


# ---- field-by-field layout: the ctypes mirrors in _lib.py against the header as gcc lays it out
_MIRRORS = {
    'navgym_map_t': 'MapT', 'navgym_step_args_t': 'StepArgs', 'navgym_her_args_t': 'HerArgs',
    'navgym_peds_args_t': 'PedsArgs', 'navgym_scan_args_t': 'ScanArgs', 'navgym_plan_map_t': 'PlanMapT',
    'navgym_plan_args_t': 'PlanArgs', 'navgym_move_args_t': 'MoveArgs', 'navgym_action_bank_t': 'ActionBank',
    'navgym_policy_params_t': 'PolicyParams',
}


def _header_structs():
    """{typedef name: [field names in declaration order]} parsed from the header's text."""
    src = open(os.path.join(ROOT, 'include', 'navgym_b200.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    out = {}
    for body, name in re.findall(r'typedef\s+struct\s*\{(.*?)\}\s*(navgym_[a-z0-9_]+)\s*;', src, flags=re.S):
        fields = []
        for decl in body.split(';'):
            decl = decl.strip()
            if not decl:
                continue
            # "const float *thr, *dthr" / "double robot_fp[8], agent_fp[8]" / "int32_t W, H"
            first, *rest = decl.split(',')
            names = [first.split()[-1]] + [r.strip() for r in rest]
            fields += [re.sub(r'\[.*?\]', '', n).replace('*', '').strip() for n in names]
        out[name] = fields
    return out


def test_every_field_offset_matches_the_header(tmp_path):
    """A C program built from the header prints offsetof / sizeof of EVERY field of every
    argument struct; the ctypes mirrors must agree name by name, in order.  (Two swapped
    same-size fields pass a sizeof check and corrupt silently.)"""
    import shutil
    import subprocess
    gcc = shutil.which('gcc')
    if gcc is None:
        pytest.skip('no gcc')
    structs = _header_structs()
    assert set(_MIRRORS) <= set(structs), sorted(set(_MIRRORS) - set(structs))
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "navgym_b200.h"', 'int main(void) {']
    for s, fields in structs.items():
        if s not in _MIRRORS:
            continue
        for f in fields:
            lines.append('  printf("%s %s %%zu %%zu\\n", offsetof(%s, %s), sizeof(((%s *)0)->%s));' % (s, f, s, f, s, f))
        lines.append('  printf("%s . %%zu 0\\n", sizeof(%s));' % (s, s))
    lines += ['  return 0;', '}']
    src = tmp_path / 'offsets.c'
    src.write_text('\n'.join(lines))
    exe = str(tmp_path / 'offsets')
    subprocess.check_call([gcc, '-std=c99', '-I', os.path.dirname(_lib.HDR), str(src), '-o', exe])
    out = subprocess.run([exe], capture_output=True, text=True, check=True).stdout
    seen = {}
    for ln in out.split('\n'):
        if ln:
            s, f, off, size = ln.split()
            seen.setdefault(s, []).append((f, int(off), int(size)))
    n_checked = 0
    for s, mirror in _MIRRORS.items():
        cls = getattr(_lib, mirror)
        c_fields = [x for x in seen[s] if x[0] != '.']
        assert [f for f, _, _ in c_fields] == [f for f, _ in cls._fields_], s
        for f, off, size in c_fields:
            d = getattr(cls, f)
            assert (d.offset, d.size) == (off, size), (s, f, (d.offset, d.size), (off, size))
            n_checked += 1
        assert C.sizeof(cls) == [x for x in seen[s] if x[0] == '.'][0][1], s
    assert n_checked > 150


# ---- argument checks of the entry points that take a navgym_step_args_t.  The blocks hold NULL
# device pointers: they are refused, or found empty, before any device work, so no GPU is needed.
def _step_args(**fields):
    a = _lib.StepArgs()
    a.num_envs, a.obs_stride, a.num_scan_stack = 4, _lib.OBS_DIM, 1
    for k, v in fields.items():
        setattr(a, k, v)
    return a


@pytest.mark.parametrize('fields', [dict(env_begin=-1), dict(env_begin=5), dict(env_count=-1),
                                    dict(env_begin=1, env_count=4), dict(obs_format=7)],
                         ids=lambda f: ','.join('%s=%d' % kv for kv in f.items()))
def test_step_entry_points_reject_a_bad_argument_block(lib, fields):
    a = C.byref(_step_args(**fields))
    mask, out = (C.c_uint8 * 4)(), (C.c_double * 4096)()
    launches = lib.navgym_launch_count()
    assert lib.navgym_step_batch(a, None) == 1   # cudaErrorInvalidValue
    assert lib.navgym_reset_obs_batch(a, None) == 1
    assert lib.navgym_reset_envs(a, C.cast(mask, C.c_void_p), None) == 1
    assert lib.navgym_export_env(a, 0, C.cast(out, C.c_void_p), None) == 1
    assert lib.navgym_launch_count() == launches


def test_step_entry_points_accept_an_empty_range(lib):
    a = C.byref(_step_args(env_begin=4, env_count=0))
    mask = (C.c_uint8 * 4)()
    launches = lib.navgym_launch_count()
    assert lib.navgym_step_batch(a, None) == 0
    assert lib.navgym_reset_obs_batch(a, None) == 0
    assert lib.navgym_reset_envs(a, C.cast(mask, C.c_void_p), None) == 0
    assert lib.navgym_launch_count() == launches
