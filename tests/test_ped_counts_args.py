"""CPU: navgym_peds_plan checks the per-episode count fields before any device work.  Every block
below is refused, so the (host) pointers in it are never dereferenced and no GPU is needed."""
import ctypes as C

import pytest

from nav_gym_b200 import _lib

_BUF = (C.c_double * 64)()
_NAMES = ('maps', 'fields', 'goals', 'map_id', 'pose', 'goal_id', 'waypoint', 'goal_local', 'free_xy', 'robot_state',
          'pose_rw', 'v_pref', 'has_legs', 'dist_travelled', 'vel', 'prev_action', 'cand_pose', 'cand_v_pref',
          'cand_legs', 'cand_goal', 'cand_rows')


def _args(**fields):
    """A block that would pass the check (4 environments x 6 slots, counts 2..6), then `fields`."""
    a = _lib.PlanArgs()
    a.num_envs, a.max_ped = 4, 6
    base = C.addressof(_BUF)
    for i, name in enumerate(_NAMES):
        setattr(a, name, base + 8 * (i % 8))
    a.nped, a.cand_nped_prev, a.cand_nped, a.nped_out = base + 256, base + 272, base + 288, base + 304
    a.num_humans_lo, a.num_humans_hi = 2, 6
    for k, v in fields.items():
        setattr(a, k, v)
    return a


@pytest.mark.parametrize('fields', [
    dict(num_humans_lo=-1), dict(num_humans_lo=4, num_humans_hi=3), dict(num_humans_hi=7),
    dict(num_humans_lo=1, num_humans_hi=0), dict(nped=None), dict(cand_nped_prev=None), dict(cand_nped=None),
    dict(nped_out=None), dict(cand_pose=None), dict(nped_out=C.addressof(_BUF) + 256),
    dict(cand_nped=C.addressof(_BUF) + 272)],
    ids=lambda f: ','.join('%s=%s' % kv for kv in f.items()))
def test_peds_plan_rejects_bad_count_fields(fields):
    _lib.build()
    lib = _lib.load()
    launches = lib.navgym_launch_count()
    assert lib.navgym_peds_plan(C.byref(_args(**fields)), None) == 1   # cudaErrorInvalidValue
    assert lib.navgym_launch_count() == launches
