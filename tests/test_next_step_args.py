"""CPU: BatchedNavGym's auto_reset argument is checked before any device work."""
import pytest


def test_unknown_auto_reset_mode_is_rejected():
    from nav_gym_b200 import _lib
    from nav_gym_b200.batched_env import BatchedNavGym
    assert _lib.AUTORESET_NEXT_STEP == 2
    for bad in ('bogus', 'same_step', ''):
        with pytest.raises(ValueError):
            BatchedNavGym(8, None, auto_reset=bad)
