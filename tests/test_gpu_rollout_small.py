"""The small-crowd form of the rollout kernel (N <= 32) against K d2d_step launches, bit for bit, with the contract of
test_gpu_rollout.py: both sides of the N = 32 boundary, and scattered poses inside or next to walls, so that static
collisions are found at kernel entry and again after every in-kernel reset."""
import pytest

from test_gpu_rollout import test_rollout_equals_single_steps as _equals_single_steps, CASES as _CASES

pytestmark = pytest.mark.gpu

CASES = {
    # N <= 32 runs the small-crowd form, N = 33 the general one
    "n32_small_form": dict(static_map="maps/empty_map.npy", agent_number=32, agent_radius=15, agent_max_speed=20, B=512,
                           scatter=True),
    "n33_general_form": dict(static_map="maps/empty_map.npy", agent_number=33, agent_radius=15, agent_max_speed=20, B=512,
                             scatter=True),
    "walls_scattered": dict(static_map="maps/shaped_obstacle_map.npy", agent_number=10, agent_radius=10, agent_max_speed=20,
                            B=512, scatter=True),
}


@pytest.mark.parametrize("name", list(CASES))
def test_small_form_rollout_equals_single_steps(name, monkeypatch):
    monkeypatch.setitem(_CASES, name, CASES[name])
    _equals_single_steps(name)
