"""Config sweeps on the host: world keys (world.world_key / split_world_key), the batch grouping of experiment.batch_groups
and the config comparison behind Drone2DVecEnv.set_world_sources.  No GPU needed."""
import numpy as np
import pytest

from gym_drone2d_activeperception_b200.params import Params
from gym_drone2d_activeperception_b200.world import split_world_key, world_key


def _P(**kw):
    base = dict(debug=False, static_map="maps/empty_map.npy", agent_number=24, agent_radius=10, agent_max_speed=20)
    base.update(kw)
    return Params(**base)


def test_world_key_round_trips_at_the_edges():
    src = np.array([0, 0, 1, 4095, 4095, 17], np.int64)
    sd = np.array([0, 2 ** 32 - 1, 0, 0, 2 ** 32 - 1, 12345], np.int64)
    k = world_key(src, sd)
    assert k.dtype == np.int64
    assert k[0] == 0 and k[1] == 2 ** 32 - 1 and k[2] == 2 ** 32 and k[4] == 4096 * 2 ** 32 - 1
    s2, d2 = split_world_key(k)
    assert np.array_equal(s2, src) and np.array_equal(d2, sd)
    assert np.array_equal(world_key(0, sd), sd)                      # source 0: the key is the seed
    assert np.array_equal(world_key(np.uint32(3), np.uint64(7)), 3 * 2 ** 32 + 7)


@pytest.mark.parametrize("sources,seeds", [([4096], [0]), ([-1], [0]), ([0], [2 ** 32]), ([0], [-1]), ([0.5], [1]),
                                           ([0], [1.0])])
def test_world_key_rejects_out_of_range(sources, seeds):
    with pytest.raises(ValueError):
        world_key(np.array(sources), np.array(seeds))


@pytest.mark.parametrize("keys", [[-1], [4096 * 2 ** 32], [1.5]])
def test_split_world_key_rejects_out_of_range(keys):
    with pytest.raises(ValueError):
        split_world_key(np.array(keys))


def test_batch_groups_partition_in_input_order():
    from gym_drone2d_activeperception_b200.experiment import batch_groups
    cfgs = [
        _P(),                                                                     # 0  C0
        _P(agent_radius=15),                                                      # 1  other agent_radius
        _P(agent_max_speed=40, pillar_number=3),                                  # 2  C1
        _P(static_map="maps/obstacle_map.npy", agent_number=10, init_pos=[60, 60]),   # 3  C2: 14 static + 10
        _P(gaze_method="Oxford"),                                                 # 4  other gaze
        _P(agent_max_speed=10, pillar_number=6),                                  # 5  C3
        _P(agent_number=23),                                                      # 6  other N
        _P(drone_max_speed=20),                                                   # 7  other drone speed
        _P(agent_radius=15, pillar_number=2),                                     # 8  with 1
        _P(gaze_method="NoControl"),                                              # 9
        _P(gaze_method="NoControl", drone_view_range=120),                        # 10 same view after the NoControl rule
        _P(gaze_method="Oxford", agent_max_speed=33),                             # 11 with 4
    ]
    groups = batch_groups(cfgs)
    assert groups == [[0, 2, 3, 5], [1, 8], [4, 11], [6], [7], [9, 10]]
    assert cfgs[10].drone_view_range == 120                                      # the caller's configs are not written to
    assert batch_groups([]) == []


def test_config_difference_names_the_first_field():
    from gym_drone2d_activeperception_b200.vec_env import config_difference, make_config
    a = make_config(_P(), 8, 24, 0)
    assert config_difference(a, make_config(_P(agent_max_speed=7, pillar_number=5), 8, 24, 0)) is None
    assert config_difference(a, make_config(_P(agent_radius=15), 8, 24, 0)) == "agent_radius"
    assert config_difference(a, make_config(_P(), 8, 25, 0)) == "num_agents"
    assert config_difference(a, make_config(_P(target_list=[[60, 460]]), 8, 24, 0)) == "targets"
