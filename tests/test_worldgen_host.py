"""World generation on the CPU: the host-compiled twin of the device generator (csrc/d2d_worldgen.cuh) against
world.generate_worlds, the reference's worlds restated on the host.  No GPU needed."""
import ctypes as C

import numpy as np
import pytest

import worldgen_twin as wt

SEEDS = np.concatenate([[0, 2 ** 32 - 1], np.arange(1, 1500), (np.arange(600, dtype=np.uint64) * 2654435761 + 12345) % 2 ** 32])


@pytest.mark.parametrize("name", list(wt.configs()))
def test_twin_equals_generate_worlds(name):
    """Every field of >= 2000 seeds, seeds 0 and 2**32 - 1 included.  Static-map group velocities may differ only where
    NumPy's cos / sin is not correctly rounded, and then equal speed * the correctly rounded value."""
    from gym_drone2d_activeperception_b200.world import generate_worlds
    p = wt.configs()[name]
    seeds = SEEDS.astype(np.int64)
    assert len(np.unique(seeds)) >= 2000
    host = generate_worlds(p, seeds)
    twin = wt.twin_worlds(p, seeds)
    assert not twin["failed"].any()
    exempt = wt.compare(p, seeds, host, twin, name)
    assert exempt <= 0.05 * len(seeds)
    if name == "empty":
        assert exempt == 0            # no static-map agents, no group velocities
    # the grid erasure squares with x*x where Python calls pow: no agent / cell pair lies near enough to a disc edge to care
    assert wt.near_disc_edge_count(host) == 0


def test_struct_layout_matches_header():
    from gym_drone2d_activeperception_b200 import _native
    assert wt.lib().wt_sizeof_source() == C.sizeof(_native.D2DWorldSource)


def test_world_source_contents():
    from gym_drone2d_activeperception_b200.params import Params
    from gym_drone2d_activeperception_b200.world import load_static_map, world_source
    p = Params(debug=False, static_map="maps/shaped_obstacle_map.npy", agent_number=7, agent_max_speed=20, init_pos=[60, 70])
    s = world_source(p)
    smap = load_static_map(p.static_map)
    assert np.array_equal(np.ctypeslib.as_array(s.static_map), smap.astype(np.uint8))
    assert (s.agent_number, s.pillar_number, s.init_x, s.init_y, s.map_w) == (7, 0, 60.0, 70.0, 500.0)
    h = np.ctypeslib.as_array(s.headings)[:7]
    ref = np.array([-20 * np.array([np.cos(2 * np.pi * k / 7), np.sin(2 * np.pi * k / 7)]) for k in range(7)])
    assert np.array_equal(h, ref)


def test_world_source_rejects_what_the_device_cannot_take():
    from gym_drone2d_activeperception_b200.params import Params
    from gym_drone2d_activeperception_b200.world import world_source
    bad_map = np.zeros((50, 50), np.int64)
    bad_map[3, 4] = 100
    with pytest.raises(ValueError):
        world_source(Params(debug=False), bad_map)
    with pytest.raises(ValueError):
        world_source(Params(debug=False, agent_number=257))
    with pytest.raises(ValueError):
        world_source(Params(debug=False, pillar_number=65))
    # the library checks the rest against the config (agent count, map, RVO pillar limit)
    p = Params(debug=False, static_map="maps/obstacle_map.npy", pillar_number=17, motion_profile="RVO")
    with pytest.raises(ValueError, match="16 pillars"):
        wt.twin_worlds(p, [1])


def test_impossible_configuration_is_given_up_not_looped():
    """The host generator would loop forever on a world that cannot be built; the device generator gives the seed up after
    65536 rejected draws in a row."""
    from gym_drone2d_activeperception_b200.params import Params
    p = Params(debug=False, agent_number=3, agent_radius=300)
    w = wt.twin_worlds(p, [0, 1])
    assert w["failed"].tolist() == [1, 1]
