"""Config sweeps on the device: per-env world sources (d2d_set_world_sources, d2d_generate_worlds_keyed,
d2d_set_world_queue), experiment.run_config_sweep and metrics.difficulty over a list of configs, each against the
one-config path it batches."""
import math
import re

import numpy as np
import pytest

import worldgen_twin as wt

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _P(**kw):
    from gym_drone2d_activeperception_b200.params import Params
    base = dict(debug=False, planner="NoMove", static_map="maps/empty_map.npy", agent_number=24, agent_radius=10,
                agent_max_speed=20)
    base.update(kw)
    return Params(**base)


def _family(**kw):
    """C0..C3 of one batch group (24 agents, radius 10), with `kw` applied to all."""
    return [_P(**kw), _P(agent_max_speed=40, pillar_number=3, **kw),
            _P(static_map="maps/obstacle_map.npy", agent_number=10, init_pos=[60, 60], **kw),
            _P(agent_max_speed=10, pillar_number=6, **kw)]


def _env(p, B, **kw):
    from gym_drone2d_activeperception_b200.vec_env import Drone2DVecEnv
    kw.setdefault("auto_reset", True)
    return Drone2DVecEnv(p, B, device=DEV, **kw)


def _snapshot(env, p, idx):
    """The reset snapshot of envs `idx`, shaped like world.generate_worlds for config p."""
    torch.cuda.synchronize()
    b = lambda n: env.buffer(n).cpu().numpy()
    bits = (b("gt_rows").view(np.uint64)[idx, :, None] >> np.arange(50, dtype=np.uint64)) & np.uint64(1)
    w = dict(agent_pos=b("agent_pos0")[idx], agent_pref=b("agent_pref0")[idx], agent_radius=b("agent_radius")[idx],
             tracker_radius=b("tracker_radius0")[idx], gt_grid=np.where(bits == 1, 1, 2).astype(np.uint8),
             drone_pose=b("drone_pose0").T[idx])
    if p.var_cam != 0:
        w.update(rng_key=b("rng_key0").view(np.uint32)[idx], rng_pos=b("rng_pos")[1][idx],
                 rng_has_gauss=b("rng_pos")[3][idx], rng_gauss=b("rng_gauss")[1][idx])
    if p.motion_profile == "RVO":
        n = int(p.pillar_number)
        w.update(agent_vel=b("agent_vel0")[idx], obstacles=b("rvo_obstacles")[idx, :n])
        assert (b("rvo_num_obstacles")[idx] == n).all()
        assert not b("rvo_obstacles")[idx, n:].any()
    return w


def _saved_bytes(env):
    s = env.save_state()
    torch.cuda.synchronize()
    return s["state"].cpu().numpy().tobytes()


# ------------------------------------------------------------------------------------------------ snapshots
@pytest.mark.parametrize("variant", [{}, {"motion_profile": "RVO"}, {"var_cam": 1}])
def test_mixed_keys_give_the_snapshots_of_generate_worlds(variant):
    from gym_drone2d_activeperception_b200.world import generate_worlds, split_world_key
    cfgs = _family(**variant)
    B = 2048
    rng = np.random.RandomState(5)
    sources = rng.randint(0, len(cfgs), B)
    seeds = rng.randint(0, 2 ** 32, B, dtype=np.int64)
    seeds[:2] = [0, 2 ** 32 - 1]
    env = _env(cfgs[0], B, seeds=seeds, sources=sources, world_sources=cfgs, world_gen="device")
    assert np.array_equal(split_world_key(env.seeds)[0], sources)
    for k, p in enumerate(cfgs):
        idx = np.nonzero(sources == k)[0]
        wt.compare(p, seeds[idx], generate_worlds(p, seeds[idx]), _snapshot(env, p, idx), ("source", k, variant))
    env.close()


def test_one_source_keyed_reseed_is_the_plain_reseed():
    p = _P(static_map="maps/obstacle_map.npy", agent_number=10)
    B = 64
    a = _env(p, B, seeds=np.arange(B), world_gen="device")
    b = _env(p, B, seeds=np.arange(B), world_gen="device")
    b.set_world_sources([p])
    envs, seeds = np.arange(0, B, 3), 7000 + np.arange(0, B, 3)
    a.reseed(envs, seeds)
    b.reseed(envs, seeds, sources=np.zeros(len(envs), np.int64))
    assert _saved_bytes(a) == _saved_bytes(b)
    assert np.array_equal(a.seeds, b.seeds)
    a.close()
    b.close()


# ------------------------------------------------------------------------------------------------ rows
def _rows_equal(got, ref, tag):
    assert got.keys() == ref.keys(), tag
    for c in ref:
        x, y = got[c], ref[c]
        if isinstance(y, float) and math.isnan(y):
            assert isinstance(x, float) and math.isnan(x), (tag, c, x, y)
        else:
            assert x == y, (tag, c, x, y)


def test_config_sweep_rows_equal_per_config_sweeps():
    from gym_drone2d_activeperception_b200.experiment import batch_groups, run_config_sweep, run_seed_sweep

    def configs():
        kw = dict(planner="Primitive", gaze_method="LookAhead", max_flight_time=20)
        return _family(**kw) + [_P(agent_radius=15, **kw), _P(planner="Primitive", gaze_method="Oxford", max_flight_time=20)]

    seeds = 11 + np.arange(96)
    assert batch_groups(configs()) == [[0, 1, 2, 3], [4], [5]]
    got = run_config_sweep(configs(), seeds, num_envs=256)        # 384 pairs of the first group through 256 envs
    assert len(got) == 6 and all(len(r) == len(seeds) for r in got)
    for k, c in enumerate(configs()):
        ref = run_seed_sweep(c, seeds, num_envs=256)
        for i, s in enumerate(seeds):
            assert got[k][i]["Map ID"] == s
            _rows_equal(got[k][i], ref[i], (k, int(s)))


def test_records_carry_the_keys_of_initial_and_queued_worlds():
    from gym_drone2d_activeperception_b200.world import split_world_key, world_key
    cfgs = _family(max_flight_time=4)
    B = 64
    init_src, init_sd = np.arange(B) % 4, 100 + np.arange(B)
    q_src, q_sd = (np.arange(3 * B) * 7) % 4, 5000 + np.arange(3 * B)
    env = _env(cfgs[0], B, seeds=init_sd, sources=init_src, world_sources=cfgs, world_gen="device")
    env.enable_episode_log(B * 16)
    env.set_seed_queue(q_sd, sources=q_src)
    act = torch.full((B,), 1.0 / 3, dtype=torch.float64, device=DEV)
    keys = []
    for _ in range(20):
        for _ in range(16):
            env.step(act)
        recs, dropped = env.read_episodes()
        assert dropped == 0
        keys += recs["seed"].tolist()
        assert np.array_equal(env.buffer("world_seed").cpu().numpy(), env.seeds)
    want = set(world_key(init_src, init_sd).tolist()) | set(world_key(q_src, q_sd).tolist())
    assert set(keys) == want
    src, sd = split_world_key(np.array(sorted(set(keys))))
    assert set(zip(src.tolist(), sd.tolist())) == set(zip(init_src.tolist(), init_sd.tolist())) | \
        set(zip(q_src.tolist(), q_sd.tolist()))
    env.close()


def test_keys_follow_reseed_clone_and_load():
    from gym_drone2d_activeperception_b200.world import world_key
    cfgs = _family()
    B = 16
    env = _env(cfgs[0], B, seeds=np.arange(B), world_sources=cfgs, sources=np.arange(B) % 4, world_gen="device")
    env.enable_episode_log(64)
    ws = lambda: env.buffer("world_seed").cpu().numpy()
    assert np.array_equal(ws(), world_key(np.arange(B) % 4, np.arange(B)))
    env.reseed([3, 4], [300, 400], lazy=True, sources=[2, 3])
    k3, k4 = world_key(2, 300), world_key(3, 400)
    assert ws()[3] == k3 and ws()[4] == k4
    env.clone_envs([3], [9])
    assert ws()[9] == k3
    saved = env.save_state([4, 9])
    env.load_state(saved, [0, 1])
    assert ws()[0] == k4 and ws()[1] == k3
    assert np.array_equal(ws(), env.seeds)
    env.close()


# ------------------------------------------------------------------------------------------------ rejected calls
def test_rejected_calls_change_nothing():
    from gym_drone2d_activeperception_b200 import _native
    from gym_drone2d_activeperception_b200.world import load_static_map, world_source
    L = _native.load()
    cfgs = _family(planner="Primitive")
    B = 16
    env = _env(cfgs[0], B, seeds=np.arange(B), world_sources=cfgs[:2], sources=np.arange(B) % 2, world_gen="device")
    env.enable_episode_log(64)
    act = torch.full((B,), 1.0 / 3, dtype=torch.float64, device=DEV)
    for _ in range(3):
        env.step(act)
    state = lambda: (_saved_bytes(env), env.stats().tolist(), env.buffer("world_seed").cpu().numpy().tolist(),
                     env.seeds.tolist())
    ref = state()
    with pytest.raises(_native.Drone2DNativeError, match="source 2 outside"):
        env.reseed([1], [5], sources=[2])                               # beyond the table of 2
    with pytest.raises(_native.Drone2DNativeError, match="source 2 outside"):
        env.set_seed_queue([5], sources=[2])
    with pytest.raises(ValueError):
        env.reseed([1, 2], [5], sources=[0, 1])                         # mismatched lengths
    with pytest.raises(ValueError):
        env.reseed([1], [5, 6], sources=[0, 1])
    with pytest.raises(ValueError):
        env.set_seed_queue([5, 6], sources=[0])
    idx = np.array([1], np.int32)
    for bad in (-1, -(2 ** 40), 2 * 2 ** 32 + 5):
        k = np.array([bad], np.int64)
        assert L.d2d_generate_worlds_keyed(env._h, idx.ctypes.data, k.ctypes.data, 1, _native.WORLD_EAGER, None) == -1
        assert L.d2d_set_world_queue(env._h, k.ctypes.data, 1, None) == -1
    assert state() == ref
    # tables the config cannot take: another N, another agent_radius, another map; 4097 sources
    for bad in (_P(agent_number=23), _P(agent_radius=15), _P(map_size=[600, 600])):
        with pytest.raises(ValueError, match="config 1 differs"):
            env.set_world_sources([cfgs[0], bad])
        srcs = (_native.D2DWorldSource * 2)(world_source(cfgs[0]), world_source(bad, load_static_map(bad.static_map)))
        assert L.d2d_set_world_sources(env._h, srcs, 2) == -1
        assert b"source 1" in L.d2d_last_error(env._h)
        assert state() == ref
    with pytest.raises(ValueError):
        env.set_world_sources([cfgs[0]] * 4097)
    many = (_native.D2DWorldSource * 4097)(*([world_source(cfgs[0])] * 4097))
    assert L.d2d_set_world_sources(env._h, many, 4097) == -1
    assert L.d2d_set_world_sources(env._h, many, 0) == -1
    assert state() == ref
    # the table is still the one of the last accepted call: source 1 builds C1's world
    env.reseed([5], [77], sources=[1])
    other = _env(cfgs[1], 1, seeds=[77], world_gen="device")
    a, b = _snapshot(env, cfgs[1], [5]), _snapshot(other, cfgs[1], [0])
    for key in a:
        assert np.array_equal(a[key], b[key]), key
    other.close()
    env.close()
    # a keyed queue without the episode log
    h = _env(cfgs[0], B, seeds=np.arange(B), world_sources=cfgs, world_gen="device")
    with pytest.raises(_native.Drone2DNativeError, match="not enabled"):
        h.set_seed_queue([1, 2], sources=[1, 3])
    h.close()


def test_unbuildable_world_names_env_seed_and_source():
    from gym_drone2d_activeperception_b200 import _native
    ok = _P(agent_number=200)
    bad = _P(agent_number=200, pillar_number=64)                       # same config: the pillars only shape the world
    seeds = np.arange(64)
    failed = wt.twin_worlds(bad, seeds)["failed"]
    assert failed.any() and not wt.twin_worlds(ok, seeds[:4])["failed"].any()
    s = int(seeds[np.nonzero(failed)[0][0]])
    env = _env(ok, 4, seeds=np.arange(4), world_sources=[ok, bad], world_gen="device")
    env.reseed([3], [s], sources=[1])
    torch.cuda.synchronize()
    # a pending failure is reported before the arguments of the next call are looked at, even an out-of-range seed
    with pytest.raises(_native.Drone2DNativeError, match=r"seed %d from source 1 \(env 3\) could not be built" % s):
        env.reseed([0], [2 ** 32])
    env.check_worlds()                                                  # reported once
    # several unbuildable worlds in one launch: one of them is reported, with its own env
    bad_seeds = seeds[np.nonzero(failed)[0][:3]]
    env.reseed([1, 2, 3], bad_seeds, sources=[1, 1, 1])
    torch.cuda.synchronize()
    with pytest.raises(_native.Drone2DNativeError) as err:
        env.check_worlds()
    m = re.search(r"seed (\d+) from source 1 \(env (\d+)\)", str(err.value))
    assert m and (int(m.group(1)), int(m.group(2))) in {(int(sd), e) for sd, e in zip(bad_seeds, (1, 2, 3))}, str(err.value)
    env.check_worlds()
    env.close()


# ------------------------------------------------------------------------------------------------ difficulty
def test_difficulty_over_configs_equals_per_config_calls():
    from gym_drone2d_activeperception_b200 import metrics
    cfgs = lambda: _family() + [_P(agent_radius=15)]
    seeds = 40 + np.arange(100)
    got = metrics.difficulty(cfgs(), seeds, num_envs=256, collision_state=True)   # 400 pairs: keyed reseed chunks
    ref = [metrics.difficulty(c, seeds, num_envs=256, collision_state=True) for c in cfgs()]
    assert set(got) == set(ref[0])
    for key in ref[0]:
        want = np.stack([r[key] for r in ref])
        assert got[key].shape == want.shape and got[key].dtype == want.dtype, key
        assert np.array_equal(got[key], want), key
    with pytest.raises(ValueError):
        metrics.difficulty(cfgs(), seeds, world_gen="host")
    with pytest.raises(ValueError):
        metrics.difficulty([], seeds)
