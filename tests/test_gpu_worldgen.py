"""Worlds generated on the GPU (d2d_set_world_source / d2d_generate_worlds, Drone2DVecEnv(world_gen="device"), reseed,
experiment.run_seed_sweep) against worlds built by world.generate_worlds on the host and uploaded with d2d_set_world.

The one documented difference: static-map group velocities where NumPy's cos / sin is not correctly rounded ("exempt"
envs, checked by worldgen_twin.compare: the device then holds speed * the correctly rounded value)."""
import json
import math
import os

import numpy as np
import pytest

import worldgen_twin as wt

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

DEV = "cuda:0"
# per-env buffers with the env on axis 0 (allocated under every configuration)
AXIS0 = ["agent_pos", "agent_pref", "agent_pos0", "agent_pref0", "agent_radius", "tracker_radius0", "gt_rows", "belief",
         "env_records", "collision_flag", "dead_lock_flag", "freezing_flag", "done", "local_map", "yaw_angle", "hit",
         "tracker_active", "tracker_mu", "tracker_sigma", "tracker_radius", "tracker_ts", "need_plan", "plan_ok", "replan",
         "oxford_calls", "owl_queue_len", "owl_queue_value", "drone_acc"]
CONTINUOUS = {"agent_pos", "agent_pref", "agent_pos0", "agent_pref0", "agent_vel", "agent_vel0", "tracker_mu", "tracker_sigma",
              "drone_acc", "traj_coeff", "owl_U", "owl_queue_value"}


def _env(p, B, **kw):
    from gym_drone2d_activeperception_b200.vec_env import Drone2DVecEnv
    kw.setdefault("auto_reset", True)
    return Drone2DVecEnv(p, B, device=DEV, **kw)


def _names(env):
    c = env.cfg
    names = list(AXIS0)
    if c.motion_profile == 1:
        names += ["agent_vel", "agent_vel0", "rvo_obstacles", "rvo_num_obstacles"]
    if c.planner == 1:
        names.append("traj_coeff")
    if c.var_cam != 0:
        names += ["rng_key", "rng_key0"]
    if c.oxford & 2:
        names.append("owl_U")
    return names


def _state(env, envs=None):
    """Every per-env state buffer (+ the [planes, B] RNG scalars and the reset pose) as host arrays, env on axis 0."""
    torch.cuda.synchronize()
    out = {n: env.buffer(n).cpu().numpy() for n in _names(env)}
    for n in ("rng_pos", "rng_gauss", "drone_pose0"):
        out[n] = env.buffer(n).cpu().numpy().T
    if envs is not None:
        out = {k: v[np.asarray(envs)] for k, v in out.items()}
    return out


def _assert_same(a, b, tag, tol_envs=()):
    """Bit-identical, except that envs in `tol_envs` may differ by 1e-9 (relative) in continuous buffers."""
    tol = np.zeros(len(a["done"]), bool)
    tol[list(tol_envs)] = True
    for k in a:
        x, y = a[k], b[k]
        if x.dtype.kind == "f":
            same = (x.view(np.int64 if x.itemsize == 8 else np.int32) == y.view(np.int64 if x.itemsize == 8 else np.int32))
            same = same.reshape(len(x), -1).all(1)
        else:
            same = (x == y).reshape(len(x), -1).all(1)
        bad = ~same & ~tol
        assert not bad.any(), (tag, k, np.nonzero(bad)[0][:8])
        if tol.any() and not same.all():
            assert k in CONTINUOUS, (tag, k, "discrete mismatch in an exempt env", np.nonzero(~same)[0][:8])
            xx, yy = x[tol].astype(np.float64), y[tol].astype(np.float64)
            assert np.all(np.abs(xx - yy) <= 1e-9 * np.maximum(1.0, np.abs(yy))), (tag, k)


def _device_world(env, p):
    """The reset snapshot of every env in the arena, shaped like world.generate_worlds."""
    torch.cuda.synchronize()
    b = lambda n: env.buffer(n).cpu().numpy()
    bits = (b("gt_rows").view(np.uint64)[:, :, None] >> np.arange(50, dtype=np.uint64)) & np.uint64(1)
    w = dict(agent_pos=b("agent_pos0"), agent_pref=b("agent_pref0"), agent_radius=b("agent_radius"),
             tracker_radius=b("tracker_radius0"), gt_grid=np.where(bits == 1, 1, 2).astype(np.uint8),
             drone_pose=b("drone_pose0").T.copy())
    if p.var_cam != 0:
        w.update(rng_key=b("rng_key0").view(np.uint32), rng_pos=b("rng_pos")[1], rng_has_gauss=b("rng_pos")[3],
                 rng_gauss=b("rng_gauss")[1])
    if p.motion_profile == "RVO":
        w.update(agent_vel=b("agent_vel0"), obstacles=b("rvo_obstacles")[:, :int(p.pillar_number)])
        assert (b("rvo_num_obstacles") == int(p.pillar_number)).all()
        assert not b("rvo_obstacles")[:, int(p.pillar_number):].any()
    return w


def _exempt(p, seeds):
    """Envs whose seed falls under the group-velocity exception (device worlds differ from generate_worlds there)."""
    from gym_drone2d_activeperception_b200.world import generate_worlds
    host, twin = generate_worlds(p, seeds), wt.twin_worlds(p, seeds)
    return set(np.nonzero((host["agent_pref"] != twin["agent_pref"]).any(axis=(1, 2)))[0].tolist())


# ------------------------------------------------------------------------------------------------ snapshots
@pytest.mark.parametrize("name", list(wt.configs()))
def test_device_snapshot_equals_generate_worlds(name):
    from gym_drone2d_activeperception_b200.world import generate_worlds
    p = wt.configs()[name]
    B = 4096
    seeds = np.concatenate([[0, 2 ** 32 - 1], 1000 + np.arange(B - 2)]).astype(np.int64)
    env = _env(p, B, seeds=seeds, world_gen="device")
    dev = _device_world(env, p)
    wt.compare(p, seeds, generate_worlds(p, seeds), dev, name)
    assert np.array_equal(env.seeds, seeds)
    env.close()


def test_device_snapshot_equals_twin_65536_random_map():
    p = wt.configs()["random0"]
    B = 65536
    seeds = np.arange(B, dtype=np.int64) * 7919 + 3
    env = _env(p, B, seeds=seeds, world_gen="device")
    dev, twin = _device_world(env, p), wt.twin_worlds(p, seeds)
    assert not twin["failed"].any()
    for k in ("agent_pos", "agent_pref", "agent_radius", "tracker_radius", "gt_grid", "drone_pose"):
        assert np.array_equal(dev[k], twin[k]), k
    env.close()


# ------------------------------------------------------------------------------------------------ stepping side by side
def _step_cases():
    from gym_drone2d_activeperception_b200.params import Params
    P = lambda **kw: Params(**dict(dict(debug=False, agent_number=10, agent_radius=15, agent_max_speed=20), **kw))
    return {
        "nomove_random0": (P(planner="NoMove", static_map="maps/random_map_0.npy"), "scripted"),
        "primitive_oxford": (P(planner="Primitive", gaze_method="Oxford", static_map="maps/shaped_obstacle_map.npy"), "Oxford"),
        "owl": (P(planner="Primitive", gaze_method="Owl", static_map="maps/obstacle_map.npy"), "Owl"),
        "jerk": (P(planner="Jerk_Primitive", gaze_method="LookGoal"), "LookGoal"),
        "rvo": (P(planner="NoMove", motion_profile="RVO", pillar_number=6, static_map="maps/obstacle_map.npy"), "scripted"),
        "noise": (P(planner="NoMove", var_cam=1, static_map="maps/random_map_0.npy"), "scripted"),
    }


@pytest.mark.parametrize("case", list(_step_cases()))
def test_host_and_device_worlds_step_identically(case):
    """300 steps of a host-world batch and a device-world batch of the same seeds: bit-identical everywhere outside the
    exempt envs.  On random_map_0 the exempt envs are included too: no discrete mismatch, continuous state within 1e-9."""
    p, policy = _step_cases()[case]
    B = 256
    seeds = 40 + np.arange(B)
    ex = _exempt(p, seeds)
    a = _env(p, B, seeds=seeds)
    d = _env(p, B, seeds=seeds, world_gen="device")
    keep = [i for i in range(B) if i not in ex]
    include_exempt = case == "nomove_random0"
    rng = np.random.RandomState(1)
    table = torch.as_tensor(np.arange(-80, 80, 80 / 3) / 80, device=DEV)
    for t in range(300):
        if policy == "scripted":
            acts = [table[torch.as_tensor(rng.randint(0, 6, B), device=DEV)]] * 2
        else:
            acts = [e.plan_gaze(policy) for e in (a, d)]
        a.step(acts[0])
        d.step(acts[1])
        if t % 50 == 49 or t == 299:
            if include_exempt:
                _assert_same(_state(d), _state(a), (case, t), tol_envs=sorted(ex))
            else:
                _assert_same(_state(d, keep), _state(a, keep), (case, t))
    assert np.array_equal(a.stats(), d.stats())
    a.close()
    d.close()


# ------------------------------------------------------------------------------------------------ reseed
def test_lazy_reseed_on_done_equals_a_fresh_env():
    from gym_drone2d_activeperception_b200.params import Params
    p = Params(debug=False, planner="NoMove", agent_number=10, agent_radius=15, agent_max_speed=20, max_flight_time=3,
               static_map="maps/random_map_0.npy")
    B = 64
    act = torch.full((B,), 1.0 / 3, dtype=torch.float64, device=DEV)
    seeds_in = np.arange(B)
    a = _env(p, B, seeds=seeds_in, world_gen="device")
    for _ in range(200):
        a.step(act)
        done = a.buffer("done").cpu().numpy().astype(bool)
        if done.any():
            break
    D = np.nonzero(done)[0]
    assert len(D)
    new = 5000 + D
    before = _state(a, D)
    stats = a.stats()
    a.reseed(D, new, lazy=True)
    after = _state(a, D)
    for k in ("done", "local_map", "yaw_angle", "belief", "collision_flag", "agent_pos", "hit"):     # terminal outputs stay
        assert np.array_equal(after[k], before[k]), k
    assert (a.buffer("pending_reset").cpu().numpy()[D] == 1).all()
    assert np.array_equal(seeds_in, np.arange(B))           # env.seeds is the env's own copy
    assert np.array_equal(a.seeds[D], new)
    assert np.array_equal(a.stats(), stats)
    seeds_c = a.seeds.copy()
    c = _env(p, B, seeds=seeds_c)            # control: fresh envs of those seeds, host-built worlds
    ex = _exempt(p, new)
    D_ok = [int(e) for k, e in enumerate(D) if k not in ex]
    for t in range(60):
        a.step(act)
        c.step(act)
        _assert_same(_state(a, D_ok), _state(c, D_ok), ("lazy reseed", t))
    a.close()
    c.close()


def test_eager_reseed_equals_set_world_and_reset():
    from gym_drone2d_activeperception_b200.world import generate_worlds
    for name in ("rvo_pillars", "noise"):
        p = wt.configs()[name]
        B = 48
        seeds = np.arange(B)
        a = _env(p, B, seeds=seeds, world_gen="device")
        c = _env(p, B, seeds=seeds, world_gen="device")
        act = torch.full((B,), -1.0 / 3, dtype=torch.float64, device=DEV)
        for _ in range(7):
            a.step(act)
            c.step(act)
        envs = np.array([3, 17, 40, 5])
        new = np.array([900, 901, 902, 2 ** 32 - 1])
        a.reseed(envs, new)
        keys = generate_worlds(p, new[:1]).keys()
        w_dev = wt.twin_worlds(p, new)              # what the device builds (generate_worlds outside the exception)
        for k, e in enumerate(envs):
            c.set_worlds({key: w_dev[key][k:k + 1] for key in keys}, first_env=int(e))
        for _ in range(5):
            _assert_same(_state(a), _state(c), (name, "eager"))
            a.step(act)
            c.step(act)
        a.close()
        c.close()


def test_reseeded_state_saves_and_loads_into_another_handle():
    p = wt.configs()["noise"]
    B = 32
    a = _env(p, B, seeds=np.arange(B), world_gen="device")
    act = torch.full((B,), 1.0 / 3, dtype=torch.float64, device=DEV)
    for _ in range(4):
        a.step(act)
    a.reseed([1, 2, 3], [77, 78, 79], lazy=True)
    a.reseed([10, 11], [80, 81])
    saved = a.save_state()
    b = _env(p, B, seeds=100 + np.arange(B))
    b.load_state(saved)
    assert np.array_equal(a.seeds, b.seeds)
    for t in range(40):
        _assert_same(_state(a), _state(b), ("load", t))
        a.step(act)
        b.step(act)
    a.close()
    b.close()


def _saved_bytes(env):
    s = env.save_state()
    torch.cuda.synchronize()
    return s["state"].cpu().numpy().tobytes()


def test_rejected_calls_change_nothing_and_statistics_stay():
    from gym_drone2d_activeperception_b200 import _native
    p = wt.configs()["rvo_pillars"]
    B = 16
    env = _env(p, B, seeds=np.arange(B), world_gen="device")
    act = torch.full((B,), 1.0 / 3, dtype=torch.float64, device=DEV)
    for _ in range(3):
        env.step(act)
    ref, st = _saved_bytes(env), env.stats()
    seeds_before = env.seeds.copy()
    for envs, seeds in (([B], [1]), ([-1], [1]), ([2, 2], [1, 2]), ([1], [-1]), ([1], [2 ** 32]), ([1, 2], [3])):
        with pytest.raises((_native.Drone2DNativeError, ValueError)):
            env.reseed(envs, seeds)
        assert _saved_bytes(env) == ref, (envs, seeds)
    L = _native.load()
    import ctypes as C
    idx, sd = np.array([1], np.int32), np.array([5], np.int64)
    for flags in (0, 3, 4):
        rc = L.d2d_generate_worlds(env._h, idx.ctypes.data, sd.ctypes.data, 1, flags, None)
        assert rc == -1
        assert _saved_bytes(env) == ref
    assert np.array_equal(env.seeds, seeds_before)
    assert np.array_equal(env.stats(), st)
    # a handle without a world source refuses generation (call sequence)
    h = _env(p, B, seeds=np.arange(B))
    rc = L.d2d_generate_worlds(h._h, idx.ctypes.data, sd.ctypes.data, 1, _native.WORLD_EAGER, None)
    assert rc == -4
    h.close()
    # reseeds (eager and lazy) leave the statistics alone
    env.reseed([0, 1], [50, 51])
    env.reseed([2], [52], lazy=True)
    assert np.array_equal(env.stats(), st)
    assert C.sizeof(_native.D2DWorldSource) == wt.lib().wt_sizeof_source()
    env.close()


def test_host_mirror_is_refreshed_after_an_eager_reseed():
    p = wt.configs()["empty"]
    B = 16
    env = _env(p, B, seeds=np.arange(B), world_gen="device")
    lm = torch.zeros((B, 1, 33, 33), dtype=torch.uint8).pin_memory()
    yaw = torch.zeros(B, dtype=torch.float32).pin_memory()
    dn = torch.zeros(B, dtype=torch.uint8).pin_memory()
    env.bind_host_mirror(lm, yaw, dn)
    a = np.full(B, 1.0 / 3)
    for _ in range(5):
        env.step_host(a, lm, yaw, dn)
    env.reseed([2, 9], [300, 301])
    env.step_host(a, lm, yaw, dn)
    torch.cuda.synchronize()
    assert np.array_equal(lm.numpy(), env.buffer("local_map").cpu().numpy())
    assert np.array_equal(yaw.numpy(), env.buffer("yaw_angle").cpu().numpy().reshape(-1))
    assert np.array_equal(dn.numpy(), env.buffer("done").cpu().numpy())
    env.close()


def test_reseed_refused_while_a_pipelined_step_is_in_flight():
    from gym_drone2d_activeperception_b200 import _native
    p = wt.configs()["empty"]
    B = 32
    env = _env(p, B, seeds=np.arange(B), world_gen="device")
    lm = torch.zeros((B, 1, 33, 33), dtype=torch.uint8).pin_memory()
    yaw = torch.zeros(B, dtype=torch.float32).pin_memory()
    dn = torch.zeros(B, dtype=torch.uint8).pin_memory()
    a_pin = torch.full((B,), 1.0 / 3, dtype=torch.float64).pin_memory()
    env.bind_host_io(a_pin, lm, yaw, dn)
    env.step_pipelined(True)
    env.step_pipelined(True)
    with pytest.raises(_native.Drone2DNativeError, match=r"\(-4\)"):
        env.reseed([0], [1])
    env.step_pipelined(False)
    env.reseed([0], [1])
    env.close()


def test_impossible_world_is_reported():
    from gym_drone2d_activeperception_b200 import _native
    from gym_drone2d_activeperception_b200.params import Params
    p = Params(debug=False, planner="NoMove", agent_number=3, agent_radius=300)
    with pytest.raises(_native.Drone2DNativeError, match="could not be built"):
        _env(p, 4, seeds=[0, 1, 2, 3], world_gen="device")
    with pytest.raises(ValueError):
        _env(p, 4, worlds={}, world_gen="device")


# ------------------------------------------------------------------------------------------------ seed sweep
def _rows_equal(got, ref, tag):
    from gym_drone2d_activeperception_b200.experiment import CSV_COLUMNS
    for c in CSV_COLUMNS:
        a, b = got[c], ref[c]
        if c in ("Initial position", "Target position"):
            assert str(list(a)) == str(b) or list(a) == list(b), (tag, c, a, b)
        elif isinstance(b, float) and math.isnan(b):
            assert isinstance(a, float) and math.isnan(a), (tag, c, a, b)
        elif c in ("Flight time", "Agent tracked time"):
            assert abs(a - b) <= 1e-12 * max(1.0, abs(b)), (tag, c, a, b)
        else:
            assert a == b, (tag, c, a, b)


def test_seed_sweep_equals_one_env_per_seed():
    from gym_drone2d_activeperception_b200.experiment import run_batched_rows, run_seed_sweep
    from gym_drone2d_activeperception_b200.params import Params
    kw = dict(debug=False, gaze_method="LookAhead", planner="Primitive", agent_number=10, agent_radius=15, agent_max_speed=20)
    seeds = 3 + np.arange(256)
    sweep = run_seed_sweep(Params(**kw), seeds, 32)
    assert np.array_equal(seeds, 3 + np.arange(256))        # the caller's seed list is not written to
    ref = run_batched_rows(Params(**kw), 256, episodes=1, seeds=seeds)
    by_env = {r["_env"]: r for r in ref}
    assert len(sweep) == 256 and len(by_env) == 256
    for k, s in enumerate(seeds):
        assert sweep[k]["Map ID"] == s
        _rows_equal(sweep[k], by_env[k], ("sweep", int(s)))


def test_seed_sweep_matches_reference_rows():
    from gym_drone2d_activeperception_b200.experiment import run_seed_sweep
    from gym_drone2d_activeperception_b200.params import Params
    with open(os.path.join(os.path.dirname(__file__), "golden", "experiment_rows.json")) as f:
        cases = json.load(f)["rows"]
    groups = {}
    for c in cases:
        kw = dict(agent_number=10, agent_radius=15, agent_max_speed=20, drone_max_speed=40, static_map="maps/empty_map.npy")
        kw.update(c["params"])
        seed = kw.pop("map_id")
        groups.setdefault(json.dumps(kw, sort_keys=True), []).append((seed, c["row"]))
    for key, items in groups.items():
        kw = json.loads(key)
        rows = run_seed_sweep(Params(debug=False, **kw), [s for s, _ in items], 2)
        for (s, ref), got in zip(items, rows):
            _rows_equal(got, ref, (kw["gaze_method"], s))
