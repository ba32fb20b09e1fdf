"""d2d_difficulty / metrics.difficulty on the device: the reference's goldens, the existing step-kernel metrics
(global_survivability, survivability, obstacle_density) on >= 512 seeds per configuration, device worlds, chunking,
read-only-ness, graph capture, a 65 536-world call and rejected calls."""
import ctypes as C

import numpy as np
import pytest

import test_difficulty_host as th

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _P(**kw):
    from gym_drone2d_activeperception_b200.params import Params
    return Params(**dict(dict(debug=False, planner="NoMove", gaze_method="NoControl"), **kw))


def test_reference_goldens():
    """metrics_survivability.npz (T = 6, two configs, densities) and metrics_global_survivability.npz (T = 24 with its
    doubled slots, position step 120), written by the unmodified reference."""
    import json
    import os
    from gym_drone2d_activeperception_b200.metrics import difficulty
    here = os.path.join(os.path.dirname(__file__), "golden")
    g = np.load(os.path.join(here, "metrics_survivability.npz"))
    T, seeds = int(g["T"]), g["seeds"].tolist()
    for ci, c in enumerate(json.loads(str(g["cases"]))):
        r = difficulty(_P(**c), seeds, T_survivability=T, world_gen="host", device=DEV)
        assert np.array_equal(r["survivability"], g["survive_%d" % ci]), c
        assert np.array_equal(r["mean_survivability"], g["survive_%d" % ci].reshape(len(seeds), -1).mean(1))
        assert np.array_equal(r["density"], g["density_%d" % ci])
    g = np.load(os.path.join(here, "metrics_global_survivability.npz"))
    r = difficulty(_P(**json.loads(str(g["params"]))), [int(g["seed"])], T_global=int(g["T"]),
                   position_step=int(g["position_step"]), world_gen="host", collision_state=True, device=DEV)
    assert r["collision_state"].shape[1:] == g["collision_state"].shape
    assert np.array_equal(r["collision_state"][0], g["collision_state"])


def _near_boundary_positions(p, seeds, xs, ys, T_surv):
    """bool [S, nx, ny]: positions with an (agent, step) pair whose distance lies within 1e-12 (relative) of
    r + drone_r during the survivability loop -- where the torch restatement's sqrt(dx*dx+dy*dy) and the reference's
    np.linalg.norm may disagree.  Trajectories from the host twin (held to the oracle by the CPU tests)."""
    from gym_drone2d_activeperception_b200.world import generate_worlds
    w = generate_worlds(p, seeds)
    L = len(np.arange(0, T_surv, 0.1))
    gx, gy = np.meshgrid(np.asarray(xs, float), np.asarray(ys, float), indexing="ij")
    out = np.zeros((len(seeds), len(xs), len(ys)), bool)
    for i in range(len(seeds)):
        tr = th.twin_trajectory(p, w["agent_pos"][i], w["agent_pref"][i], w["agent_radius"][i], L)     # [L, N, 2]
        R = w["agent_radius"][i] + p.drone_radius
        d = np.sqrt((tr[:, :, 0, None, None] - gx) ** 2 + (tr[:, :, 1, None, None] - gy) ** 2)   # [L, N, nx, ny]
        out[i] = (np.abs(d - R[None, :, None, None]) <= 1e-12 * R[None, :, None, None]).any((0, 1))
    return out


CONFIGS = {
    "empty": (dict(agent_number=20, agent_radius=15), 60),
    "obstacle": (dict(static_map="maps/obstacle_map.npy", agent_number=30, agent_radius=20), 60),
    "random0_pillars": (dict(static_map="maps/random_map_0.npy", pillar_number=8), 60),
    "shaped": (dict(static_map="maps/shaped_obstacle_map.npy", agent_number=12), 60),
    "random_radius": (dict(agent_radius=-1, agent_number=25), 60),
    "slow": (dict(agent_max_speed=4, agent_number=20, agent_radius=25), 60),
    "step30": (dict(static_map="maps/obstacle_map.npy", agent_number=20), 30),
}


@pytest.mark.parametrize("name", list(CONFIGS))
def test_equals_step_kernel_metrics(name):
    """512 seeds: collision_state, global survival time and density exactly; survivability exactly except at positions
    with a pair within 1e-12 of the boundary (counted and reported; none expected)."""
    from gym_drone2d_activeperception_b200.metrics import (difficulty, global_survivability, mean_survival_time,
                                                           obstacle_density, survivability, survivability_positions)
    kw, step = CONFIGS[name]
    p = _P(**kw)
    seeds = np.arange(1000, 1512)
    r = difficulty(p, seeds, position_step=step, world_gen="host", collision_state=True, num_envs=200, device=DEV)
    cs = global_survivability(p, seeds, T=24, position_step=step, device=DEV)
    assert np.array_equal(r["collision_state"], cs)
    assert np.array_equal(r["global_survival_time"], mean_survival_time(cs))
    assert np.array_equal(r["density"], obstacle_density(p, seeds))
    st, mean = survivability(p, seeds, T=12, position_step=step, device=DEV)
    xs, ys = survivability_positions(p, step)
    near = _near_boundary_positions(p, seeds, xs, ys, 12)
    bad = r["survivability"] != st
    print("%s: %d positions near the boundary, %d differ" % (name, int(near.sum()), int(bad.sum())))
    assert not (bad & ~near).any()
    assert np.array_equal(r["mean_survivability"][~bad.any((1, 2))], mean[~bad.any((1, 2))])
    assert cs.any() and (r["survivability"] < 12 - 0.1).any()


def test_device_worlds():
    """world_gen="device" equals world_gen="host" except on seeds whose static-map group velocities fall in the documented
    1-ulp set (found by comparing the device snapshots with generate_worlds)."""
    from gym_drone2d_activeperception_b200.metrics import difficulty
    from gym_drone2d_activeperception_b200.vec_env import Drone2DVecEnv
    from gym_drone2d_activeperception_b200.world import generate_worlds
    p = _P(static_map="maps/random_map_0.npy", pillar_number=4)
    seeds = np.arange(4096)
    rh = difficulty(p, seeds, world_gen="host", collision_state=True, device=DEV)
    rd = difficulty(p, seeds, world_gen="device", collision_state=True, device=DEV)
    env = Drone2DVecEnv(p, len(seeds), seeds=seeds, device=DEV, auto_reset=False, trackers=False, world_gen="device")
    w = generate_worlds(p, seeds)
    same = ((env.buffer("agent_pref0").cpu().numpy() == w["agent_pref"]).all((1, 2)) &
            (env.buffer("agent_pos0").cpu().numpy() == w["agent_pos"]).all((1, 2)))
    env.close()
    assert same.sum() >= 0.9 * len(seeds)
    for k in rh:
        assert np.array_equal(rd[k][same], rh[k][same]), k


def test_chunking():
    """10 000 seeds through a 4096-env handle equal one call over all of them (the planner of the params does not matter:
    the scratch handle is NoMove)."""
    from gym_drone2d_activeperception_b200.metrics import difficulty
    p = _P(agent_number=15)
    seeds = np.arange(50000, 60000)
    a = difficulty(p, seeds, num_envs=4096, collision_state=True, device=DEV)
    b = difficulty(_P(agent_number=15, planner="Primitive", gaze_method="Oxford"), seeds, num_envs=len(seeds),
                   collision_state=True, device=DEV)
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def _env(p, B, **kw):
    from gym_drone2d_activeperception_b200.vec_env import Drone2DVecEnv
    return Drone2DVecEnv(p, B, device=DEV, **kw)


def _saved(env):
    torch.cuda.synchronize()
    return env.save_state()["state"].cpu().numpy()


GRID = (20, 20, 60, 8, 8)


def _host(res):
    return {k: v.cpu().numpy() for k, v in res.items()}


def test_handle_method_reads_the_snapshot_only():
    from gym_drone2d_activeperception_b200.metrics import global_slots
    p = _P(static_map="maps/shaped_obstacle_map.npy", max_flight_time=8)
    B, T = 64, 200
    n_slots, table = global_slots(24, p.dt, 240)
    envs = [_env(p, B, world_gen="device") for _ in range(2)]
    for e in envs:
        e.enable_episode_log(B * T)
    first = _host(envs[0].difficulty(240, GRID, slots=table, n_slots=n_slots, collision_state=True))
    acts = (np.arange(-80, 80, 80 / 3) / 80)[np.random.RandomState(3).randint(0, 6, (T, B))]
    for t in range(T):
        for k, e in enumerate(envs):
            e.step(torch.as_tensor(acts[t], device=DEV))
            if k == 0 and t % 7 == 0:
                got = _host(e.difficulty(240, GRID, envs=range(3, 40) if t % 2 else None, slots=table, n_slots=n_slots,
                                         collision_state=True))
                sl = slice(3, 40) if t % 2 else slice(0, B)
                for key in first:
                    assert np.array_equal(got[key], first[key][sl]), (t, key)
    assert np.array_equal(_saved(envs[0]), _saved(envs[1]))
    assert np.array_equal(envs[0].stats(), envs[1].stats())
    ra, _ = envs[0].read_episodes()
    rb, _ = envs[1].read_episodes()
    assert len(ra) > 0 and ra.tobytes() == rb.tobytes()
    for e in envs:
        e.close()
    # the host observation mirror of a bound step_host run
    envs = [_env(p, B) for _ in range(2)]
    mirrors = []
    for e in envs:
        m = (torch.zeros((B, 1, 33, 33), dtype=torch.uint8).pin_memory(),
             torch.zeros((B, 1), dtype=torch.float32).pin_memory(), torch.zeros(B, dtype=torch.uint8).pin_memory())
        e.bind_host_mirror(*m)
        mirrors.append(m)
    for t in range(50):
        for k, e in enumerate(envs):
            e.step_host(np.ascontiguousarray(acts[t]), *mirrors[k])
            if k == 0:
                e.difficulty(100, GRID)
    for a, b in zip(*mirrors):
        assert torch.equal(a, b)
    assert np.array_equal(_saved(envs[0]), _saved(envs[1]))
    for e in envs:
        e.close()


def test_graph_capture_equals_eager():
    p = _P(agent_number=30)
    B = 512
    env = _env(p, B, world_gen="device", auto_reset=False)
    eager = _host(env.difficulty(240, GRID, collision_state=True))
    out = (torch.zeros((B, 8, 8), dtype=torch.int16, device=DEV), torch.zeros((B, 8, 8), dtype=torch.uint8, device=DEV),
           torch.zeros((B, 8, 8, 240), dtype=torch.uint8, device=DEV))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        env.difficulty(240, GRID, collision_state=True, out=out)          # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    for t in out:
        t.zero_()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        env.difficulty(240, GRID, collision_state=True, out=out)
    g.replay()
    torch.cuda.synchronize()
    for k, t in zip(("first_hit", "static_hit", "collision_state"), out):
        assert np.array_equal(t.cpu().numpy(), eager[k]), k
    env.close()


def test_65536_worlds_one_call():
    """One call over 65 536 device worlds; 64 sampled envs equal the host twin and the NumPy static probes."""
    p = _P(static_map="maps/random_map_0.npy", agent_number=10)
    B = 65536
    env = _env(p, B, world_gen="device", auto_reset=False, trackers=False)
    r = _host(env.difficulty(240, GRID))
    pos0, pref0 = env.buffer("agent_pos0").cpu().numpy(), env.buffer("agent_pref0").cpu().numpy()
    rad, rows = env.buffer("agent_radius").cpu().numpy(), env.buffer("gt_rows").cpu().numpy()
    env.close()
    xs = [20 + 60 * i for i in range(8)]
    for e in np.random.RandomState(5).choice(B, 64, replace=False).tolist():
        assert np.array_equal(r["first_hit"][e], th.twin_first_hit(p, pos0[e], pref0[e], rad[e], GRID, 240)), e
        gt = np.where((rows[e].astype(np.uint64)[:, None] >> np.arange(50, dtype=np.uint64)) & np.uint64(1), 1, 2)
        sh = np.array([[th.is_static(p, gt, x, y) for y in xs] for x in xs])
        assert np.array_equal(r["static_hit"][e].astype(bool), sh), e
    assert (r["first_hit"] > 0).mean() > 0.05


def _raw(env, spec, first, count, outs):
    return env._lib.d2d_difficulty(env._h, C.byref(spec), first, count, *[C.c_void_p(o) for o in outs], env._stream())


def test_rejected_calls_change_nothing():
    from gym_drone2d_activeperception_b200 import _native
    from gym_drone2d_activeperception_b200.vec_env import difficulty_spec
    p = _P(agent_number=10)
    B = 32
    env = _env(p, B, world_gen="device")
    env.step(torch.zeros(B, dtype=torch.float64, device=DEV))
    before = _saved(env)
    stats = env.stats()
    fh = torch.full((B, 64), 77, dtype=torch.int16, device=DEV)
    sh = torch.full((B, 64), 77, dtype=torch.uint8, device=DEV)
    cs = torch.full((B, 64, 240), 77, dtype=torch.uint8, device=DEV)
    ok = (fh.data_ptr(), sh.data_ptr(), cs.data_ptr())
    spec, _ = difficulty_spec(240, GRID, collision_state=True)
    assert _raw(env, spec, 0, B, ok) == 0
    torch.cuda.synchronize()
    fh.fill_(77); sh.fill_(77); cs.fill_(77)

    def bad(mut=None, first=0, count=B, outs=ok):
        s, _ = difficulty_spec(240, GRID, collision_state=True)
        if mut:
            mut(s)
        assert _raw(env, s, first, count, outs) == -1                     # D2D_ERR_INVALID
    bad(first=1)                                                          # range beyond the handle
    bad(first=-1, count=2)
    bad(count=-1)
    bad(lambda s: setattr(s, "nx", 33) or setattr(s, "ny", 32))           # 1056 positions
    bad(lambda s: setattr(s, "steps", _native.DIFF_MAX_STEPS + 1))
    bad(lambda s: setattr(s, "steps", 0))
    bad(lambda s: setattr(s, "step", 0.0))
    bad(lambda s: setattr(s, "struct_size", 8))
    bad(lambda s: s.slot.__setitem__(5, 2))                               # decreasing
    bad(lambda s: s.slot.__setitem__(239, 240))                           # beyond n_slots
    bad(lambda s: setattr(s, "n_slots", 0))                               # collision_state given without slots
    host = np.zeros(B * 64 * 240, np.uint8)
    bad(outs=(fh.data_ptr(), sh.data_ptr(), host.ctypes.data))            # host pointers
    bad(outs=(host.ctypes.data, sh.data_ptr(), cs.data_ptr()))
    with pytest.raises(ValueError):
        env.difficulty(240, GRID, envs=[0, 2])
    with pytest.raises(ValueError):
        env.difficulty(240, GRID, out=(fh, sh))                           # wrong shapes
    torch.cuda.synchronize()
    assert (fh == 77).all() and (sh == 77).all() and (cs == 77).all()
    assert np.array_equal(_saved(env), before) and np.array_equal(env.stats(), stats)
    env.close()
    rvo = _env(_P(motion_profile="RVO", pillar_number=4, static_map="maps/obstacle_map.npy"), 8)
    with pytest.raises(_native.Drone2DNativeError, match="RVO"):
        rvo.difficulty(240, GRID)
    rvo.close()
