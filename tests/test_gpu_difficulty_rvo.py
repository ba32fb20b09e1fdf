"""d2d_grid_hits / Drone2DVecEnv.grid_hits and the RVO path of metrics.difficulty on the device: the step-kernel metrics
(global_survivability, survivability, obstacle_density) under RVO, the snapshot kernel under CVM, device and host worlds,
config lists, graph capture, read-only-ness and rejected calls."""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

DEV = "cuda:0"
GRID = (20, 20, 60, 8, 8)


def _P(**kw):
    from gym_drone2d_activeperception_b200.params import Params
    return Params(**dict(dict(debug=False, planner="NoMove", gaze_method="NoControl", motion_profile="RVO"), **kw))


def _env(p, B, **kw):
    from gym_drone2d_activeperception_b200.vec_env import Drone2DVecEnv
    return Drone2DVecEnv(p, B, device=DEV, **kw)


def _host(res):
    return {k: v.cpu().numpy() for k, v in res.items()}


def _saved(env):
    torch.cuda.synchronize()
    return env.save_state()["state"].cpu().numpy()


def _near_boundary_positions(p, seeds, xs, ys, T_surv):
    """bool [S, nx, ny]: positions with an (agent, step) pair whose distance lies within 1e-12 (relative) of
    r + drone_r during the survivability loop -- where the torch restatement's sqrt(dx*dx+dy*dy) and the kernel's
    sqrt(fma(y, y, x*x)) may disagree.  Agent positions recorded from an RVO env after every step."""
    L = len(np.arange(0, T_surv, 0.1))
    env = _env(p, len(seeds), seeds=np.asarray(seeds), auto_reset=False, trackers=False, oxford=False)
    zero = torch.zeros(len(seeds), dtype=torch.float64, device=DEV)
    pos = env.buffer("agent_pos")
    R = (env.buffer("agent_radius") + float(p.drone_radius))[:, :, None, None]                  # [S, N, 1, 1]
    gx = torch.tensor(np.asarray(xs, float), device=DEV)[:, None]
    gy = torch.tensor(np.asarray(ys, float), device=DEV)[None, :]
    near = torch.zeros((len(seeds), len(xs), len(ys)), dtype=torch.bool, device=DEV)
    for _ in range(L):                  # loop index i of the script sees the state after step i + 1
        env.step(zero)
        d = torch.sqrt((pos[:, :, 0, None, None] - gx) ** 2 + (pos[:, :, 1, None, None] - gy) ** 2)   # [S, N, nx, ny]
        near |= ((d - R).abs() <= 1e-12 * R).any(1)
    out = near.cpu().numpy()
    env.close()
    return out


# (params, position step, seeds): crowds of static-map agents get fewer seeds and a coarser grid
CONFIGS = {
    "empty_pillars": (dict(agent_number=20, agent_radius=15, pillar_number=4), 60, 256),
    "obstacle_pillars": (dict(static_map="maps/obstacle_map.npy", agent_number=10, pillar_number=4), 120, 96),
    "random_radius": (dict(agent_radius=-1, agent_number=20, pillar_number=2), 60, 256),
    "slow": (dict(agent_max_speed=4, agent_number=20, agent_radius=25), 60, 256),
    "step30": (dict(agent_number=15, agent_radius=20, pillar_number=3), 30, 192),
}


@pytest.mark.parametrize("name", list(CONFIGS))
def test_equals_step_kernel_metrics(name):
    """collision_state, global survival time and density exactly; survivability exactly except at positions with a pair
    within 1e-12 of the boundary (counted and reported).  num_envs below the seed count: an eager chunk, then graph
    replays of two chunk sizes."""
    from gym_drone2d_activeperception_b200.metrics import (difficulty, global_survivability, mean_survival_time,
                                                           obstacle_density, survivability, survivability_positions)
    kw, step, n = CONFIGS[name]
    p = _P(**kw)
    seeds = np.arange(2000, 2000 + n)
    r = difficulty(p, seeds, position_step=step, world_gen="host", collision_state=True, num_envs=n * 3 // 8,
                   device=DEV)
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


def test_cvm_grid_hits_equal_the_snapshot_kernel():
    """Under CVM, grid_hits after each of 240 steps from reset equals d2d_difficulty on every output."""
    from gym_drone2d_activeperception_b200.metrics import global_slots
    p = _P(motion_profile="CVM", static_map="maps/random_map_0.npy", agent_number=10)
    B = 4096
    env = _env(p, B, world_gen="device", auto_reset=False, trackers=False)
    n_slots, table = global_slots(24, p.dt, 240)
    ref = _host(env.difficulty(240, GRID, slots=table, n_slots=n_slots, collision_state=True))
    out = (torch.full((B, 8, 8), 77, dtype=torch.int16, device=DEV), torch.full((B, 8, 8), 77, dtype=torch.uint8, device=DEV),
           torch.full((B, 8, 8, n_slots), 77, dtype=torch.uint8, device=DEV))
    zero = torch.zeros(B, dtype=torch.float64, device=DEV)
    for t in range(1, 241):
        env.step(zero)
        env.grid_hits(t, GRID, slots=table, n_slots=n_slots, collision_state=True, out=out)
    got = _host(env.difficulty(240, GRID, slots=table, n_slots=n_slots, collision_state=True, out=None))
    env.close()
    for k, o in zip(("first_hit", "static_hit", "collision_state"), out):
        assert np.array_equal(o.cpu().numpy(), ref[k]), k
        assert np.array_equal(got[k], ref[k]), k
    assert (ref["first_hit"] > 0).mean() > 0.05 and ref["collision_state"].any()


def test_device_worlds_equal_host_worlds():
    """world_gen="device" equals "host" for RVO worlds, on every seed whose device snapshot equals generate_worlds."""
    from gym_drone2d_activeperception_b200.metrics import difficulty
    from gym_drone2d_activeperception_b200.world import generate_worlds
    p = _P(agent_number=12, pillar_number=4)
    seeds = np.arange(700, 1212)
    rh = difficulty(p, seeds, world_gen="host", collision_state=True, num_envs=200, device=DEV)
    rd = difficulty(p, seeds, world_gen="device", collision_state=True, num_envs=200, device=DEV)
    env = _env(p, len(seeds), seeds=seeds, auto_reset=False, trackers=False, world_gen="device")
    w = generate_worlds(p, seeds)
    b = lambda k: env.buffer(k).cpu().numpy()           # noqa: E731
    same = ((b("agent_pref0") == w["agent_pref"]).all((1, 2)) & (b("agent_pos0") == w["agent_pos"]).all((1, 2)) &
            (b("agent_vel0") == w["agent_vel"]).all((1, 2)) &
            (b("rvo_obstacles")[:, :4] == np.asarray(w["obstacles"]).reshape(len(seeds), -1, 3)).all((1, 2)))
    env.close()
    assert same.sum() >= 0.9 * len(seeds)
    for k in rh:
        assert np.array_equal(rd[k][same], rh[k][same]), k
    assert rh["collision_state"].any()


def test_config_list_equals_per_config_calls():
    """RVO configs that differ in agent speed and pillars share one batch group; the list call equals the per-config
    calls stacked."""
    from gym_drone2d_activeperception_b200.metrics import difficulty
    configs = [_P(agent_number=10, agent_max_speed=s, pillar_number=k) for s, k in ((20, 0), (20, 4), (8, 2))]
    seeds = np.arange(300, 428)
    got = difficulty(configs, seeds, collision_state=True, num_envs=160, device=DEV)
    for k, p in enumerate(configs):
        one = difficulty(p, seeds, collision_state=True, num_envs=160, device=DEV)
        for key in one:
            assert np.array_equal(got[key][k], one[key]), (k, key)


def test_graph_capture_equals_eager_and_writes_only_outputs():
    """A captured loop of step + grid_hits equals the eager loop; the env state and statistics equal those of envs that
    only stepped."""
    from gym_drone2d_activeperception_b200.metrics import global_slots
    p = _P(agent_number=16, pillar_number=4, static_map="maps/random_map_0.npy")
    B, K = 512, 240
    n_slots, table = global_slots(24, p.dt, K)
    envs = [_env(p, B, world_gen="device", auto_reset=False, trackers=False) for _ in range(3)]
    zero = torch.zeros(B, dtype=torch.float64, device=DEV)

    def outs():
        return (torch.zeros((B, 8, 8), dtype=torch.int16, device=DEV), torch.zeros((B, 8, 8), dtype=torch.uint8, device=DEV),
                torch.zeros((B, 8, 8, n_slots), dtype=torch.uint8, device=DEV))

    def loop(e, out, steps=range(1, K + 1)):
        for t in steps:
            e.step(zero)
            e.grid_hits(t, GRID, slots=table, n_slots=n_slots, collision_state=True, out=out)
    eager = outs()
    loop(envs[0], eager)
    # graph: warm up one step outside the capture, then capture steps 2..K; the step-only env takes the same steps
    graphed = outs()
    loop(envs[1], graphed, range(1, 2))
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        loop(envs[1], graphed, range(2, K + 1))
    g.replay()
    for _ in range(K):
        envs[2].step(zero)
    torch.cuda.synchronize()
    for a, b in zip(eager, graphed):
        assert torch.equal(a, b)
    assert eager[2].any()
    for e in envs[1:]:
        assert np.array_equal(_saved(e), _saved(envs[0]))
        assert np.array_equal(e.stats(), envs[0].stats())
    for e in envs:
        e.close()


def _raw(env, spec, t, first, count, outs):
    return env._lib.d2d_grid_hits(env._h, C.byref(spec), t, first, count, *[C.c_void_p(o) for o in outs], env._stream())


def test_rejected_calls_change_nothing():
    from gym_drone2d_activeperception_b200 import _native
    from gym_drone2d_activeperception_b200.vec_env import difficulty_spec
    p = _P(agent_number=10, pillar_number=4, static_map="maps/obstacle_map.npy")
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
    assert _raw(env, spec, 240, 0, B, ok) == 0
    torch.cuda.synchronize()
    fh.fill_(77); sh.fill_(77); cs.fill_(77)

    def bad(mut=None, t=1, first=0, count=B, outs=ok):
        s, _ = difficulty_spec(240, GRID, collision_state=True)
        if mut:
            mut(s)
        assert _raw(env, s, t, first, count, outs) == -1                  # D2D_ERR_INVALID
    bad(t=0)
    bad(t=241)
    bad(t=-5, count=0)
    bad(first=1)                                                          # range beyond the handle
    bad(first=-1, count=2)
    bad(count=-1)
    bad(lambda s: setattr(s, "nx", 33) or setattr(s, "ny", 32))           # 1056 positions
    bad(lambda s: setattr(s, "steps", _native.DIFF_MAX_STEPS + 1), t=1)
    bad(lambda s: setattr(s, "steps", 0))
    bad(lambda s: setattr(s, "step", float("nan")))
    bad(lambda s: setattr(s, "struct_size", 8))
    bad(lambda s: s.slot.__setitem__(5, 2))                               # decreasing
    bad(lambda s: s.slot.__setitem__(239, 240))                           # beyond n_slots
    bad(lambda s: setattr(s, "n_slots", 0))                               # collision_state given without slots
    host = np.zeros(B * 64 * 240, np.uint8)
    bad(outs=(fh.data_ptr(), sh.data_ptr(), host.ctypes.data))            # host pointers
    bad(outs=(host.ctypes.data, sh.data_ptr(), cs.data_ptr()))
    bad(outs=(fh.data_ptr(), 0, cs.data_ptr()))                           # null output
    assert "d2d_grid_hits" in env._lib.d2d_last_error(env._h).decode()
    with pytest.raises(ValueError):
        env.grid_hits(0, GRID)
    with pytest.raises(ValueError):
        env.grid_hits(1, GRID, envs=[0, 2])
    with pytest.raises(ValueError):
        env.grid_hits(1, GRID, out=(fh, sh))                              # wrong shapes
    with pytest.raises(ValueError):
        env.grid_hits(1, GRID, collision_state=True)                      # no slot table
    with pytest.raises(ValueError):
        env.grid_hits(_native.DIFF_MAX_STEPS + 1, GRID)
    torch.cuda.synchronize()
    assert (fh == 77).all() and (sh == 77).all() and (cs == 77).all()
    assert np.array_equal(_saved(env), before) and np.array_equal(env.stats(), stats)
    with pytest.raises(_native.Drone2DNativeError, match="RVO"):       # the snapshot kernel keeps refusing RVO handles
        env.difficulty(240, GRID)
    env.close()
