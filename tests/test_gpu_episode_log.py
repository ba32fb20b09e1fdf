"""The episode log (d2d_enable_episode_log / d2d_read_episode_log) and the seed queue (d2d_set_seed_queue) against the
buffers and statistics they summarise, through every step entry point, under graph capture, and against fresh envs."""

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

DEV = "cuda:0"
STEPS = 300


def _P(**kw):
    from gym_drone2d_activeperception_b200.params import Params
    return Params(**dict(dict(debug=False, agent_number=10, agent_radius=15, agent_max_speed=20), **kw))


def _cases():
    return {
        "nomove_cfg2": (_P(planner="NoMove", static_map="maps/empty_map.npy", max_flight_time=8), "scripted"),
        "primitive_oxford": (_P(planner="Primitive", gaze_method="Oxford", static_map="maps/shaped_obstacle_map.npy"),
                             "step_plan_oxford"),
        "owl": (_P(planner="Primitive", gaze_method="Owl", static_map="maps/obstacle_map.npy"), "Owl"),
        "jerk": (_P(planner="Jerk_Primitive", gaze_method="LookGoal"), "LookGoal"),
        "rvo": (_P(planner="NoMove", motion_profile="RVO", pillar_number=6, static_map="maps/obstacle_map.npy",
                   max_flight_time=8), "scripted"),
        "noise": (_P(planner="NoMove", var_cam=1, static_map="maps/random_map_0.npy", max_flight_time=8), "scripted"),
    }


def _env(p, B, **kw):
    from gym_drone2d_activeperception_b200.vec_env import Drone2DVecEnv
    kw.setdefault("auto_reset", True)
    return Drone2DVecEnv(p, B, device=DEV, **kw)


def _scripted(B, steps, seed=1):
    table = np.arange(-80, 80, 80 / 3) / 80
    return table[np.random.RandomState(seed).randint(0, 6, (steps, B))]


def _from_buffers(env, step):
    """The records the log must hold for the step just taken, read from the buffers the way the host loop used to."""
    from gym_drone2d_activeperception_b200 import _native
    b = env.buffer
    idx = torch.nonzero(b("done")).flatten()
    out = np.zeros(int(idx.numel()), dtype=_native.EPISODE_DTYPE)
    if not len(out):
        return out
    g = lambda name: b(name)[idx].cpu().numpy()
    out["seed"] = env.seeds[idx.cpu().numpy()]
    out["step"] = step
    out["tracked_steps"] = g("tracker_buffer_ts")
    out["env"] = idx.cpu().numpy()
    out["steps"] = g("steps")
    out["grid_discovered"] = (b("belief")[idx] != 0).sum((1, 2)).cpu().numpy()
    out["trackers"] = g("tracker_buffer_count")
    out["state_machine"] = g("state_machine")
    out["collision_flag"] = g("collision_flag")
    out["freezing_flag"] = g("freezing_flag")
    out["dead_lock_flag"] = g("dead_lock_flag")
    return out


def _stepper(env, policy, B, steps):
    acts = _scripted(B, steps)
    nxt = env.plan_oxford() if policy == "step_plan_oxford" else None

    def step(t):
        nonlocal nxt
        if policy == "scripted":
            env.step(torch.as_tensor(acts[t], device=DEV))
        elif policy == "step_plan_oxford":
            env.step_plan_oxford(nxt, nxt)
        else:
            env.step(env.plan_gaze(policy))
    return step


@pytest.mark.parametrize("case", list(_cases()))
def test_records_match_buffers_and_statistics(case):
    from gym_drone2d_activeperception_b200 import _native
    p, policy = _cases()[case]
    B = 128
    env = _env(p, B, seeds=7 + np.arange(B))
    env.enable_episode_log(B * (STEPS + 1))
    env.stats(reset=True)
    step = _stepper(env, policy, B, STEPS + 1)
    expect = []
    for t in range(STEPS):
        step(t)
        expect.append(_from_buffers(env, t))
    st = env.stats()
    step(STEPS)                                   # one step more: its records are counted by the statistics as well
    st_grid = env.stats()[_native.STAT_NAMES.index("grid_discovered")]
    recs, dropped = env.read_episodes()
    expect = np.concatenate(expect)
    assert dropped == 0
    assert st_grid == int(recs["grid_discovered"].sum())
    recs = recs[recs["step"] < STEPS]
    assert len(expect) > 0, case
    assert recs.tobytes() == expect.tobytes(), case
    S = dict(zip(_native.STAT_NAMES, st.tolist()))
    assert S["episodes"] == len(recs)
    assert S["success"] == int((recs["state_machine"] == 1).sum())
    assert S["static_collision"] == int((recs["collision_flag"] == 1).sum())
    assert S["dynamic_collision"] == int((recs["collision_flag"] == 2).sum())
    assert S["freezing"] == int(recs["freezing_flag"].sum())
    assert S["dead_lock"] == int(recs["dead_lock_flag"].sum())
    assert S["flight_steps"] == int(recs["steps"].sum())
    assert S["agents_tracked"] == int(recs["trackers"].sum())
    assert S["tracked_steps"] == int(recs["tracked_steps"].sum())
    assert S["grid_discovered"] == int(recs["grid_discovered"].sum())
    env.close()


def _run_entry(entry, p, B, T, seeds):
    """T steps of the same scripted actions through one entry point, log enabled; returns the records."""
    env = _env(p, B, seeds=seeds)
    env.enable_episode_log(B * T)
    acts = _scripted(B, T)
    if entry == "step":
        for t in range(T):
            env.step(torch.as_tensor(acts[t], device=DEV))
    elif entry in ("step_host", "step_host_mirror"):
        if entry == "step_host_mirror":
            lm = torch.zeros((B, 1, 33, 33), dtype=torch.uint8).pin_memory()
            yaw = torch.zeros((B, 1), dtype=torch.float32).pin_memory()
            done = torch.zeros(B, dtype=torch.uint8).pin_memory()
            env.bind_host_mirror(lm, yaw, done)
        else:
            lm, yaw, done = np.zeros((B, 1, 33, 33), np.uint8), np.zeros((B, 1), np.float32), np.zeros(B, np.uint8)
        for t in range(T):
            env.step_host(np.ascontiguousarray(acts[t]), lm, yaw, done)
    elif entry in ("step_bound", "step_pipelined"):
        a = torch.zeros(B, dtype=torch.float64).pin_memory()
        env.bind_host_io(a, torch.zeros((B, 1, 33, 33), dtype=torch.uint8).pin_memory(),
                         torch.zeros((B, 1), dtype=torch.float32).pin_memory(), torch.zeros(B, dtype=torch.uint8).pin_memory())
        for t in range(T):
            a.copy_(torch.as_tensor(acts[t]))
            if entry == "step_bound":
                env.step_bound()
            else:
                env.step_pipelined(prelaunch_next=t < T - 1)
    elif entry == "rollout":
        for t0 in range(0, T, 50):
            env.rollout(torch.as_tensor(acts[t0:t0 + 50], device=DEV))
    recs, dropped = env.read_episodes()
    assert dropped == 0
    env.close()
    return recs


def test_every_entry_point_logs_the_same():
    p = _P(planner="NoMove", static_map="maps/random_map_0.npy", max_flight_time=6)
    B, T = 64, STEPS
    seeds = 3 + np.arange(B)
    ref = _run_entry("step", p, B, T, seeds)
    assert len(ref) > B
    for entry in ("step_host", "step_host_mirror", "step_bound", "step_pipelined", "rollout"):
        got = _run_entry(entry, p, B, T, seeds)
        assert got.tobytes() == ref.tobytes(), entry


def test_oxford_entry_points_log_the_same():
    p = _P(planner="Primitive", gaze_method="Oxford", static_map="maps/obstacle_map.npy", max_flight_time=10)
    B, T = 48, 150
    seeds = 11 + np.arange(B)
    out = {}
    for entry in ("plan_then_step", "step_plan_oxford", "step_bound_plan_oxford"):
        env = _env(p, B, seeds=seeds)
        env.enable_episode_log(B * T)
        if entry == "plan_then_step":
            for _ in range(T):
                env.step(env.plan_oxford())
        elif entry == "step_plan_oxford":
            a = env.plan_oxford()
            for _ in range(T):
                env.step_plan_oxford(a, a)
        else:
            env.bind_host_io(None, torch.zeros((B, 1, 33, 33), dtype=torch.uint8).pin_memory(),
                             torch.zeros((B, 1), dtype=torch.float32).pin_memory(), torch.zeros(B, dtype=torch.uint8).pin_memory())
            env.plan_oxford(env.buffer("actions_staging")[:B])
            for _ in range(T):
                env.step_bound_plan_oxford()
        out[entry], dropped = env.read_episodes()
        assert dropped == 0
        env.close()
    assert len(out["plan_then_step"]) > 0
    for k in out:
        assert out[k].tobytes() == out["plan_then_step"].tobytes(), k


def _all_buffers(env):
    names = ["agent_pos", "agent_pref", "belief", "env_records", "collision_flag", "dead_lock_flag", "freezing_flag", "done",
             "local_map", "yaw_angle", "hit", "tracker_active", "tracker_mu", "tracker_sigma", "tracker_radius", "tracker_ts",
             "need_plan", "plan_ok", "replan", "oxford_calls", "stats"]
    if env.cfg.planner == 1:
        names.append("traj_coeff")
    torch.cuda.synchronize()
    return {n: env.buffer(n).cpu().numpy().tobytes() for n in names}


@pytest.mark.parametrize("planner,gaze", [("NoMove", "LookAhead"), ("Primitive", "LookAhead")])
def test_log_does_not_perturb_the_simulation(planner, gaze):
    p = _P(planner=planner, gaze_method=gaze, static_map="maps/obstacle_map.npy", max_flight_time=10)
    B = 96
    seeds = 21 + np.arange(B)
    a, b = _env(p, B, seeds=seeds), _env(p, B, seeds=seeds)
    b.enable_episode_log(B * STEPS)
    la, lb = a.launch_count(), b.launch_count()
    for _ in range(STEPS):
        a.step(a.plan_gaze(gaze))
        b.step(b.plan_gaze(gaze))
    assert (b.launch_count() - lb) - (a.launch_count() - la) == STEPS
    assert _all_buffers(a) == _all_buffers(b)
    recs, _ = b.read_episodes()
    assert len(recs) > 0
    a.close()
    b.close()


def test_full_log_keeps_the_first_records_and_counts_the_rest():
    p = _P(planner="NoMove", static_map="maps/random_map_0.npy", max_flight_time=6)
    B, T, cap = 64, 200, 37
    seeds = 5 + np.arange(B)
    full = _run_entry("step", p, B, T, seeds)
    assert len(full) > cap
    env = _env(p, B, seeds=seeds)
    env.enable_episode_log(cap)
    acts = _scripted(B, T)
    for t in range(T):
        env.step(torch.as_tensor(acts[t], device=DEV))
    recs, dropped = env.read_episodes()
    assert recs.tobytes() == full[:cap].tobytes()
    assert dropped == len(full) - cap
    # the read emptied the log: one more step logs from slot 0 again
    env.step(torch.as_tensor(acts[0], device=DEV))
    more, dropped = env.read_episodes()
    assert dropped == 0 and len(more) == int(env.buffer("done").sum())
    env.close()


def test_seed_queue_rows_equal_fresh_envs():
    """2000 seeds through 64 envs: every seed's first record gives the row of a fresh host-built env of that seed."""
    from gym_drone2d_activeperception_b200.experiment import episode_row, run_batched_rows
    p = _P(planner="NoMove", gaze_method="LookAhead", static_map="maps/empty_map.npy", max_flight_time=5)
    S, B = 2000, 64
    seeds = 1000 + 7 * np.arange(S)
    env = _env(p, B, seeds=seeds[:B], world_gen="device")
    env.enable_episode_log(B * 64)
    env.set_seed_queue(seeds[B:])
    first = {}
    for _ in range(40):
        for _ in range(64):
            env.step(env.plan_gaze("LookAhead"))
        recs, dropped = env.read_episodes()
        assert dropped == 0
        for r in recs:
            first.setdefault(int(r["seed"]), episode_row(p, r))
        if len(first) == S:
            break
    assert set(first) == set(seeds.tolist())
    assert int(env.buffer("episode_log_head")[2]) == S - B
    env.close()
    ref = {r["Map ID"]: r for r in run_batched_rows(_P(planner="NoMove", gaze_method="LookAhead",
                                                        static_map="maps/empty_map.npy", max_flight_time=5),
                                                    S, episodes=1, seeds=seeds)}
    for s in seeds.tolist():
        a, b = first[s], ref[s]
        for k in a:
            if isinstance(b[k], float) and b[k] != b[k]:
                assert a[k] != a[k], (s, k)
            else:
                assert a[k] == b[k], (s, k, a[k], b[k])


def _saved(env):
    torch.cuda.synchronize()
    return env.save_state()["state"].cpu().numpy()


def test_queue_world_equals_lazy_reseed():
    p = _P(planner="NoMove", static_map="maps/random_map_0.npy", max_flight_time=4)
    B = 64
    a = _env(p, B, seeds=np.arange(B), world_gen="device")
    b = _env(p, B, seeds=np.arange(B), world_gen="device")
    for e in (a, b):
        e.enable_episode_log(B * 100)
    queue = 9000 + np.arange(3 * B)
    a.set_seed_queue(queue)
    act = torch.full((B,), 1.0 / 3, dtype=torch.float64, device=DEV)
    used = 0
    for _ in range(100):
        a.step(act)
        b.step(act)
        D = torch.nonzero(b.buffer("done")).flatten().cpu().numpy()
        if len(D):
            n = min(len(D), len(queue) - used)
            b.reseed(D[:n], queue[used:used + n], lazy=True)
            used += n
            assert np.array_equal(_saved(a), _saved(b))
            assert torch.equal(a.buffer("world_seed"), b.buffer("world_seed"))
        if used >= 2 * B:
            break
    assert used >= 2 * B
    ra, _ = a.read_episodes()
    rb, _ = b.read_episodes()
    assert ra.tobytes() == rb.tobytes()
    assert np.array_equal(a.seeds, b.seeds)
    a.close()
    b.close()


def test_rejected_queue_calls_change_nothing():
    from gym_drone2d_activeperception_b200 import _native
    L = _native.load()
    p = _P(planner="NoMove", static_map="maps/empty_map.npy")
    B = 16
    sd = np.array([1, 2, 3], np.int64)
    env = _env(p, B, seeds=np.arange(B), world_gen="device")
    with pytest.raises(_native.Drone2DNativeError, match="not enabled"):        # no log
        env.set_seed_queue(sd)
    env.enable_episode_log(64)
    env.set_seed_queue(sd)
    head = env.buffer("episode_log_head").clone()
    for bad in ([-1], [2 ** 32], [5, 2 ** 40]):
        with pytest.raises(_native.Drone2DNativeError):
            env.set_seed_queue(np.array(bad, np.int64))
        assert torch.equal(env.buffer("episode_log_head"), head)
    env.close()
    h = _env(p, B, seeds=np.arange(B))                                          # no world source
    h.enable_episode_log(64)
    assert L.d2d_set_seed_queue(h._h, sd.ctypes.data, 3, None) == -4
    assert int(h.buffer("episode_log_head")[3]) == 0
    h.close()
    r = _env(p, B, seeds=np.arange(B), world_gen="device", auto_reset=False)   # auto_reset = 0
    r.enable_episode_log(64)
    with pytest.raises(_native.Drone2DNativeError, match="auto_reset"):
        r.set_seed_queue(sd)
    assert int(r.buffer("episode_log_head")[3]) == 0
    r.close()


def test_graph_capture_gives_the_same_records():
    p = _P(planner="Primitive", gaze_method="LookAhead", static_map="maps/obstacle_map.npy", max_flight_time=4)
    B, K = 64, 64
    seeds = 100 + np.arange(B)
    queue = 5000 + np.arange(4 * B)
    envs = []
    for _ in range(2):
        e = _env(p, B, seeds=seeds, world_gen="device")
        e.enable_episode_log(B * (K + 8))
        e.set_seed_queue(queue)
        envs.append(e)
    acts = [torch.empty(B, dtype=torch.float64, device=DEV) for _ in envs]
    for e, a in zip(envs, acts):                       # one-time set-up of the launch paths
        for _ in range(8):
            e.step(e.plan_gaze("LookAhead", a))
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(K):
            envs[0].step(envs[0].plan_gaze("LookAhead", acts[0]))
    g.replay()
    for _ in range(K):
        envs[1].step(envs[1].plan_gaze("LookAhead", acts[1]))
    ra, _ = envs[0].read_episodes()
    rb, _ = envs[1].read_episodes()
    assert len(rb) > B and ra.tobytes() == rb.tobytes()
    assert np.array_equal(envs[0].seeds, envs[1].seeds)
    assert np.array_equal(_saved(envs[0]), _saved(envs[1]))
    for e in envs:
        e.close()


def test_world_seed_follows_reseed_clone_and_load():
    p = _P(planner="NoMove", static_map="maps/empty_map.npy")
    B = 16
    env = _env(p, B, seeds=np.arange(B), world_gen="device")
    env.enable_episode_log(64)
    ws = lambda: env.buffer("world_seed").cpu().numpy()
    assert np.array_equal(ws(), np.arange(B))
    env.reseed([3, 4], [300, 400], lazy=True)
    assert ws()[3] == 300 and ws()[4] == 400
    env.clone_envs([3], [9])
    assert ws()[9] == 300
    saved = env.save_state([4, 9])
    env.load_state(saved, [0, 1])
    assert ws()[0] == 400 and ws()[1] == 300
    assert np.array_equal(ws(), env.seeds)
    env.enable_episode_log(0)
    with pytest.raises(Exception):
        env.buffer("world_seed")
    env.close()
