"""Per-env state clone / save / load (d2d_clone_envs, d2d_save_state, d2d_load_state).

Every case runs a twin check and a bystander check after the call and at every later step:
  twin      -- each dst env equals its src env bit for bit on every per-env buffer (live state, reset snapshot, RNG stream,
               policy state, step outputs) and on the materialised Oxford map, drone_pose0 and the facade fields;
  bystander -- every env outside dst equals a control handle that was stepped identically without the call."""
import ctypes as C

import numpy as np
import pytest

import util

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

DEV = "cuda:0"
# per-env buffers with the env on axis 0 (allocated per env under every configuration)
AXIS0 = ["agent_pos", "agent_pref", "agent_pos0", "agent_pref0", "agent_radius", "tracker_radius0", "gt_rows", "belief",
         "env_records", "collision_flag", "dead_lock_flag", "freezing_flag", "done", "local_map", "yaw_angle", "hit",
         "tracker_active", "tracker_mu", "tracker_sigma", "tracker_radius", "tracker_ts", "need_plan", "plan_ok", "replan",
         "oxford_calls", "owl_queue_len", "owl_queue_value", "drone_acc"]
AXIS1 = ["rng_pos", "rng_gauss", "drone_pose0"]      # [planes, B] (B a multiple of 16 here: the views' plane stride is B)
FACADE = ["drone_x", "drone_y", "drone_yaw", "drone_vx", "drone_vy", "state_machine", "target_x", "target_y", "steps",
          "tracker_buffer_count", "tracker_buffer_ts", "traj_nseg", "traj_cursor", "pending_reset", "oxford_fresh",
          "owl_fresh", "obs_ix", "obs_iy"]


def _params(**kw):
    from gym_drone2d_activeperception_b200.params import Params
    base = dict(debug=False, planner="NoMove", map_id=5, agent_number=10, agent_radius=15, agent_max_speed=40)
    base.update(kw)
    return Params(**base)


def _env(p, B, worlds, **kw):
    from gym_drone2d_activeperception_b200.vec_env import Drone2DVecEnv
    kw.setdefault("auto_reset", True)
    return Drone2DVecEnv(p, B, worlds=worlds, device=DEV, **kw)


def _worlds(p, B, seed0=11):
    from gym_drone2d_activeperception_b200 import generate_worlds
    return generate_worlds(p, seed0 + np.arange(B))


def _names(env):
    c = env.cfg
    names = [(n, 0) for n in AXIS0 + FACADE] + [(n, 1) for n in AXIS1]
    if c.motion_profile == 1:
        names += [("agent_vel", 0), ("agent_vel0", 0), ("rvo_obstacles", 0), ("rvo_num_obstacles", 0)]
    if c.planner == 1:
        names.append(("traj_coeff", 0))
    if c.var_cam != 0:
        names += [("rng_key", 0), ("rng_key0", 0)]
    if c.oxford & 2:
        names.append(("owl_U", 0))
    if c.oxford & 1:
        names.append(("oxford_last_time_observed", 0))
    return names


def _bits(t):
    """Exact comparison (NaN-safe): floats reinterpreted as integers of the same width."""
    if t.dtype == torch.float64:
        return t.view(torch.int64)
    if t.dtype == torch.float32:
        return t.view(torch.int32)
    return t


def _state(env):
    return {n: (ax, _bits(env.buffer(n))) for n, ax in _names(env)}


def check_twins(env, src, dst, tag):
    s = torch.as_tensor(np.asarray(src), device=DEV, dtype=torch.long)
    d = torch.as_tensor(np.asarray(dst), device=DEV, dtype=torch.long)
    for n, (ax, t) in _state(env).items():
        assert torch.equal(t.index_select(ax, d), t.index_select(ax, s)), ("twin", n, tag)


def check_bystanders(env, ctl, dst, tag):
    keep = torch.as_tensor(np.setdiff1d(np.arange(env.num_envs), np.asarray(dst)), device=DEV, dtype=torch.long)
    a, b = _state(env), _state(ctl)
    for n, (ax, t) in a.items():
        assert torch.equal(t.index_select(ax, keep), b[n][1].index_select(ax, keep)), ("bystander", n, tag)


def _scripted(B, steps, seed):
    table = torch.as_tensor(util.action_table(), device=DEV)
    g = torch.Generator().manual_seed(seed)
    return table[torch.randint(0, 6, (steps, B), generator=g).to(DEV)]


def _twin_actions(a, src, dst):
    """The action vector of the cloned handle: every dst env gets its src env's action."""
    b = a.clone()
    b[torch.as_tensor(dst, device=DEV)] = a[torch.as_tensor(src, device=DEV)]
    return b


SRC = [3, 3, 7, 12, 20, 20, 20, 31]
DST = [0, 25, 30, 13, 5, 6, 22, 16]


def _run_scripted(p, B=32, pre=40, post=150, src=SRC, dst=DST, before=None, **kw):
    w = _worlds(p, B)
    env, ctl = _env(p, B, w, **kw), _env(p, B, w, **kw)
    acts = _scripted(B, pre + post, 7)
    for t in range(pre):
        env.step(acts[t]); ctl.step(acts[t])
    if before is not None:
        src, dst = before(env, ctl, src, dst)
    n0 = env.launch_count()
    env.clone_envs(src, dst)
    assert env.launch_count() == n0 + 1, "a clone is one kernel launch"
    check_twins(env, src, dst, "clone")
    check_bystanders(env, ctl, dst, "clone")
    dones = 0
    for t in range(pre, pre + post):
        env.step(_twin_actions(acts[t], src, dst)); ctl.step(acts[t])
        check_twins(env, src, dst, t)
        check_bystanders(env, ctl, dst, t)
        dones += int(env.buffer("done")[torch.as_tensor(src, device=DEV)].sum())
    assert np.array_equal(env.seeds[dst], env.seeds[src])
    env.close(); ctl.close()
    return dones


@pytest.mark.parametrize("static_map", ["maps/empty_map.npy", "maps/obstacle_map.npy"])
def test_clone_nomove_scripted(static_map):
    assert _run_scripted(_params(static_map=static_map)) > 0, "the run must cross auto-resets of the sources"


def test_clone_nomove_noisy_rng_stream():
    p = _params(var_cam=0.5)
    assert _run_scripted(p) > 0


def test_clone_rvo_pillars():
    p = _params(motion_profile="RVO", pillar_number=5, agent_number=8)
    _run_scripted(p)


def test_clone_carries_pending_lazy_reset():
    def before(env, ctl, src, dst):
        mask = torch.zeros(env.num_envs, dtype=torch.uint8, device=DEV)
        mask[torch.as_tensor(src, device=DEV)] = 1
        env.reset(mask, lazy=True); ctl.reset(mask, lazy=True)
        assert int(env.buffer("pending_reset")[src[0]].item()) == 1
        return src, dst
    _run_scripted(_params(), post=60, before=before)


def test_clone_right_after_done_with_auto_reset():
    p = _params(agent_number=20)
    B = 32
    w = _worlds(p, B)
    env, ctl = _env(p, B, w), _env(p, B, w)
    acts = _scripted(B, 600, 9)
    t = 0
    while True:
        env.step(acts[t]); ctl.step(acts[t]); t += 1
        done = env.buffer("done").cpu().numpy()
        if done.any() or t == 400:
            break
    assert done.any(), "no episode ended"
    src = [int(np.nonzero(done)[0][0])] * 2
    dst = [e for e in range(B) if e not in src][:2]
    terminal = env.buffer("local_map")[src[0]].clone()
    env.clone_envs(src, dst)
    check_twins(env, src, dst, "clone")
    check_bystanders(env, ctl, dst, "clone")
    assert torch.equal(env.buffer("local_map")[dst[0]], terminal), "the clone holds the terminal observation"
    for k in range(t, t + 150):
        env.step(_twin_actions(acts[k], src, dst)); ctl.step(acts[k])
        if k == t:
            assert int(env.buffer("steps")[dst[0]].item()) <= 1, "the clone is reset by its next step"
        check_twins(env, src, dst, k)
        check_bystanders(env, ctl, dst, k)
    env.close(); ctl.close()


def test_clone_primitive_oxford_policy():
    p = _params(planner="Primitive", gaze_method="Oxford", static_map="maps/obstacle_map.npy", agent_number=10,
                agent_radius=10, agent_max_speed=20)
    B = 32
    w = _worlds(p, B)
    env, ctl = _env(p, B, w, oxford=True), _env(p, B, w, oxford=True)
    a, b = env.plan_oxford(), ctl.plan_oxford()
    for t in range(40):
        a = env.step_plan_oxford(a, out=a); b = ctl.step_plan_oxford(b, out=b)
    assert int(env.buffer("traj_nseg")[torch.as_tensor(SRC, device=DEV)].max()) > 0, "the sources are mid-trajectory"
    env.clone_envs(SRC, DST)
    a = _twin_actions(a, SRC, DST)           # the next actions are caller data: the clone's come from its source
    check_twins(env, SRC, DST, "clone")
    check_bystanders(env, ctl, DST, "clone")
    dones = 0
    for t in range(150):
        a = env.step_plan_oxford(a, out=a); b = ctl.step_plan_oxford(b, out=b)
        assert torch.equal(_bits(a[DST]), _bits(a[SRC])), ("policy actions", t)
        check_twins(env, SRC, DST, t)
        check_bystanders(env, ctl, DST, t)
        dones += int(env.buffer("done")[SRC].sum())
    assert dones > 0
    env.close(); ctl.close()


@pytest.mark.parametrize("policy,planner,kw", [
    ("LookGoal", "Jerk_Primitive", {}),
    ("Owl", "Primitive", dict(owl=True)),
], ids=["jerk_lookgoal", "owl_queue"])
def test_clone_gaze_policy(policy, planner, kw):
    p = _params(planner=planner, gaze_method=policy, agent_number=10, agent_radius=15, agent_max_speed=20, drone_max_speed=40)
    B = 32
    w = _worlds(p, B)
    env, ctl = _env(p, B, w, **kw), _env(p, B, w, **kw)
    src, dst = list(SRC), list(DST)
    for t in range(40):
        env.step(env.plan_gaze(policy)); ctl.step(ctl.plan_gaze(policy))
    a, b = env.plan_gaze(policy), ctl.plan_gaze(policy)      # the policy call of the next step; the clone comes in between
    if policy == "Owl":
        q = env.buffer("owl_queue_len").cpu().numpy()
        busy = [int(e) for e in np.nonzero(q > 0)[0]]
        assert busy, "no env has a queued Owl action"
        src = [busy[0]] * 3 + busy[1:3]
        dst = [e for e in range(B) if e not in src][:len(src)]
    else:
        assert float(env.buffer("drone_acc")[SRC].abs().max()) > 0, "the jerk path keeps a non-zero acceleration"
    env.clone_envs(src, dst)
    a = _twin_actions(a, src, dst)
    check_twins(env, src, dst, "clone")
    check_bystanders(env, ctl, dst, "clone")
    for t in range(150):
        env.step(a); ctl.step(b)
        check_twins(env, src, dst, t)
        check_bystanders(env, ctl, dst, t)
        a, b = env.plan_gaze(policy), ctl.plan_gaze(policy)
        assert torch.equal(_bits(a[dst]), _bits(a[src])), ("policy actions", t)
    env.close(); ctl.close()


# ------------------------------------------------------------------------------------------ save / load
def _snapshot(env):
    return {n: t.clone() for n, (ax, t) in _state(env).items()}


def _equal_snap(x, y, tag):
    for n in x:
        assert torch.equal(x[n], y[n]), (n, tag)


def test_save_load_replay():
    p = _params(var_cam=0.5)
    B = 32
    env = _env(p, B, _worlds(p, B))
    acts = _scripted(B, 80, 3)
    for t in range(20):
        env.step(acts[t])
    saved = env.save_state()
    nbytes, fp = env.state_layout()
    assert saved["state"].shape == (B, nbytes) and nbytes % 128 == 0 and saved["fingerprint"] == fp
    first = []
    for t in range(20, 80):
        env.step(acts[t]); first.append(_snapshot(env))
    env.load_state(saved)
    for k, t in enumerate(range(20, 80)):
        env.step(acts[t]); _equal_snap(first[k], _snapshot(env), t)
    env.close()


def test_save_load_cross_handle_and_host_round_trip(tmp_path):
    p = _params(planner="Primitive", gaze_method="Oxford")
    B = 32
    A = _env(p, B, _worlds(p, B, 100), oxford=True)
    Bh = _env(p, B, _worlds(p, B, 500), oxford=True)
    assert A.state_layout() == Bh.state_layout(), "same params, different seeds: same layout"
    a = A.plan_oxford()
    for t in range(30):
        a = A.step_plan_oxford(a, out=a)
    envs = [5, 9, 17, 30]
    saved = A.save_state(envs)
    disk = {"fingerprint": saved["fingerprint"], "state": saved["state"].cpu(), "seeds": saved["seeds"]}
    torch.save(disk, str(tmp_path / "state.pt"))
    back = torch.load(str(tmp_path / "state.pt"), weights_only=False)     # "seeds" is a numpy array
    back["state"] = back["state"].to(DEV)
    targets = [1, 2, 3, 4]
    Bh.load_state(back, targets)
    assert np.array_equal(Bh.seeds[targets], A.seeds[envs])
    sa, sb = _state(A), _state(Bh)
    ia, ib = torch.as_tensor(envs, device=DEV), torch.as_tensor(targets, device=DEV)
    for n, (ax, t) in sa.items():
        assert torch.equal(t.index_select(ax, ia), sb[n][1].index_select(ax, ib)), n
    b = Bh.plan_oxford()
    a = A.plan_oxford()
    for t in range(80):
        assert torch.equal(_bits(a[ia]), _bits(b[ib])), ("policy actions", t)
        a = A.step_plan_oxford(a, out=a); b = Bh.step_plan_oxford(b, out=b)
        sa, sb = _state(A), _state(Bh)
        for n, (ax, x) in sa.items():
            assert torch.equal(x.index_select(ax, ia), sb[n][1].index_select(ax, ib)), (n, t)
    A.close(); Bh.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_save_on_one_gpu_load_on_another():
    from gym_drone2d_activeperception_b200.vec_env import Drone2DVecEnv
    p = _params()
    B = 16
    w = _worlds(p, B)
    A = Drone2DVecEnv(p, B, worlds=w, device="cuda:0")
    Bh = Drone2DVecEnv(p, B, worlds=_worlds(p, B, 77), device="cuda:1")
    acts = _scripted(B, 30, 1)
    for t in range(30):
        A.step(acts[t])
    s = A.save_state()
    with pytest.raises(ValueError):
        Bh.load_state(s)                       # still on cuda:0
    s["state"] = s["state"].to("cuda:1")
    Bh.load_state(s)
    torch.cuda.synchronize("cuda:1")
    for n in ("belief", "env_records", "agent_pos", "tracker_sigma", "local_map"):
        assert torch.equal(A.buffer(n).cpu(), Bh.buffer(n).cpu()), n
    A.close(); Bh.close()


def test_load_rejects_foreign_layouts_and_host_memory():
    from gym_drone2d_activeperception_b200 import _native
    p = _params()
    B = 16
    env = _env(p, B, _worlds(p, B))
    env.step(_scripted(B, 1, 0)[0])
    before = _snapshot(env)
    other_planner = _env(_params(planner="Primitive"), B, _worlds(p, B))
    other_agents = _env(_params(agent_number=11), B, _worlds(_params(agent_number=11), B))
    for other in (other_planner, other_agents):
        assert other.state_layout()[1] != env.state_layout()[1]
        s = other.save_state()
        s["state"] = torch.zeros((B, env.state_layout()[0]), dtype=torch.uint8, device=DEV)   # right shape, wrong layout
        with pytest.raises(_native.Drone2DNativeError, match="fingerprint"):
            env.load_state(s)
    good = env.save_state()
    with pytest.raises(ValueError):
        env.load_state({"fingerprint": good["fingerprint"], "state": good["state"].cpu(), "seeds": good["seeds"]})
    host = good["state"].cpu()                 # the library itself refuses host memory and misaligned buffers
    rc = env._lib.d2d_load_state(env._h, None, B, C.c_void_p(host.data_ptr()), C.c_uint64(good["fingerprint"]), env._stream())
    assert rc == -1
    dev = torch.zeros(B * good["state"].shape[1] + 16, dtype=torch.uint8, device=DEV)
    rc = env._lib.d2d_load_state(env._h, None, 1, C.c_void_p(dev.data_ptr() + 8), C.c_uint64(good["fingerprint"]), env._stream())
    assert rc == -1 and b"aligned" in env._lib.d2d_last_error(env._h)
    _equal_snap(before, _snapshot(env), "after rejected loads")
    for e in (env, other_planner, other_agents):
        e.close()


# ------------------------------------------------------------------------------------------ validation, mirror, pipelining
def test_clone_index_validation():
    from gym_drone2d_activeperception_b200 import _native
    p = _params()
    B = 16
    env = _env(p, B, _worlds(p, B))
    env.step(_scripted(B, 1, 0)[0])
    before = _snapshot(env)
    n0 = env.launch_count()
    bad = [([0], [B]), ([B + 3], [1]), ([-1], [2]), ([0, 1], [2, 2]), ([0, 1], [1, 3]), ([4], [4])]
    for src, dst in bad:
        with pytest.raises(_native.Drone2DNativeError):
            env.clone_envs(src, dst)
    with pytest.raises(_native.Drone2DNativeError):
        env.save_state([B])
    with pytest.raises(_native.Drone2DNativeError):
        env.load_state(env.save_state([0, 1]), [3, 3])
    assert env.launch_count() == n0 + 1     # only the valid save above ran a kernel
    env.clone_envs([], [])
    env.clone_envs(np.array([], dtype=np.int64), torch.tensor([], dtype=torch.int32))
    assert env.launch_count() == n0 + 1, "count = 0 is a no-op"
    _equal_snap(before, _snapshot(env), "after rejected calls")
    env.clone_envs(np.array([1]), torch.tensor([2]))    # numpy / CPU tensor indices
    check_twins(env, [1], [2], "numpy+tensor")
    env.close()


def test_state_calls_before_set_world_and_layout_anytime():
    p = _params()
    env = _env(p, 16, _worlds(p, 16))
    L = env._lib
    cfg = env.cfg
    h = C.c_void_p()
    assert L.d2d_create(C.byref(cfg), C.byref(h)) == 0
    nb, fp = C.c_int64(), C.c_uint64()
    assert L.d2d_state_layout(h, C.byref(nb), C.byref(fp)) == 0
    assert (nb.value, fp.value) == env.state_layout()
    idx = (C.c_int32 * 1)(0)
    idx2 = (C.c_int32 * 1)(1)
    assert L.d2d_clone_envs(h, idx, idx2, 1, None) == -4
    assert L.d2d_save_state(h, None, 1, None, None) == -4
    assert L.d2d_load_state(h, None, 1, None, fp, None) == -4
    L.d2d_destroy(h)
    env.close()


@pytest.mark.parametrize("bound", [False, True], ids=["bind_host_mirror", "bind_host_io"])
def test_clone_refreshes_host_mirror(bound):
    p = _params()
    B = 32
    env = _env(p, B, _worlds(p, B))
    lm = torch.zeros((B, 1, 33, 33), dtype=torch.uint8).pin_memory()
    yaw = torch.zeros(B, dtype=torch.float32).pin_memory()
    dn = torch.zeros(B, dtype=torch.uint8).pin_memory()
    acts = _scripted(B, 60, 4).cpu()
    a_pin = torch.zeros(B, dtype=torch.float64).pin_memory()
    if bound:
        env.bind_host_io(a_pin, lm, yaw, dn)
    else:
        env.bind_host_mirror(lm, yaw, dn)

    def step(t):
        a = _twin_actions(acts[t].to(DEV), SRC, DST).cpu()
        if bound:
            a_pin.copy_(a); env.step_bound()
        else:
            env.step_host(a.pin_memory(), lm, yaw, dn)
    for t in range(30):
        step(t)
    env.clone_envs(SRC, DST)
    for t in range(30, 60):
        step(t)
        assert torch.equal(lm, env.buffer("local_map").cpu()), t
        assert torch.equal(yaw, env.buffer("yaw_angle").cpu()[:, 0]), t
        assert torch.equal(dn, env.buffer("done").cpu()), t
    check_twins(env, SRC, DST, "end")
    env.close()


def test_clone_refused_while_a_pipelined_step_is_in_flight():
    from gym_drone2d_activeperception_b200 import _native
    p = _params()
    B = 32
    env = _env(p, B, _worlds(p, B))
    lm = torch.zeros((B, 1, 33, 33), dtype=torch.uint8).pin_memory()
    yaw = torch.zeros(B, dtype=torch.float32).pin_memory()
    dn = torch.zeros(B, dtype=torch.uint8).pin_memory()
    a_pin = torch.full((B,), 1.0 / 3, dtype=torch.float64).pin_memory()
    env.bind_host_io(a_pin, lm, yaw, dn)
    env.step_pipelined(True)
    env.step_pipelined(True)
    with pytest.raises(_native.Drone2DNativeError, match=r"\(-4\)"):
        env.clone_envs([0], [1])
    env.step_pipelined(False)
    env.clone_envs([0], [1])
    torch.cuda.synchronize()
    check_twins(env, [0], [1], "after the run")
    env.close()


def test_stats_unchanged_by_clone_and_load():
    p = _params(agent_number=20)
    B = 32
    env = _env(p, B, _worlds(p, B))
    acts = _scripted(B, 120, 5)
    for t in range(120):
        env.step(acts[t])
    st = env.stats()
    assert st[1] > 0
    env.clone_envs(SRC, DST)
    assert np.array_equal(env.stats(), st)
    env.load_state(env.save_state([1, 2]), [8, 9])
    assert np.array_equal(env.stats(), st)
    env.close()


def test_facade_get_set_state():
    from gym_drone2d_activeperception_b200.env import Drone2DEnv2
    p = _params(planner="Primitive", gaze_method="LookAhead", map_id=3, agent_number=6)
    e = Drone2DEnv2(p)
    for _ in range(10):
        e.step(0.5)
    s = e.get_state()
    first = [e.step(a)[1:3] + (e.drone.x, e.drone.y, e.steps) for a in (1.0, -1.0, 0.0, 0.5)]
    e.set_state(s)
    again = [e.step(a)[1:3] + (e.drone.x, e.drone.y, e.steps) for a in (1.0, -1.0, 0.0, 0.5)]
    assert first == again
    e.close()


# ------------------------------------------------------------------------------------------ scale: config 4 fan-out
def test_clone_fanout_config4_scale():
    from gym_drone2d_activeperception_b200 import Params
    p = Params(debug=False, planner="Primitive", gaze_method="Oxford", static_map="maps/obstacle_map.npy", agent_number=10,
               agent_radius=10, agent_max_speed=20, map_id=1)
    B, S = 32768, 4096
    uniq = _worlds(p, 128, 1)
    w = {k: np.ascontiguousarray(np.concatenate([v] * (B // 128))) for k, v in uniq.items()}
    env = _env(p, B, w, oxford=True)
    a = env.plan_oxford()
    for t in range(50):
        a = env.step_plan_oxford(a, out=a)
    src = np.tile(np.arange(S), 7)
    dst = np.arange(S, B)
    env.clone_envs(src, dst)
    a = _twin_actions(a, src, dst)
    names = util.BATCH_FIELDS + util.TRACKER_FIELDS + util.PLANNER_FIELDS + ["env_records"]
    si, di = torch.as_tensor(src, device=DEV), torch.as_tensor(dst, device=DEV)
    for t in range(61):
        if t:
            a = env.step_plan_oxford(a, out=a)
        for n in names:
            x = _bits(env.buffer(n))
            assert torch.equal(x.index_select(0, di), x.index_select(0, si)), (n, t)
    env.close()
