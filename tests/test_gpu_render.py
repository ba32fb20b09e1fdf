"""d2d_render against its NumPy twin (tests/render_reference.py) byte for byte, read-only-ness, env selection and argument
rejection, CUDA-graph capture, the Drone2DEnv2 facade, and a full-size batch."""
import ctypes as C

import numpy as np
import pytest

import render_reference as rr

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

DEV = "cuda:0"
PPCS = (1, 2, 3, 7, 10)
SINGLE = (rr.GROUND_TRUTH, rr.BELIEF, rr.VIEW, rr.PLAN, rr.TRACKERS, rr.AGENTS, rr.DRONE)


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
        "n142": (_P(planner="Primitive", gaze_method="LookAhead", static_map="maps/random_map_0.npy", agent_number=20,
                    agent_max_speed=40), "LookAhead"),
    }


def _env(p, B, **kw):
    from gym_drone2d_activeperception_b200.vec_env import Drone2DVecEnv
    kw.setdefault("auto_reset", True)
    return Drone2DVecEnv(p, B, device=DEV, **kw)


def _stepper(env, policy, B, steps, seed=1):
    table = np.arange(-80, 80, 80 / 3) / 80
    acts = table[np.random.RandomState(seed).randint(0, 6, (steps, B))]
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


class _Tally:
    def __init__(self):
        self.pixels, self.exempt = 0, 0

    def check(self, env, envs, ppc, layers, frames=None, what=""):
        if frames is None:
            frames = env.render(list(envs), ppc, layers)
        got = frames.cpu().numpy()
        for k, e in enumerate(envs):
            want, ex = rr.render(rr.env_state(env, e), env.cfg, ppc, layers)
            bad = (got[k] != want).any(2) & ~ex
            assert not bad.any(), (what, e, ppc, layers, np.argwhere(bad)[:5].tolist(), got[k][bad][:3].tolist(),
                                   want[bad][:3].tolist())
            self.pixels += ex.size
            self.exempt += int(ex.sum())


@pytest.mark.parametrize("name", list(_cases()))
def test_kernel_equals_twin(name):
    p, policy = _cases()[name]
    B = 48
    env = _env(p, B)
    step = _stepper(env, policy, B, 300)
    tally = _Tally()
    rng = np.random.RandomState(7)
    t = 0
    for upto in (0, 1, 50, 300):
        while t < upto:
            step(t)
            t += 1
        torch.cuda.synchronize()
        pick = list(rng.choice(B, 3, replace=False))
        done = np.nonzero(env.buffer("done").cpu().numpy())[0]
        pick += list(done[:2])                                  # envs that just reported done: their terminal state
        if upto == 50:                                          # a pending lazy reseed still shows the old world
            env.reseed([int(pick[0]), int(pick[1])], [9000 + upto, 9001 + upto], lazy=True)
        for ppc in PPCS:
            tally.check(env, pick, ppc, rr.ALL, what=(name, upto))
        for layers in SINGLE:
            tally.check(env, pick[:2], 3 if layers != rr.VIEW else 7, layers, what=(name, upto))
    assert tally.exempt <= 1e-5 * tally.pixels, (tally.exempt, tally.pixels)
    env.close()


def _saved(env):
    torch.cuda.synchronize()
    return env.save_state()["state"].cpu().numpy()


def test_render_is_read_only():
    p = _P(planner="Primitive", gaze_method="Oxford", static_map="maps/shaped_obstacle_map.npy")
    B, T = 64, 300
    envs = [_env(p, B) for _ in range(2)]
    for e in envs:
        e.enable_episode_log(B * T)
    steps = [_stepper(e, "step_plan_oxford", B, T) for e in envs]
    for t in range(T):
        for k, e in enumerate(envs):
            steps[k](t)
            if k == 0:
                e.render([5, 3, 3, 60] if t % 2 else range(0, B), 2)
    assert np.array_equal(_saved(envs[0]), _saved(envs[1]))
    assert np.array_equal(envs[0].stats(), envs[1].stats())
    ra, _ = envs[0].read_episodes()
    rb, _ = envs[1].read_episodes()
    assert len(ra) > 0 and ra.tobytes() == rb.tobytes()
    for e in envs:
        e.close()

    # the host observation mirror of a bound step_host run
    p = _P(planner="NoMove", static_map="maps/empty_map.npy", max_flight_time=8)
    envs = [_env(p, B) for _ in range(2)]
    mirrors = []
    for e in envs:
        m = (torch.zeros((B, 1, 33, 33), dtype=torch.uint8).pin_memory(), torch.zeros((B, 1), dtype=torch.float32).pin_memory(),
             torch.zeros(B, dtype=torch.uint8).pin_memory())
        e.bind_host_mirror(*m)
        mirrors.append(m)
    acts = (np.arange(-80, 80, 80 / 3) / 80)[np.random.RandomState(3).randint(0, 6, (T, B))]
    for t in range(T):
        for k, e in enumerate(envs):
            e.step_host(np.ascontiguousarray(acts[t]), *mirrors[k])
            if k == 0:
                e.render(range(B) if t % 2 else [1, 1, 40], 1)
    for a, b in zip(*mirrors):
        assert torch.equal(a, b)
    assert np.array_equal(_saved(envs[0]), _saved(envs[1]))
    assert np.array_equal(envs[0].stats(), envs[1].stats())
    for e in envs:
        e.close()


def _raw(env, envs, first, count, ppc, layers, ptr):
    lst = None if envs is None else np.ascontiguousarray(envs, dtype=np.int32)
    return env._lib.d2d_render(env._h, None if lst is None else lst.ctypes.data_as(C.c_void_p), first, count, ppc, layers,
                               C.c_void_p(ptr), env._stream())


def test_selection_and_rejection():
    from gym_drone2d_activeperception_b200 import _native
    p = _P(planner="Primitive", gaze_method="Oxford", static_map="maps/obstacle_map.npy")
    B = 1100
    env = _env(p, B, world_gen="device")
    step = _stepper(env, "step_plan_oxford", B, 20)
    for t in range(20):
        step(t)
    whole = env.render(None, 3)
    assert torch.equal(env.render([7, 2, 7, 9], 3), whole[[7, 2, 7, 9]])
    assert torch.equal(env.render(range(10, 20), 3), whole[10:20])
    assert torch.equal(env.render(list(range(10, 20)), 3), env.render(np.array([10, 11, 12, 13, 14, 15, 16, 17, 19, 18]), 3)[
        [0, 1, 2, 3, 4, 5, 6, 7, 9, 8]])
    assert env.render([], 3).shape == (0, 150, 150, 3)
    assert env.render(range(5, 5), 3).shape == (0, 150, 150, 3)
    n0 = env.launch_count()
    assert _raw(env, [], 0, 0, 3, rr.ALL, 0) == 0 and env.launch_count() == n0
    lst = list(np.random.RandomState(1).randint(0, B, 1024))
    assert torch.equal(env.render(lst, 1), env.render(None, 1)[lst])
    assert env.launch_count() == n0 + 2
    with pytest.raises(ValueError):
        env.render(lst + [0], 1)

    out = torch.full((4, 30, 30, 3), 77, dtype=torch.uint8, device=DEV)
    H = (4, 30, 30, 3)
    cases = [([0, B, 1, 2], 0, 4, 3, rr.ALL, out.data_ptr()),                # env out of range
             ([0, -1], 0, 2, 3, rr.ALL, out.data_ptr()),
             (None, B - 1, 2, 3, rr.ALL, out.data_ptr()),                # range past the end
             (None, -1, 2, 3, rr.ALL, out.data_ptr()),
             (None, 0, -1, 3, rr.ALL, out.data_ptr()),                   # negative count
             (None, 0, 4, 0, rr.ALL, out.data_ptr()),                    # ppc 0 and 11
             (None, 0, 4, 11, rr.ALL, out.data_ptr()),
             (None, 0, 4, 3, 128, out.data_ptr()),                       # unknown layer bits
             (None, 0, 4, 3, rr.ALL | 256, out.data_ptr()),
             (None, 0, 4, 3, rr.ALL, 0),                                 # null pointer
             (list(range(1025)), 0, 1025, 1, rr.ALL, out.data_ptr())]   # list too long
    host = torch.zeros(H, dtype=torch.uint8).pin_memory()
    cases.append((None, 0, 4, 3, rr.ALL, host.data_ptr()))              # pinned host memory
    pageable = np.zeros(H, np.uint8)
    cases.append((None, 0, 4, 3, rr.ALL, pageable.ctypes.data))         # pageable host memory
    if torch.cuda.device_count() > 1:
        other = torch.zeros(H, dtype=torch.uint8, device="cuda:1")
        cases.append((None, 0, 4, 3, rr.ALL, other.data_ptr()))
    n0 = env.launch_count()
    for c in cases:
        assert _raw(env, *c) == -1, c
    torch.cuda.synchronize()
    assert (out == 77).all() and (host == 0).all() and not pageable.any()
    assert env.launch_count() == n0

    # an unaligned out[t] slice (odd ppc: a frame is 3 * 150 * 150 bytes)
    frames = torch.full((3, 5, 150, 150, 3), 5, dtype=torch.uint8, device=DEV)
    for t in range(3):
        env.render([3, 8, 1000, 2, 7], 3, out=frames[t, :])
    for t in range(3):
        assert torch.equal(frames[t], whole[[3, 8, 1000, 2, 7]])
    sub = torch.full((1 + 2 * 150 * 150 * 3,), 9, dtype=torch.uint8, device=DEV)
    assert _raw(env, [11, 12], 0, 2, 3, rr.ALL, sub.data_ptr() + 1) == 0
    assert torch.equal(sub[1:].view(2, 150, 150, 3), whole[11:13]) and int(sub[0]) == 9
    env.close()

    # D2D_ERR_STATE before set_world and during a pipelined step
    from gym_drone2d_activeperception_b200.vec_env import make_config
    from gym_drone2d_activeperception_b200.world import count_agents
    L = _native.load()
    cfg = make_config(p, 4, count_agents(p), 0)
    h = C.c_void_p()
    assert L.d2d_create(C.byref(cfg), C.byref(h)) == 0
    buf = torch.zeros((4, 50, 50, 3), dtype=torch.uint8, device=DEV)
    assert L.d2d_render(h, None, 0, 4, 1, rr.ALL, C.c_void_p(buf.data_ptr()), None) == -4
    L.d2d_destroy(h)
    p2 = _P(planner="NoMove", static_map="maps/empty_map.npy")
    env = _env(p2, 64)
    a = torch.zeros(64, dtype=torch.float64).pin_memory()
    env.bind_host_io(a, torch.zeros((64, 1, 33, 33), dtype=torch.uint8).pin_memory(),
                     torch.zeros((64, 1), dtype=torch.float32).pin_memory(), torch.zeros(64, dtype=torch.uint8).pin_memory())
    env.step_pipelined(prelaunch_next=True)           # the first call after binding refreshes the mirror synchronously
    env.step_pipelined(prelaunch_next=True)           # this one leaves the next step in flight
    buf = torch.full((2, 50, 50, 3), 77, dtype=torch.uint8, device=DEV)
    assert _raw(env, None, 0, 2, 1, rr.ALL, buf.data_ptr()) == -4
    env.step_pipelined(prelaunch_next=False)
    torch.cuda.synchronize()
    assert (buf == 77).all()
    assert _raw(env, None, 0, 2, 1, rr.ALL, buf.data_ptr()) == 0
    env.close()


def test_graph_capture_equals_eager():
    p = _P(planner="Primitive", gaze_method="Oxford", static_map="maps/obstacle_map.npy", agent_radius=10)
    B, K = 256, 64
    pick = list(np.random.RandomState(2).choice(B, 16, replace=False))
    envs = [_env(p, B, world_gen="device") for _ in range(2)]
    acts = [e.plan_oxford() for e in envs]
    frames = [torch.zeros((K, 16, 200, 200, 3), dtype=torch.uint8, device=DEV) for _ in envs]
    for e, a in zip(envs, acts):                       # one-time set-up of the launch paths
        for _ in range(4):
            e.step_plan_oxford(a, a)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for t in range(K):
            envs[0].step_plan_oxford(acts[0], acts[0])
            envs[0].render(pick, 4, out=frames[0][t])
    g.replay()
    for t in range(K):
        envs[1].step_plan_oxford(acts[1], acts[1])
        envs[1].render(pick, 4, out=frames[1][t])
    torch.cuda.synchronize()
    assert torch.equal(frames[0], frames[1])
    assert not torch.equal(frames[0][0], frames[0][K - 1])
    assert np.array_equal(_saved(envs[0]), _saved(envs[1]))
    for e in envs:
        e.close()


def test_facade_rgb_array():
    from gym_drone2d_activeperception_b200.env import Drone2DEnv2
    env = Drone2DEnv2(_P(planner="Primitive", gaze_method="LookAhead"), device=DEV)
    for _ in range(5):
        env.step(0.5)
    img = env.render("rgb_array")
    assert isinstance(img, np.ndarray) and img.shape == (500, 500, 3) and img.dtype == np.uint8
    assert np.array_equal(img, env._vec.render([0], 10)[0].cpu().numpy())
    with pytest.raises(NotImplementedError, match="rgb_array"):
        env.render()
    assert env._vec.metadata["render.modes"] == ["rgb_array"]
    env.close()


def test_full_size_config4():
    p = _P(planner="Primitive", gaze_method="Oxford", static_map="maps/obstacle_map.npy", agent_radius=10)
    B = 65536
    env = _env(p, B, world_gen="device")
    a = env.plan_oxford()
    for _ in range(30):
        env.step_plan_oxford(a, a)
    frames = env.render(None, 1)
    torch.cuda.synchronize()
    assert frames.numel() == B * 50 * 50 * 3
    tally = _Tally()
    sample = sorted(np.random.RandomState(11).choice(B, 256, replace=False).tolist())
    got = frames[sample]
    tally.check(env, sample, 1, rr.ALL, frames=got, what="full")
    assert tally.exempt <= 1e-5 * tally.pixels
    env.close()
