"""Difficulty metrics on the CPU: the host-compiled twin of the agent stepping and hit search of d2d_difficulty_kernel
(tests/helpers/difficulty_twin.cpp over csrc/d2d_agent_math.cuh) against the oracle's agents and against a direct NumPy
restatement of survivability_calculator.py and glob_survivability_calculator.py.  No GPU needed."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import util

_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        so = os.path.join(tempfile.mkdtemp(prefix="d2d_dt_"), "libdifficulty_twin.so")
        src = os.path.join(util.ROOT, "tests", "helpers", "difficulty_twin.cpp")
        subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-o", so, src, "-lm"])
        L = C.CDLL(so)
        vp, d, i = C.c_void_p, C.c_double, C.c_int
        L.dt_trajectory.argtypes = [C.c_long, vp, vp, vp, d, d, d, d, C.c_long, vp]
        L.dt_first_hit.argtypes = [C.c_long, vp, vp, vp, d, d, d, d, d, d, d, d, i, i, i, vp]
        L.dt_agent_hits.argtypes = [d, d, d, d, d]
        L.dt_sizeof_spec.restype = L.dt_offsetof_slot.restype = C.c_long
        _LIB = L
    return _LIB


def _c(a, dt=np.float64):
    return np.ascontiguousarray(a, dtype=dt)


def twin_trajectory(p, pos, pref, rad, steps):
    n = len(rad)
    out = np.zeros((steps, n, 2))
    pos, pref, rad = _c(pos), _c(pref), _c(rad)
    lib().dt_trajectory(n, pos.ctypes.data, pref.ctypes.data, rad.ctypes.data, p.dt, float(p.map_scale),
                        float(p.map_size[0]), float(p.map_size[1]), steps, out.ctypes.data)
    return out


def twin_first_hit(p, pos, pref, rad, grid, steps):
    x0, y0, step, nx, ny = grid
    out = np.zeros(nx * ny, np.int16)
    pos, pref, rad = _c(pos), _c(pref), _c(rad)
    lib().dt_first_hit(len(rad), pos.ctypes.data, pref.ctypes.data, rad.ctypes.data, float(p.drone_radius), p.dt,
                       float(p.map_scale), float(p.map_size[0]), float(p.map_size[1]), float(x0), float(y0), float(step),
                       nx, ny, steps, out.ctypes.data)
    return out.reshape(nx, ny)


def configs():
    from gym_drone2d_activeperception_b200.params import Params
    P = lambda **kw: Params(**dict(dict(debug=False, planner="NoMove", gaze_method="NoControl"), **kw))
    return {
        "empty": P(agent_number=20, agent_radius=15),
        "obstacle": P(static_map="maps/obstacle_map.npy", agent_number=30, agent_radius=20),
        "random0_pillars": P(static_map="maps/random_map_0.npy", pillar_number=8),       # static-map agents too
        "shaped": P(static_map="maps/shaped_obstacle_map.npy", agent_number=12),
        "random_radius": P(agent_radius=-1, agent_number=25),
        "slow": P(agent_max_speed=4, agent_number=20, agent_radius=25),                  # the <= 5 px/s rotation branch
    }


SEEDS = [0, 5, 11, 2 ** 32 - 1]
STEPS = 240


@pytest.mark.parametrize("name", list(configs()))
def test_twin_agents_equal_oracle(name):
    """Agent positions after each of 240 steps: the twin equals the oracle env (NoMove) bit for bit."""
    from gym_drone2d_activeperception_b200.world import generate_worlds
    p = configs()[name]
    w = generate_worlds(p, SEEDS)
    rotated = 0
    for i in range(len(SEEDS)):
        tw = twin_trajectory(p, w["agent_pos"][i], w["agent_pref"][i], w["agent_radius"][i], STEPS)
        e = util.oracle_env_from_world(p, w, i)
        n = e.n
        for k in range(STEPS):
            e.step(0.0)
            assert np.array_equal(e.apos[:n], tw[k]), (name, SEEDS[i], k)
        e.close()
        rotated += int((np.hypot(w["agent_pref"][i][:, 0], w["agent_pref"][i][:, 1]) <= 5).sum())
    if name == "slow":
        assert rotated > 0


def is_static(p, gt_grid, x, y):
    """Drone2D.is_collide's five static probes (utils.py:766-771) at (x, y) on one ground-truth grid (1 = occupied)."""
    r = p.drone_radius
    for dx, dy in ((-r, 0), (0, 0), (r, 0), (0, -r), (0, r)):
        px, py = x + dx, y + dy
        if px >= p.map_size[0] or px < 0 or py >= p.map_size[1] or py < 0:
            return True
        if gt_grid[int(px // p.map_scale), int(py // p.map_scale)] == 1:
            return True
    return False


def hits(pos, rad, drone_r, x, y):
    """Per agent: np.linalg.norm(agent.position - p) < agent.radius + drone.radius, evaluated as the scripts do (the
    vectorised distance only pre-sorts; every pair near the boundary is decided by np.linalg.norm itself)."""
    d = pos - np.array([x, y], dtype=np.float64)
    R = rad + drone_r
    approx = np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1])
    out = approx < R
    near = np.nonzero(np.abs(approx - R) <= 1e-9 * R)[0]
    for a in near.tolist():
        out[a] = np.linalg.norm(pos[a] - np.array([x, y])) < R[a]
    return out


def script_metrics(p, traj, rad, gt_grid, xs, ys, T_surv, T_glob):
    """survivability_calculator.py:24-47 and glob_survivability_calculator.py:24-41 loop for loop on one world, from the
    agent positions after each step (traj[k-1]: after step k) -- no env needed, since under NoMove nothing else moves."""
    st = np.ones((len(xs), len(ys))) * T_surv
    for i, t in enumerate(np.arange(0, T_surv, 0.1)):            # the script steps once before its loop
        for a, x in enumerate(xs):
            for b, y in enumerate(ys):
                if hits(traj[i], rad, p.drone_radius, x, y).any():
                    st[a, b] = min(t, st[a, b])
    st = st - 0.1
    st[st < 0] = 0
    steps = int(T_glob / p.dt)
    cs = np.zeros((len(xs), len(ys), steps), np.uint8)
    for a, x in enumerate(xs):
        for b, y in enumerate(ys):
            if is_static(p, gt_grid, x, y):                       # collision_flag 1, never 2
                continue
            for k, t in enumerate(np.arange(0, T_glob, 0.1)[:steps]):
                if hits(traj[k], rad, p.drone_radius, x, y).any():
                    cs[a, b, int(t / 0.1)] = 1
    return st, cs


@pytest.mark.parametrize("name,position_step", [("empty", 60), ("obstacle", 60), ("random0_pillars", 30),
                                                ("shaped", 60), ("random_radius", 60), ("slow", 60)])
def test_twin_metrics_equal_scripts(name, position_step):
    from gym_drone2d_activeperception_b200.metrics import (global_slots, mean_survival_time, survival_from_hits,
                                                           survivability_positions)
    from gym_drone2d_activeperception_b200.world import generate_worlds
    p = configs()[name]
    xs, ys = survivability_positions(p, position_step)
    grid = (xs[0], ys[0], position_step, len(xs), len(ys))
    T_surv, T_glob = 12, 24
    steps = max(int(T_glob / p.dt), len(np.arange(0, T_surv, 0.1)))
    n_slots, table = global_slots(T_glob, p.dt, steps)
    seeds = SEEDS[:2]
    w = generate_worlds(p, seeds)
    for i in range(len(seeds)):
        pos, pref, rad = w["agent_pos"][i], w["agent_pref"][i], w["agent_radius"][i]
        fh = twin_first_hit(p, pos, pref, rad, grid, steps)
        sh = np.array([[is_static(p, w["gt_grid"][i], x, y) for y in ys] for x in xs])
        got = survival_from_hits(fh[None], sh[None], T_surv, n_slots, table)
        st, cs = script_metrics(p, twin_trajectory(p, pos, pref, rad, steps), rad, w["gt_grid"][i], xs, ys, T_surv, T_glob)
        assert np.array_equal(got["survivability"][0], st), (name, seeds[i])
        assert np.array_equal(got["mean_survivability"], st.reshape(1, -1).mean(1))
        assert np.array_equal(got["global_survival_time"][0], mean_survival_time(cs)), (name, seeds[i])
        assert (fh > 0).any()


def test_boundary_distance_is_not_a_hit():
    """`<` excludes an agent at exactly r + drone_r from a position, on an axis and on a 3-4-5 diagonal."""
    from gym_drone2d_activeperception_b200.params import Params
    L = lib()
    assert L.dt_agent_hits(105.0, 200.0, 5.0, 100.0, 200.0) == 0
    assert L.dt_agent_hits(np.nextafter(105.0, 0), 200.0, 5.0, 100.0, 200.0) == 1
    assert L.dt_agent_hits(103.0, 204.0, 5.0, 100.0, 200.0) == 0
    assert L.dt_agent_hits(103.0, np.nextafter(204.0, 0), 5.0, 100.0, 200.0) == 1
    # a resting agent (pref 0: the rotation branch keeps it at rest) next to grid positions of a 3 x 3 grid, step 60
    p = Params(debug=False, planner="NoMove", agent_radius=10)
    R = 10 + p.drone_radius
    pos = np.array([[100.0 + R, 100.0], [220.0 + 3 * R / 5, 160.0 + 4 * R / 5], [np.nextafter(100.0 + R, 0), 220.0]])
    fh = twin_first_hit(p, pos, np.zeros((3, 2)), np.full(3, 10.0), (100.0, 100.0, 60.0, 3, 3), 4)
    expect = np.zeros((3, 3), np.int16)
    expect[0, 2] = 1                                              # (100, 220): the third agent, just inside
    assert np.array_equal(fh, expect), fh


def test_slot_table():
    from gym_drone2d_activeperception_b200 import _native
    from gym_drone2d_activeperception_b200.metrics import global_slots
    n, tab = global_slots(24, 0.1, 240)
    ref = [int(t / 0.1) for t in np.arange(0, 24, 0.1)]
    assert n == 240 and tab == ref and sum(1 for k, s in enumerate(tab) if s != k) == 10
    assert all(a <= b for a, b in zip(tab, tab[1:]))
    n, tab = global_slots(6, 0.1, 240)
    assert n == 60 and tab[:60] == [int(t / 0.1) for t in np.arange(0, 6, 0.1)]
    assert tab[60:] == [_native.DIFF_NO_SLOT] * 180


def test_spec_building():
    from gym_drone2d_activeperception_b200 import _native
    from gym_drone2d_activeperception_b200.vec_env import difficulty_spec
    L = lib()
    assert L.dt_sizeof_spec() == C.sizeof(_native.D2DDifficultySpec)
    assert L.dt_offsetof_slot() == _native.D2DDifficultySpec.slot.offset
    spec, n = difficulty_spec(240, (20, 30, 60, 8, 7))
    assert n == 0 and spec.n_slots == 0 and (spec.nx, spec.ny, spec.x0, spec.y0, spec.step, spec.steps) == (8, 7, 20.0, 30.0, 60.0, 240)
    assert spec.struct_size == C.sizeof(_native.D2DDifficultySpec)
    spec, n = difficulty_spec(5, (0, 0, 1, 1, 1), collision_state=True)
    assert n == 5 and list(spec.slot[:5]) == [0, 1, 2, 3, 4]
    spec, n = difficulty_spec(5, (0, 0, 1, 1, 1), collision_state=True, slots=[0, 0, 2], n_slots=4)
    assert n == 4 and list(spec.slot[:5]) == [0, 0, 2, _native.DIFF_NO_SLOT, _native.DIFF_NO_SLOT]
    for bad in (dict(steps=0), dict(steps=_native.DIFF_MAX_STEPS + 1), dict(slots=[0] * 6), dict(slots=[-1])):
        kw = dict(steps=5, grid=(0, 0, 1, 1, 1), collision_state=True)
        kw.update(bad)
        with pytest.raises(ValueError):
            difficulty_spec(**kw)
