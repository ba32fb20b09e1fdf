"""The host-compiled twin of the device world generator (tests/helpers/worldgen_twin.cpp over csrc/d2d_worldgen.cuh) and
the comparison of generated worlds with world.generate_worlds, shared by the CPU and GPU world-generation tests."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

import util

_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        so = os.path.join(tempfile.mkdtemp(prefix="d2d_wt_"), "libworldgen_twin.so")
        src = os.path.join(util.ROOT, "tests", "helpers", "worldgen_twin.cpp")
        subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-o", so, src, "-lm"])
        L = C.CDLL(so)
        L.wt_sizeof_source.restype = C.c_long
        vp = C.c_void_p
        L.wt_generate.restype = C.c_long
        L.wt_generate.argtypes = [vp, vp, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int, vp, C.c_long] + [vp] * 11 + \
                                 [C.POINTER(C.c_char_p)]
        _LIB = L
    return _LIB


def twin_worlds(params, seeds):
    """The worlds the device generator builds for `seeds`, computed on the host: a dict shaped like generate_worlds'
    (gt_grid rebuilt from the row bitmasks, 1 = occupied, 2 otherwise) plus "failed" [S] (seeds given up)."""
    from gym_drone2d_activeperception_b200.world import count_agents, load_static_map, world_source
    smap = load_static_map(params.static_map)
    src = world_source(params, smap)
    N = count_agents(params, smap)
    S = len(seeds)
    rvo = 1 if params.motion_profile == "RVO" else 0
    noisy = 1 if params.var_cam != 0 else 0
    tg = np.ascontiguousarray(np.asarray(params.target_list, dtype=np.float64).reshape(-1, 2))
    sd = np.ascontiguousarray(np.asarray(seeds, dtype=np.uint32))
    out = dict(agent_pos=np.zeros((S, N, 2)), agent_pref=np.zeros((S, N, 2)), agent_radius=np.zeros((S, N)),
               tracker_radius=np.zeros((S, N)), gt_rows=np.zeros((S, 50), np.uint64), drone_pose=np.zeros((S, 3)),
               rng_key=np.zeros((S if noisy else 1, 624), np.uint32), agent_vel=np.zeros((S if rvo else 1, max(N, 1), 2)),
               obstacles=np.zeros((S if rvo else 1, 16, 3)), num_obstacles=np.zeros(S if rvo else 1, np.int32),
               failed=np.zeros(S, np.int32))
    why = C.c_char_p()
    order = ("agent_pos", "agent_pref", "agent_radius", "tracker_radius", "gt_rows", "drone_pose", "rng_key", "agent_vel",
             "obstacles", "num_obstacles", "failed")
    rc = lib().wt_generate(C.byref(src), tg.ctypes.data, len(tg), float(params.map_scale), N, rvo, noisy, sd.ctypes.data, S,
                           *[out[k].ctypes.data for k in order], C.byref(why))
    if rc < 0:
        raise ValueError(why.value.decode())
    bits = (out.pop("gt_rows")[:, :, None] >> np.arange(50, dtype=np.uint64)) & np.uint64(1)
    out["gt_grid"] = np.where(bits == 1, 1, 2).astype(np.uint8)
    if noisy:
        out.update(rng_pos=np.full(S, 200, np.int32), rng_has_gauss=np.zeros(S, np.int32), rng_gauss=np.zeros(S))
    if rvo:
        out["obstacles"] = out["obstacles"][:, :int(params.pillar_number)]
    return out


def gt_rows(gt_grid):
    """[S, 50, 50] ground-truth grids -> the [S, 50] row bitmasks the arena stores (bit j of row i: cell (i, j) == 1)."""
    w = (np.asarray(gt_grid) == 1).astype(np.uint64) << np.arange(50, dtype=np.uint64)
    return np.bitwise_or.reduce(w, axis=2).view(np.int64)


def _cr_cos_sin(d):
    import mpmath as mp
    mp.mp.prec = 120
    x = mp.mpf(float(d))
    return float(mp.cos(x)), float(mp.sin(x))


def group_velocity_exceptions(params, seeds, host_pref, other_pref):
    """Where the static-map agents' velocities of `other_pref` differ from `host_pref` (generate_worlds), check the
    documented exception: NumPy's cos / sin of that group's heading differ from the correctly rounded value, and
    `other_pref` is agent_max_speed times the correctly rounded value.  Returns (exempt bool [S], exempt evaluations)."""
    n_rand = int(params.agent_number)
    S = len(seeds)
    exempt = np.zeros(S, bool)
    n_eval = 0
    bad = np.nonzero((host_pref[:, n_rand:] != other_pref[:, n_rand:]).any(axis=(1, 2)))[0]
    if not len(bad):
        return exempt, 0
    from gym_drone2d_activeperception_b200.world import load_static_map
    smap = load_static_map(params.static_map)
    xs, ys = np.nonzero(smap)
    groups = smap[xs, ys].astype(np.int64)
    v = params.agent_max_speed
    for s in bad.tolist():
        direction = np.random.RandomState(int(seeds[s])).rand(100) * 2 * np.pi
        for m, g in enumerate(groups.tolist()):
            k = n_rand + m
            hp, op = host_pref[s, k], other_pref[s, k]
            if (hp == op).all():
                continue
            c, sn = _cr_cos_sin(direction[g])
            assert (np.cos(direction[g]), np.sin(direction[g])) != (c, sn), (s, k, "differs where NumPy is correctly rounded")
            assert op[0] == v * c and op[1] == v * sn, (s, k, "not speed * the correctly rounded cos / sin")
            n_eval += 1
        exempt[s] = True
    return exempt, n_eval


def near_disc_edge_count(world, n_cells=50, scale=10.0):
    """Agent / cell-centre pairs whose squared distance lies within 1e-12 (relative) of r**2: the only pairs on which the
    device's x*x and Python's pow could reach different erasure verdicts."""
    c = scale * (np.arange(n_cells) + 0.5)
    ap, ar = world["agent_pos"], world["agent_radius"]
    dx = c[None, None, :] - ap[:, :, 0:1]            # [S, N, 50]
    dy = c[None, None, :] - ap[:, :, 1:2]
    r2 = (ar * ar)[:, :, None, None]
    d2 = dx[:, :, :, None] ** 2 + dy[:, :, None, :] ** 2
    return int((np.abs(d2 - r2) <= 1e-12 * r2).sum())


def compare(params, seeds, host, other, name):
    """Every field of `other` (twin or device) equals generate_worlds' `host`, except group velocities under the exception
    rule.  Returns the number of seeds exempted."""
    exempt, _ = group_velocity_exceptions(params, seeds, host["agent_pref"], other["agent_pref"])
    n_rand = int(params.agent_number)
    assert np.array_equal(host["agent_pref"][:, :n_rand], other["agent_pref"][:, :n_rand]), name
    for k in ("agent_pos", "agent_radius", "tracker_radius", "drone_pose"):
        assert np.array_equal(host[k], other[k]), (name, k)
    assert np.array_equal(host["gt_grid"] == 1, other["gt_grid"] == 1), (name, "gt_grid")
    if params.var_cam != 0:
        for k in ("rng_key", "rng_pos", "rng_has_gauss", "rng_gauss"):
            assert np.array_equal(np.asarray(host[k]), np.asarray(other[k])), (name, k)
    if params.motion_profile == "RVO":
        n_map_ok = ~exempt
        assert np.array_equal(host["agent_vel"][n_map_ok], other["agent_vel"][n_map_ok]), (name, "agent_vel")
        assert np.array_equal(host["agent_vel"][:, :n_rand], other["agent_vel"][:, :n_rand]), (name, "agent_vel")
        assert np.array_equal(other["agent_vel"][:, n_rand:], other["agent_pref"][:, n_rand:]), (name, "agent_vel")
        assert np.array_equal(host["obstacles"], other["obstacles"]), (name, "obstacles")
    return int(exempt.sum())


def configs():
    """The parameter sets of the world-generation tests: the four shipped maps, pillars with RVO, measurement noise,
    random radii, 50 agents, several targets with another init position."""
    from gym_drone2d_activeperception_b200.params import Params
    base = dict(debug=False, planner="NoMove")
    P = lambda **kw: Params(**dict(base, **kw))
    return {
        "empty": P(static_map="maps/empty_map.npy"),
        "obstacle": P(static_map="maps/obstacle_map.npy"),
        "random0": P(static_map="maps/random_map_0.npy"),
        "shaped": P(static_map="maps/shaped_obstacle_map.npy"),
        "rvo_pillars": P(static_map="maps/obstacle_map.npy", pillar_number=8, motion_profile="RVO"),
        "noise": P(static_map="maps/random_map_0.npy", var_cam=1),
        "random_radius": P(static_map="maps/empty_map.npy", agent_radius=-1),
        "agents50": P(static_map="maps/empty_map.npy", agent_number=50, agent_radius=8),
        "targets": P(static_map="maps/shaped_obstacle_map.npy", pillar_number=3, init_pos=[120, 80],
                     target_list=[[50, 460], [400, 420], [450, 100]]),
    }
