"""Host-side world generation: what `Drone2DEnv2.__init__` produces from a seed (reference envs/drone_v2.py:69-117,
init_obstacles_random_size :12-66, OccupancyGridMap.init_obstacles utils.py:508-525).

`map_id` is only an RNG seed in the reference (drone_v2.py:79-80): the global `random` and `np.random` streams
are both seeded with it, consumed in a fixed order (pillars -> agents -> 100 group headings).  Here each env gets
private `random.Random(seed)` / `np.random.RandomState(seed)` instances, which produce the identical streams.
"""
import os
import random

import numpy as np
from numpy.linalg import norm

_MAP_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "maps")


def load_static_map(static_map):
    """Resolves the reference's 'maps/<name>.npy' paths against the package's own copy of the four shipped maps
    (data files), or any readable path."""
    if isinstance(static_map, np.ndarray):
        return static_map
    if os.path.isfile(static_map):
        return np.load(static_map)
    cand = os.path.join(_MAP_DIR, os.path.basename(static_map))
    if os.path.isfile(cand):
        return np.load(cand)
    raise FileNotFoundError(static_map)


def count_agents(params, static_map=None):
    m = load_static_map(params.static_map if static_map is None else static_map)
    return int(params.agent_number) + int(np.count_nonzero(m))


def generate_world(params, seed, static_map=None):
    """Returns dict(agent_pos [N,2], agent_pref [N,2], agent_radius [N], tracker_radius [N], gt_grid [gw,gh] u8
    (1 = OCCUPIED, 2 otherwise), drone_pose [3], obstacles [P,3])."""
    rnd = random.Random(seed)
    nrs = np.random.RandomState(seed)
    W, H = params.map_size
    scale = params.map_scale
    dx, dy = params.init_position
    drone_xy = np.array([dx, dy])

    # pillars (drone_v2.py:14-26)
    obstacles = []
    while len(obstacles) < params.pillar_number:
        obs = np.array([rnd.randint(50, W - 50), rnd.randint(50, H - 50), rnd.randint(15, 20)])
        free = True
        for target in params.target_list:
            if norm(np.asarray(target) - obs[:-1]) <= params.drone_radius + 20 + obs[-1]:
                free = False
                break
        if norm(drone_xy - obs[:-1]) <= params.drone_radius + 70:
            free = False
        if free:
            obstacles.append(obs)

    # random disc agents (drone_v2.py:28-47)
    pos, pref, rad, trk_rad = [], [], [], []
    n_rand = params.agent_number
    P_arr = np.empty((max(n_rand, 1), 2), dtype=np.float64)     # accepted positions / radii for the vectorised check
    R_arr = np.empty(max(n_rand, 1), dtype=np.float64)
    headings = [-params.agent_max_speed * np.array([np.cos(2 * np.pi * k / n_rand), np.sin(2 * np.pi * k / n_rand)])
                for k in range(n_rand)]
    while len(pos) < n_rand:
        p = np.array((rnd.uniform(20, W - 20), rnd.uniform(20, H - 20)))
        r = rnd.uniform(5, 15) if params.agent_radius == -1 else rnd.uniform(params.agent_radius - 2,
                                                                                  params.agent_radius + 2)
        k = len(pos)
        free = True
        if k:
            # norm(q - p) <= rq + r for every accepted agent (drone_v2.py:36-38).  Decided by a vectorised distance;
            # only pairs within 1e-12 relative of the threshold are re-evaluated with np.linalg.norm itself.
            d = P_arr[:k] - p
            approx = np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1])
            thr = R_arr[:k] + r
            if (approx <= thr * (1 - 1e-12)).any():
                free = False
            else:
                for j in np.nonzero(np.abs(approx - thr) <= thr * 1e-12)[0].tolist():
                    if norm(P_arr[j] - p) <= R_arr[j] + r:
                        free = False
        for ob in obstacles:
            if norm(np.array([ob[0], ob[1]]) - p) <= ob[2] + r + 10:
                free = False
        if norm(p - drone_xy) <= params.drone_radius + 70:
            free = False
        if free:
            P_arr[k] = p
            R_arr[k] = r
            pos.append(p)
            pref.append(headings[k])
            rad.append(r)
            trk_rad.append(r)           # drone_v2.py:46

    # every non-zero cell of the "static" map is a moving radius-5 agent (drone_v2.py:49-66)
    smap = load_static_map(params.static_map if static_map is None else static_map)
    vel = params.agent_max_speed
    direction = nrs.rand(100) * 2 * np.pi          # same stream as 100 sequential np.random.rand() calls
    vels = np.stack([vel * np.cos(direction), vel * np.sin(direction)], axis=1)
    xs, ys = np.nonzero(smap)                      # row-major order == the reference's nested x, y loops
    n_rnd, n_map = len(pos), len(xs)
    n = n_rnd + n_map
    agent_pos = np.empty((n, 2), dtype=np.float64)
    agent_pref = np.empty((n, 2), dtype=np.float64)
    agent_radius = np.empty(n, dtype=np.float64)
    tracker_radius = np.empty(n, dtype=np.float64)
    if n_rnd:
        agent_pos[:n_rnd] = np.array(pos, dtype=np.float64).reshape(n_rnd, 2)
        agent_pref[:n_rnd] = np.array(pref, dtype=np.float64).reshape(n_rnd, 2)
        agent_radius[:n_rnd] = rad
        tracker_radius[:n_rnd] = trk_rad
    if n_map:
        agent_pos[n_rnd:, 0] = 5 + xs * 10         # int64 cell centres (become float after the first step)
        agent_pos[n_rnd:, 1] = 5 + ys * 10
        agent_pref[n_rnd:] = vels[smap[xs, ys].astype(np.int64)]
        agent_radius[n_rnd:] = 5.0
        tracker_radius[n_rnd:] = float(params.agent_radius)   # KalmanFilter.__init__ default, utils.py:184

    # ground truth grid (utils.py:495-525).  Only cells == 1 matter downstream (utils.py:666,770).  NB: a cell
    # whose CENTRE lies inside an agent disc is overwritten with DYNAMIC_OCCUPIED even if it was a border / pillar
    # cell, and update_dynamic_grid (utils.py:527-530) then turns it into UNOCCUPIED for good -- so such cells are
    # not occupancy from the first perception pass on.
    gw, gh = W // scale, H // scale
    gt = np.full((gw, gh), 2, dtype=np.uint8)
    gt[0, :] = 1
    gt[-1, :] = 1
    gt[:, 0] = 1
    gt[:, -1] = 1
    for ob in obstacles:
        for i in range(max(0, int((ob[0] - ob[2]) // scale) - 1), min(gw, int((ob[0] + ob[2]) // scale) + 2)):
            for j in range(max(0, int((ob[1] - ob[2]) // scale) - 1), min(gh, int((ob[1] + ob[2]) // scale) + 2)):
                if norm(np.array([scale * (i + 0.5), scale * (j + 0.5)]) - np.array([ob[0], ob[1]])) <= ob[2]:
                    gt[i, j] = 1
    occ = np.argwhere(gt == 1)
    if n and len(occ):
        cxs, cys = scale * (occ[:, 0] + 0.5), scale * (occ[:, 1] + 0.5)
        # cheap vectorised reject, then the reference's scalar expression on the few candidate pairs
        # (`**2` on Python floats / NumPy scalars is libm pow there, utils.py:523)
        near = (np.abs(agent_pos[None, :, 0] - cxs[:, None]) <= agent_radius[None, :] + 1) & \
               (np.abs(agent_pos[None, :, 1] - cys[:, None]) <= agent_radius[None, :] + 1)
        for m, k in np.argwhere(near).tolist():
            cx, cy = float(cxs[m]), float(cys[m])
            ax, ay, r = float(agent_pos[k, 0]), float(agent_pos[k, 1]), float(agent_radius[k])
            if (cx - ax) ** 2 + (cy - ay) ** 2 <= r ** 2:
                gt[occ[m, 0], occ[m, 1]] = 2
    yaw0 = -90 % 360                                # Drone2D(init_yaw=-90): yaw = init_yaw % 360 (utils.py:718)
    st = nrs.get_state()                            # legacy np.random stream after the 100 heading draws (utils.py:605 continues it)
    return dict(rng_key=np.asarray(st[1], dtype=np.uint32).copy(), rng_pos=np.int32(st[2]), rng_has_gauss=np.int32(st[3]),
                rng_gauss=np.float64(st[4]),
                agent_pos=agent_pos, agent_pref=agent_pref, agent_radius=agent_radius, tracker_radius=tracker_radius,
                agent_vel=_initial_velocities(agent_pref, params.agent_number),
                gt_grid=gt, drone_pose=np.array([float(dx), float(dy), float(yaw0)]),
                obstacles=np.array(obstacles, dtype=np.float64).reshape(len(obstacles), 3))


def world_source(params, static_map=None):
    """The seed-independent inputs of generate_world as the d2d_world_source struct of d2d_set_world_source: the counts,
    radii, speed, init position and map size, the static map's group ids, and the random agents' headings evaluated with
    the same NumPy expression generate_world uses."""
    from ._native import D2DWorldSource, WORLD_MAX_RANDOM, WORLD_MAX_PILLARS, WORLD_GROUPS
    import ctypes as C
    smap = load_static_map(params.static_map if static_map is None else static_map)
    n_rand = int(params.agent_number)
    if not 0 <= n_rand <= WORLD_MAX_RANDOM:
        raise ValueError("device world generation: at most %d random agents (agent_number)" % WORLD_MAX_RANDOM)
    if not 0 <= int(params.pillar_number) <= WORLD_MAX_PILLARS:
        raise ValueError("device world generation: at most %d pillars (pillar_number)" % WORLD_MAX_PILLARS)
    if smap.shape != (50, 50) or smap.min() < 0 or smap.max() >= WORLD_GROUPS or np.any(smap != np.floor(smap)):
        raise ValueError("device world generation: the static map must be 50x50 integral group ids in [0, %d)" % WORLD_GROUPS)
    s = D2DWorldSource()
    s.struct_size = C.sizeof(D2DWorldSource)
    s.agent_number, s.pillar_number = n_rand, int(params.pillar_number)
    s.agent_radius, s.agent_max_speed, s.drone_radius = params.agent_radius, params.agent_max_speed, params.drone_radius
    s.init_x, s.init_y = params.init_position
    s.map_w, s.map_h = params.map_size
    for k in range(n_rand):          # generate_world's heading table, element for element
        h = -params.agent_max_speed * np.array([np.cos(2 * np.pi * k / n_rand), np.sin(2 * np.pi * k / n_rand)])
        s.headings[k][0], s.headings[k][1] = float(h[0]), float(h[1])
    groups = np.ascontiguousarray(smap, dtype=np.uint8)
    C.memmove(C.addressof(s.static_map), groups.ctypes.data, groups.nbytes)
    return s


def world_key(sources, seeds):
    """World keys `source * 2**32 + seed` (int64 array, broadcast) for d2d_generate_worlds_keyed and the keyed seed queue:
    `source` indexes the handle's table of world sources (`Drone2DVecEnv.set_world_sources`), [0, WORLD_MAX_SOURCES), and
    `seed` is the reference's map_id, [0, 2**32).  With source 0 the key is the seed."""
    from ._native import WORLD_MAX_SOURCES
    src, sd = np.asarray(sources), np.asarray(seeds)
    for name, a, hi in (("sources", src, WORLD_MAX_SOURCES), ("seeds", sd, 2 ** 32)):
        if a.size and a.dtype.kind not in "iu":
            raise ValueError("world_key: %s must be integers, got %s" % (name, a.dtype))
        if a.size and (a.min() < 0 or a.max() >= hi):
            raise ValueError("world_key: %s outside [0, %d)" % (name, hi))
    return (src.astype(np.int64) << np.int64(32)) | sd.astype(np.int64)


def split_world_key(keys):
    """(sources, seeds) of world keys, both int64 arrays; the inverse of world_key."""
    from ._native import WORLD_MAX_SOURCES
    k = np.asarray(keys)
    if k.size and k.dtype.kind not in "iu":
        raise ValueError("split_world_key: keys must be integers, got %s" % k.dtype)
    k = k.astype(np.int64)
    if k.size and (k.min() < 0 or k.max() >= np.int64(WORLD_MAX_SOURCES) << np.int64(32)):
        raise ValueError("split_world_key: keys outside [0, %d * 2**32)" % WORLD_MAX_SOURCES)
    return k >> np.int64(32), k & np.int64(0xFFFFFFFF)


def _initial_velocities(agent_pref, agent_number):
    """Agent.velocity right after __init__: `(0., 0.)` for the random agents (drone_v2.py:19), the group velocity for the
    map-cell agents (drone_v2.py:62).  Only read under the RVO motion profile (CVM overwrites it with pref_velocity)."""
    v = np.array(agent_pref, dtype=np.float64, copy=True).reshape(-1, 2)
    v[:agent_number] = 0.0
    return v


def generate_worlds(params, seeds, static_map=None):
    """Stacks generate_world over seeds -> arrays with a leading env axis."""
    smap = load_static_map(params.static_map if static_map is None else static_map)
    ws = [generate_world(params, int(s), smap) for s in seeds]
    keys = ("agent_pos", "agent_pref", "agent_radius", "tracker_radius", "gt_grid", "drone_pose")
    if getattr(params, "var_cam", 0) != 0:
        keys = keys + ("rng_key", "rng_pos", "rng_has_gauss", "rng_gauss")
    if getattr(params, "motion_profile", "CVM") == "RVO":       # RVO.RVO_update reads velocities and the pillars
        keys = keys + ("agent_vel", "obstacles")
    return {k: np.ascontiguousarray(np.stack([w[k] for w in ws])) for k in keys}
