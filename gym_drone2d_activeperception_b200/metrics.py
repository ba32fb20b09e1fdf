"""Difficulty metrics of the reference on the batched env (SURVEY.md §8f rank 1).

`global_survivability` is script/difficulty_calculator/glob_survivability_calculator.py:13-44: for every world and every
start position of an 8x8 grid (x, y in range(map_scale + drone_radius, size - map_scale - drone_radius, 60)) the drone is
pinned at the position (`env.drone.x = x` before every step), the env is stepped with the NoMove planner and action 0 for
T / dt steps, and `collision_state[ix, iy, int(t / 0.1)] = 1` whenever `info['collision_flag'] == 2`.  The reference runs the
64 x 240 steps of one world sequentially on one env object; here all (world, position) pairs are one batch."""
import copy

import numpy as np
import torch

from . import _native
from .params import Params
from .vec_env import Drone2DVecEnv
from .world import generate_worlds


def survivability_positions(params, position_step=60):
    lo = params.map_scale + params.drone_radius
    xs = list(range(lo, params.map_size[0] - params.map_scale - params.drone_radius, position_step))
    ys = list(range(lo, params.map_size[1] - params.map_scale - params.drone_radius, position_step))
    return xs, ys


def global_survivability(params, seeds, T=24, position_step=60, device="cuda:0"):
    """Returns collision_state uint8 [len(seeds), len(xs), len(ys), int(T / dt)] (numpy)."""
    if params.planner != "NoMove":
        raise ValueError("the metric is defined with planner='NoMove' (glob_survivability_calculator.py:20)")
    xs, ys = survivability_positions(params, position_step)
    seeds = np.asarray(seeds, dtype=np.int64)
    nw, npos = len(seeds), len(xs) * len(ys)
    steps = int(T / params.dt)
    w = generate_worlds(params, seeds)
    worlds = {k: np.repeat(v, npos, axis=0) for k, v in w.items()}          # env = world * npos + position
    env = Drone2DVecEnv(params, nw * npos, seeds=np.repeat(seeds, npos), worlds=worlds, device=device, auto_reset=False,
                        trackers=True, oxford=False)
    pose = worlds["drone_pose"].copy()
    grid = np.array([(x, y) for x in xs for y in ys], dtype=np.float64)
    pose[:, 0] = np.tile(grid[:, 0], nw)
    pose[:, 1] = np.tile(grid[:, 1], nw)
    env.set_drone_pose(pose)            # NoMove never moves the drone, so pinning once == pinning before every step
    zero = torch.zeros(nw * npos, dtype=torch.float64, device=env.device)
    out = torch.zeros((steps, nw * npos), dtype=torch.uint8, device=env.device)
    col = env.buffer("collision_flag")
    # the reference walks `for t in np.arange(0, T, 0.1)` and writes slot int(t / 0.1) (glob_survivability_calculator.py:34-39):
    # t is k * 0.1 rounded, so for some k the slot is k - 1 (T = 24: k = 43, 81, 86, ...) -- that slot then collects two
    # steps and slot k stays 0.  Reproduced, not corrected.
    slots = [int(t / 0.1) for t in np.arange(0, T, 0.1)][:steps]
    for k in range(len(slots)):
        env.step(zero)
        out[slots[k]] |= (col == 2).to(torch.uint8)
    res = out.cpu().numpy().T.reshape(nw, len(xs), len(ys), steps)
    env.close()
    return res


def mean_survival_time(collision_state, dt=0.1):
    """Time of the first dynamic collision per (world, position), T if none -- the quantity survivability_calculator.py
    averages (utils of the paper's 'survivability' metric)."""
    steps = collision_state.shape[-1]
    hit = collision_state.astype(bool)
    first = np.where(hit.any(-1), hit.argmax(-1), steps)
    return first * dt


def survivability(params, seeds, T=12, position_step=60, device="cuda:0"):
    """script/difficulty_calculator/survivability_calculator.py:13-48 for every seed at once.  The reference builds one
    NoMove env per world, steps it once, then for t in np.arange(0, T, 0.1): marks every position of the 8x8 grid that lies
    inside an agent disc grown by the drone radius (`norm(agent.position - p) < agent.radius + drone.radius`) with
    min(t, ...), and steps again (it keeps stepping after `done`; nothing is reset).  Returns (survive_times
    float64 [len(seeds), len(xs), len(ys)], mean per seed) with the script's post-processing (-0.1, clamped at 0).
    One env per world here; the 64 positions are evaluated from the agent positions on the device."""
    if params.planner != "NoMove":
        raise ValueError("the metric is defined with planner='NoMove' (survivability_calculator.py:20)")
    xs, ys = survivability_positions(params, position_step)
    seeds = np.asarray(seeds, dtype=np.int64)
    nw = len(seeds)
    env = Drone2DVecEnv(params, nw, seeds=seeds, device=device, auto_reset=False, trackers=True, oxford=False)
    dev = env.device
    grid = torch.tensor([(x, y) for x in xs for y in ys], dtype=torch.float64, device=dev)        # [P, 2]
    zero = torch.zeros(nw, dtype=torch.float64, device=dev)
    pos, rad = env.buffer("agent_pos"), env.buffer("agent_radius")
    ts = np.arange(0, T, 0.1)
    first = torch.full((nw, grid.shape[0]), len(ts), dtype=torch.int64, device=dev)               # index of the first hit
    env.step(zero)
    for i in range(len(ts)):
        dx = pos[:, :, None, 0] - grid[None, None, :, 0]
        dy = pos[:, :, None, 1] - grid[None, None, :, 1]
        hit = (torch.sqrt(dx * dx + dy * dy) < (rad + float(params.drone_radius))[:, :, None]).any(1)   # [nw, P]
        first = torch.where(hit & (first == len(ts)), torch.full_like(first, i), first)
        env.step(zero)
    first = first.cpu().numpy()
    env.close()
    tv = np.concatenate([ts, [float(T)]])               # never hit: stays at T (np.ones(...) * T)
    st = tv[first].reshape(nw, len(xs), len(ys)) - 0.1
    st[st < 0] = 0
    return st, st.reshape(nw, -1).mean(1)


def obstacle_density(params, seeds):
    """script/difficulty_calculator/density_calculator.py:13-30: sum of 3.14 * r^2 over the agents / map area (host only)."""
    w = generate_worlds(params, np.asarray(seeds, dtype=np.int64))
    return _density(params, w["agent_radius"])


def _density(params, agent_radius):
    out = []
    for radii in agent_radius:
        area = 0
        for r in radii.tolist():        # the script's own accumulation order and scalar `**` (libm pow)
            area += 3.14 * r ** 2
        out.append(area / (params.map_size[0] * params.map_size[1]))
    return np.array(out)


def global_slots(T, dt, steps):
    """The slot table of `global_survivability` for a difficulty call of `steps` agent steps: (n_slots, table) with
    n_slots = int(T / dt) and table[k-1] the slot agent step k writes -- the script's int(t / 0.1), doubled slots included
    -- or DIFF_NO_SLOT for the steps beyond the script's loop."""
    n_slots = int(T / dt)
    table = [int(t / 0.1) for t in np.arange(0, T, 0.1)][:n_slots]
    return n_slots, table[:steps] + [_native.DIFF_NO_SLOT] * (steps - len(table))


def survival_from_hits(first_hit, static_hit, T_survivability, n_slots, table):
    """survivability, its per-seed mean and the global survival time from d2d_difficulty's outputs (first_hit int [S, ...],
    static_hit bool [S, ...]) and the slot table of `global_slots`, with the scripts' own host arithmetic."""
    fh = np.asarray(first_hit, dtype=np.int64)
    S = fh.shape[0]
    # survivability_calculator.py: loop index i (time ts[i]) sees the state after agent step i + 1
    ts = np.arange(0, T_survivability, 0.1)
    L = len(ts)
    tv = np.concatenate([ts, [float(T_survivability)]])
    st = tv[np.where((fh >= 1) & (fh <= L), fh - 1, L)] - 0.1
    st[st < 0] = 0
    # mean_survival_time: the first slot written -- slots never decrease, so the slot of the first dynamic hit -- unless
    # the position is static, where collision_flag is never 2
    tab = np.array(list(table) + [_native.DIFF_NO_SLOT], dtype=np.int64)
    slot = tab[np.where(fh >= 1, fh - 1, len(table))]
    first = np.where(np.asarray(static_hit, dtype=bool) | (slot == _native.DIFF_NO_SLOT), n_slots, slot)
    return {"survivability": st, "mean_survivability": st.reshape(S, -1).mean(1), "global_survival_time": first * 0.1}


def difficulty(params, seeds, T_global=24, T_survivability=12, position_step=60, num_envs=65536, world_gen="device",
               collision_state=False, device="cuda:0"):
    """`survivability`, `global_survivability` (as `mean_survival_time`) and `obstacle_density` of every seed from ONE
    kernel per chunk of seeds (d2d_difficulty): the agents are stepped alone from each world's reset state and every grid
    position is tested after every step, the way both scripts test it.  Under CVM no agent looks at the drone, so one agent
    trajectory per world answers all positions.  The seeds stream through one scratch handle of min(num_envs, len(seeds))
    NoMove envs; each chunk is an eager `reseed` (world_gen="device") or `set_worlds` (world_gen="host") and one
    `difficulty` call into preallocated device outputs, with one synchronisation at the end.  Any planner (the scratch
    handle is NoMove, as in the scripts); CVM only (RVO: use the functions above).
    Returns a dict of numpy arrays, S = len(seeds):
      survivability        float64 [S, nx, ny]  == survivability(params, seeds, T_survivability, position_step)[0]
      mean_survivability   float64 [S]          == its second output
      global_survival_time float64 [S, nx, ny]  == mean_survival_time(global_survivability(params, seeds, T_global, ...))
      density              float64 [S]          == obstacle_density(params, seeds)
      collision_state      uint8 [S, nx, ny, int(T_global / dt)] == global_survivability(...), with collision_state=True.
    Device worlds equal host worlds except for the documented group-velocity rounding of static-map agents (DESIGN.md
    section 2).
    `params` may be a list of K configs (world_gen="device" only): every key then has a leading config axis, [K, S, ...],
    equal to the per-config calls stacked.  The configs are split into batch groups (experiment.batch_groups of their
    NoMove scratch configs); each group streams its (config, seed) pairs through one scratch handle with keyed `reseed`
    chunks.  The configs must share the position grid and dt (the output shapes)."""
    if world_gen not in ("host", "device"):
        raise ValueError("world_gen must be 'host' or 'device', got %r" % (world_gen,))
    kw = dict(T_global=T_global, T_survivability=T_survivability, position_step=position_step, num_envs=num_envs,
              collision_state=collision_state, device=device)
    if not isinstance(params, (list, tuple)):
        return _difficulty([_scratch(params)], np.asarray(seeds, dtype=np.int64).reshape(-1), world_gen=world_gen, **kw)
    if world_gen != "device":
        raise ValueError("difficulty over a list of configs generates the worlds on the device (world_gen='device')")
    from .experiment import batch_groups
    from .world import world_key
    configs = [_scratch(p) for p in params]
    seeds = np.asarray(seeds, dtype=np.int64).reshape(-1)
    K, S = len(configs), len(seeds)
    if K == 0 or S == 0:
        raise ValueError("difficulty: no configs or no seeds")
    res = None
    for group in batch_groups(configs):
        keys = world_key(np.repeat(np.arange(len(group)), S), np.tile(seeds, len(group)))
        r = _difficulty([configs[k] for k in group], keys, world_gen="device", **kw)
        if res is None:
            res = {n: np.empty((K, S) + v.shape[1:], v.dtype) for n, v in r.items()}
        for n, v in r.items():
            if v.shape[1:] != res[n].shape[2:]:
                raise ValueError("difficulty: configs %s give %s of shape %s, others %s (position grid or dt differ)"
                                 % (group, n, v.shape[1:], res[n].shape[2:]))
            res[n][group] = v.reshape((len(group), S) + v.shape[1:])
    return res


def _scratch(p):
    """The scratch config of the difficulty handle: NoMove, as both scripts; the worlds and the agents do not depend on
    the planner.  The handle runs no gaze policy, so one gaze value keeps the gaze out of the batch grouping."""
    p = copy.copy(p)
    p.planner = "NoMove"
    p.gaze_method = "LookAhead"
    return p


def _difficulty(configs, seeds, T_global, T_survivability, position_step, num_envs, world_gen, collision_state, device):
    """difficulty over `seeds` on one scratch handle: world seeds of configs[0] (one config), or world keys over
    `configs` (one batch group, world_gen="device")."""
    params = configs[0]
    keyed = len(configs) > 1            # else the keys of source 0 are the seeds
    xs, ys = survivability_positions(params, position_step)
    nx, ny = len(xs), len(ys)
    S = len(seeds)
    ts = np.arange(0, T_survivability, 0.1)
    steps = max(int(T_global / params.dt), len(ts))
    n_slots, table = global_slots(T_global, params.dt, steps)
    B = min(int(num_envs), S)
    if B == 0 or nx * ny == 0:
        raise ValueError("difficulty: no seeds or an empty position grid")
    grid = (xs[0], ys[0], position_step, nx, ny)
    if keyed:
        from .world import split_world_key
        src, sd = split_world_key(seeds)
        env = Drone2DVecEnv(params, B, seeds=sd[:B], device=device, auto_reset=False, trackers=False, oxford=False,
                            owl=False, world_gen="device", world_sources=configs, sources=src[:B])
    else:
        env = Drone2DVecEnv(params, B, seeds=seeds[:B], device=device, auto_reset=False, trackers=False, oxford=False,
                            owl=False, world_gen=world_gen)
    try:
        dev = env.device
        first_hit = torch.empty((S, nx, ny), dtype=torch.int16, device=dev)
        static_hit = torch.empty((S, nx, ny), dtype=torch.uint8, device=dev)
        cs = torch.empty((S, nx, ny, n_slots), dtype=torch.uint8, device=dev) if collision_state else None
        radius = torch.empty((S, env.num_agents), dtype=torch.float64, device=dev)
        for c0 in range(0, S, B):
            n = min(B, S - c0)
            if c0 > 0:
                if keyed:
                    env.reseed(np.arange(n), sd[c0:c0 + n], sources=src[c0:c0 + n])
                elif world_gen == "device":
                    env.reseed(np.arange(n), seeds[c0:c0 + n])
                else:
                    torch.cuda.current_stream(dev).synchronize()      # the last call has read the snapshot it replaces
                    env.set_worlds(generate_worlds(params, seeds[c0:c0 + n], env._smap))
            out = (first_hit[c0:c0 + n], static_hit[c0:c0 + n]) + ((cs[c0:c0 + n],) if collision_state else ())
            env.difficulty(steps, grid, envs=range(0, n), slots=table, n_slots=n_slots, collision_state=collision_state,
                           out=out)
            radius[c0:c0 + n] = env.buffer("agent_radius")[:n]
        torch.cuda.current_stream(dev).synchronize()
        env.check_worlds()
        fh = first_hit.cpu().numpy().astype(np.int64)
        sh = static_hit.cpu().numpy().astype(bool)
        rad = radius.cpu().numpy()
        cs = cs.cpu().numpy() if collision_state else None
    finally:
        env.close()
    res = survival_from_hits(fh, sh, T_survivability, n_slots, table)
    res["density"] = _density(params, rad)
    if collision_state:
        res["collision_state"] = cs
    return res
