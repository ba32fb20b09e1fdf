"""`Experiment`: the reference's episode driver (experiment.py:26-106) on the device-backed facade, plus a batched
runner that plays many seeded episodes at once and reports the same per-episode statistics as totals."""
import os

import numpy as np

from . import _native
from .env import make
from .params import state_machine
from .policies import policy_list

CSV_COLUMNS = ["Method", "Planner", "Motion Profile", "Map ID", "Agent size", "Number of agents", "Number of pillars",
               "Agent speed", "Drone speed", "Depth variance", "Initial position", "Target position", "Flight time",
               "Grid discovered", "Agent tracked", "Agent tracked time", "Success", "Static Collision",
               "Dynamic Collision", "Freezing", "Dead Lock", "state machine"]


class Experiment(object):
    def __init__(self, params, dir=None):
        if params.gaze_method == "NoControl":
            params.drone_view_range = 360                        # experiment.py:28-29
        self.params = params
        self.env = make(params.env, params=params)
        self.dt = params.dt
        self.policy = policy_list[params.gaze_method](params)
        self.result_dir = dir
        self.rows = []

    def run(self, max_steps=None):
        """One episode (experiment.py:65-106); returns the CSV row as a dict (and appends it to `dir` if recording)."""
        self.env.reset()
        done, n = False, 0
        info = self.env.info
        while not done:
            a = self.policy.plan(info)
            _, _, done, info = self.env.step(a)
            n += 1
            if max_steps is not None and n >= max_steps:
                break
        p = self.params
        buf = info["tracker_buffer"]
        tracking_time = float(np.array([len(t.ts) * 0.1 for t in buf]).sum())
        grid = info["drone"].map.grid_map
        row = dict(zip(CSV_COLUMNS, [
            p.gaze_method, p.planner, p.motion_profile, p.map_id, p.agent_radius, p.agent_number, p.pillar_number,
            p.agent_max_speed, p.drone_max_speed, p.var_cam, p.init_position, p.target_list[0], info["flight_time"],
            int(grid.shape[0] * grid.shape[1] - np.sum(grid == 0)), len(buf),
            tracking_time / len(buf) if len(buf) else float("nan"),
            1 if info["state_machine"] == state_machine["GOAL_REACHED"] else 0, 1 if info["collision_flag"] == 1 else 0,
            1 if info["collision_flag"] == 2 else 0, info["freezing_flag"], info["dead_lock_flag"], info["state_machine"]]))
        self.rows.append(row)
        if self.result_dir and getattr(p, "record", False):
            import pandas as pd
            df = pd.DataFrame([row])
            df.to_csv(self.result_dir, mode="a", index=False, header=not os.path.isfile(self.result_dir))
        return row


def run_batched(params, num_envs, steps, device="cuda:0", seeds=None):
    """Plays `steps` env-steps of `num_envs` seeded envs (auto-reset on) with the params' gaze method (Oxford, Owl,
    LookAhead, LookGoal, Rotating, NoControl) evaluated on the device.  Returns the statistics dict."""
    import torch
    from .vec_env import Drone2DVecEnv
    if params.gaze_method == "NoControl":
        params.drone_view_range = 360                            # experiment.py:28-29
    env = Drone2DVecEnv(params, num_envs, seeds=seeds, device=device, auto_reset=True,
                        oxford=params.gaze_method == "Oxford")
    out = torch.empty(num_envs, dtype=torch.float64, device=env.device)
    for _ in range(steps):
        env.step(env.plan_gaze(params.gaze_method, out))
    st = env.stats()
    env.close()
    return dict(zip(_native.STAT_NAMES, [int(v) for v in st]))


def run_batched_rows(params, num_envs, episodes=1, max_steps=100000, device="cuda:0", seeds=None, sync_every=64):
    """The reference's experiment loop (experiment.py:65-106: one env, one policy, one CSV row per episode) for `num_envs`
    seeded worlds at once: every env plays `episodes` episodes (auto-reset on, the gaze policy evaluated on the device) and
    every finished episode yields the row `Experiment.run` would have produced for that world -- same columns, same
    expressions ("Map ID" is the env's seed: the reference seeds its world with `map_id`).  Returns the rows in completion
    order; `row["_env"]` / `row["_episode"]` say which env and which of its episodes a row belongs to.  The rows are
    written on the device by the episode log and read every `sync_every` steps."""
    import torch
    from .vec_env import Drone2DVecEnv
    if params.gaze_method == "NoControl":
        params.drone_view_range = 360                            # experiment.py:28-29
    seeds = np.asarray(seeds if seeds is not None else params.map_id + np.arange(num_envs), dtype=np.int64)
    sync_every = max(1, int(sync_every))
    env = Drone2DVecEnv(params, num_envs, seeds=seeds, device=device, auto_reset=True,
                        oxford=params.gaze_method == "Oxford")
    try:
        env.enable_episode_log(num_envs * sync_every)
        act = torch.empty(num_envs, dtype=torch.float64, device=env.device)
        played = np.zeros(num_envs, dtype=np.int64)
        rows = []
        t = 0
        while t < max_steps and not (played >= episodes).all():
            k = min(sync_every, max_steps - t)
            for _ in range(k):
                env.step(env.plan_gaze(params.gaze_method, act))
            t += k
            recs, dropped = env.read_episodes()
            assert dropped == 0
            for r in recs:
                i = int(r["env"])
                if played[i] >= episodes:
                    continue
                row = episode_row(params, r)
                row["_env"], row["_episode"] = i, int(played[i])
                rows.append(row)
                played[i] += 1
    finally:
        env.close()
    return rows


def episode_row(p, rec):
    """The CSV row `Experiment.run` produces for the episode of one episode-log record (`_native.EPISODE_DTYPE`), read on
    the device by the step that reported done; "Map ID" is the seed of the record's world key (its low 32 bits)."""
    # 'Agent tracked time': the reference sums len(ts) * 0.1 per archived tracker (experiment.py:74, 94) and the float sum
    # depends on how the total splits over the trackers; the device keeps the count and the total only, so the column
    # is the reference's value up to that rounding (<= a few ulp; compared at 1e-9 against reference rows in the tests)
    n = int(rec["trackers"])
    base, rem = divmod(int(rec["tracked_steps"]), n) if n else (0, 0)
    tracking_time = float(np.array([(base + (1 if j < rem else 0)) * 0.1 for j in range(n)]).sum())
    sm, col = int(rec["state_machine"]), int(rec["collision_flag"])
    return dict(zip(CSV_COLUMNS, [
        p.gaze_method, p.planner, p.motion_profile, int(rec["seed"]) & 0xFFFFFFFF, p.agent_radius, p.agent_number, p.pillar_number,
        p.agent_max_speed, p.drone_max_speed, p.var_cam, p.init_position, p.target_list[0], int(rec["steps"]) * p.dt,
        int(rec["grid_discovered"]), n, tracking_time / n if n else float("nan"),
        1 if sm == state_machine["GOAL_REACHED"] else 0, 1 if col == 1 else 0, 1 if col == 2 else 0,
        int(rec["freezing_flag"]), int(rec["dead_lock_flag"]), sm]))


SWEEP_CHUNK = 64                        # steps between two reads of the episode log in run_config_sweep (one CUDA graph)


def _no_control_view(p):
    if p.gaze_method == "NoControl":
        p.drone_view_range = 360                                 # experiment.py:28-29


def batch_groups(configs):
    """Partitions `configs` (Params) into the groups that can share one handle: two configs share a batch exactly when
    their d2d_config structs (make_config, with the NoControl view-range rule applied; device and num_envs aside) are
    byte-equal and their gaze methods are the same.  What is left to differ only shapes the worlds -- the static map,
    agent_number at equal agent count, pillar_number, agent_max_speed, init_pos -- and travels per env as a world source.
    Returns lists of indices into `configs`, each in input order, the groups ordered by their first member."""
    import ctypes as C
    import copy
    from .vec_env import make_config
    from .world import count_agents
    groups = {}
    for k, p in enumerate(configs):
        q = copy.copy(p)
        _no_control_view(q)
        g = q.gaze_method
        cfg = make_config(q, 0, count_agents(q), 0, auto_reset=True, oxford=g == "Oxford", owl=g == "Owl")
        groups.setdefault((C.string_at(C.addressof(cfg), C.sizeof(cfg)), g), []).append(k)
    return list(groups.values())


def run_seed_sweep(params, seeds, num_envs, max_steps=1000000, device="cuda:0"):
    """A seed sweep (one reference experiment row per `(config, map_id)`, the map_id being the seed) streamed through a
    fixed batch of `num_envs` envs whose worlds are generated on the GPU: run_config_sweep([params], ...)[0].  Returns one
    row per entry of `seeds`, in that order (equal seeds give equal rows); a row equals the one `run_batched_rows` produces
    for that seed (on maps with static agents, up to the group-velocity rounding of device worlds, DESIGN.md section 2).
    `max_steps` bounds the number of batch steps (RuntimeError when reached)."""
    return run_config_sweep([params], seeds, num_envs, max_steps=max_steps, device=device)[0]


def run_config_sweep(configs, seeds, num_envs, max_steps=1000000, device="cuda:0"):
    """A sweep over configurations and seeds: rows[k][i] is the reference experiment row of `configs[k]` on map_id
    `seeds[i]`.  The configs are split into `batch_groups`; each group runs on one handle of min(num_envs, pairs) envs
    whose worlds are generated on the GPU from world keys (source = the config's index in its group, seed = map_id).  The
    first pairs are the envs' initial worlds, the rest a device-side queue of keys: an env that reports done takes the
    next key and starts that world at its next step, and its row is written by the episode log, all without the host.
    The host steps SWEEP_CHUNK steps at a time (replayed from a CUDA graph) and reads the log in between.  A row equals
    the one `run_seed_sweep(configs[k], seeds)` gives.  `max_steps` bounds the batch steps of each group (RuntimeError
    when reached).  Configs with the NoControl gaze get drone_view_range = 360, as the reference's Experiment does."""
    from .world import world_key
    configs = list(configs)
    for p in configs:
        _no_control_view(p)
    seeds = np.asarray(seeds, dtype=np.int64).reshape(-1)
    rows = [[None] * len(seeds) for _ in configs]
    if len(seeds) == 0:
        return rows
    for group in batch_groups(configs):
        keys = world_key(np.repeat(np.arange(len(group)), len(seeds)), np.tile(seeds, len(group)))
        by_key = _sweep_group([configs[k] for k in group], keys, num_envs, max_steps, device)
        for j, k in enumerate(group):
            rows[k] = [dict(by_key[int(x)]) for x in keys[j * len(seeds):(j + 1) * len(seeds)]]
    return rows


def _sweep_group(configs, keys, num_envs, max_steps, device):
    """{key: row} for world keys over `configs` (one batch group) on one handle, streamed through the keyed queue."""
    import torch
    from .vec_env import Drone2DVecEnv
    from .world import split_world_key
    p0 = configs[0]
    B = min(int(num_envs), len(keys))
    chunk = SWEEP_CHUNK
    src, sd = split_world_key(keys)
    env = Drone2DVecEnv(p0, B, seeds=sd[:B], device=device, auto_reset=True, oxford=p0.gaze_method == "Oxford",
                        world_gen="device", world_sources=configs, sources=src[:B])
    by_key = {}                         # key -> row of its first record
    want = set(keys.tolist())
    try:
        env.enable_episode_log(B * chunk)
        env.set_seed_queue(sd[B:], sources=src[B:])
        act = torch.empty(B, dtype=torch.float64, device=env.device)

        def steps(k):
            for _ in range(k):
                env.step(env.plan_gaze(p0.gaze_method, act))

        graph = None
        t = 0
        while len(by_key) < len(want):
            if t >= max_steps:
                raise RuntimeError("run_config_sweep: %d of %d worlds unfinished after %d steps"
                                   % (len(want) - len(by_key), len(want), max_steps))
            k = min(chunk, max_steps - t)
            if graph is None and t > 0 and k == chunk:
                # the first chunk ran eagerly (one-time set-up of the launch paths); the later ones replay its graph
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    steps(chunk)
                graph.replay()
            elif graph is not None and k == chunk:
                graph.replay()
            else:
                steps(k)
            t += k
            recs, dropped = env.read_episodes()
            assert dropped == 0
            for r in recs:
                key = int(r["seed"])
                if key in want and key not in by_key:
                    by_key[key] = episode_row(configs[key >> 32], r)
    finally:
        env.close()
    return by_key
