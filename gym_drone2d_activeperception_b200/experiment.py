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
    the device by the step that reported done; "Map ID" is the record's seed."""
    # 'Agent tracked time': the reference sums len(ts) * 0.1 per archived tracker (experiment.py:74, 94) and the float sum
    # depends on how the total splits over the trackers; the device keeps the count and the total only, so the column
    # is the reference's value up to that rounding (<= a few ulp; compared at 1e-9 against reference rows in the tests)
    n = int(rec["trackers"])
    base, rem = divmod(int(rec["tracked_steps"]), n) if n else (0, 0)
    tracking_time = float(np.array([(base + (1 if j < rem else 0)) * 0.1 for j in range(n)]).sum())
    sm, col = int(rec["state_machine"]), int(rec["collision_flag"])
    return dict(zip(CSV_COLUMNS, [
        p.gaze_method, p.planner, p.motion_profile, int(rec["seed"]), p.agent_radius, p.agent_number, p.pillar_number,
        p.agent_max_speed, p.drone_max_speed, p.var_cam, p.init_position, p.target_list[0], int(rec["steps"]) * p.dt,
        int(rec["grid_discovered"]), n, tracking_time / n if n else float("nan"),
        1 if sm == state_machine["GOAL_REACHED"] else 0, 1 if col == 1 else 0, 1 if col == 2 else 0,
        int(rec["freezing_flag"]), int(rec["dead_lock_flag"]), sm]))


SWEEP_CHUNK = 64                        # steps between two reads of the episode log in run_seed_sweep (one CUDA graph)


def run_seed_sweep(params, seeds, num_envs, max_steps=1000000, device="cuda:0"):
    """A seed sweep (one reference experiment row per `(config, map_id)`, the map_id being the seed) streamed through a
    fixed batch of `num_envs` envs whose worlds are generated on the GPU.  The first `num_envs` seeds are the envs' initial
    worlds, the rest a device-side seed queue: an env that reports done takes the next seed and starts that world at its
    next step, and its row is written by the episode log, all without the host.  The host steps SWEEP_CHUNK steps at a time
    (replayed from a CUDA graph) and reads the log in between.  Any number of seeds, one handle of `num_envs` envs.  Returns
    one row per entry of `seeds`, in that order (equal seeds give equal rows); a row equals the one `run_batched_rows`
    produces for that seed (on maps with static agents, up to the group-velocity rounding of device worlds, DESIGN.md
    section 2).  `max_steps` bounds the number of batch steps (RuntimeError when reached)."""
    import torch
    from .vec_env import Drone2DVecEnv
    if params.gaze_method == "NoControl":
        params.drone_view_range = 360                            # experiment.py:28-29
    seeds = np.asarray(seeds, dtype=np.int64).reshape(-1)
    S = len(seeds)
    if S == 0:
        return []
    B = min(int(num_envs), S)
    chunk = SWEEP_CHUNK
    env = Drone2DVecEnv(params, B, seeds=seeds[:B], device=device, auto_reset=True, oxford=params.gaze_method == "Oxford",
                        world_gen="device")
    by_seed = {}                        # seed -> row of its first record
    want = set(seeds.tolist())
    try:
        env.enable_episode_log(B * chunk)
        env.set_seed_queue(seeds[B:])
        act = torch.empty(B, dtype=torch.float64, device=env.device)

        def steps(k):
            for _ in range(k):
                env.step(env.plan_gaze(params.gaze_method, act))

        graph = None
        t = 0
        while len(by_seed) < len(want):
            if t >= max_steps:
                raise RuntimeError("run_seed_sweep: %d of %d seeds unfinished after %d steps"
                                   % (len(want) - len(by_seed), len(want), max_steps))
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
                sd = int(r["seed"])
                if sd in want and sd not in by_seed:
                    by_seed[sd] = episode_row(params, r)
    finally:
        env.close()
    return [dict(by_seed[int(sd)]) for sd in seeds]
