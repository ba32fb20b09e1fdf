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


def run_batched_rows(params, num_envs, episodes=1, max_steps=100000, device="cuda:0", seeds=None):
    """The reference's experiment loop (experiment.py:65-106: one env, one policy, one CSV row per episode) for `num_envs`
    seeded worlds at once: every env plays `episodes` episodes (auto-reset on, the gaze policy evaluated on the device) and
    every finished episode yields the row `Experiment.run` would have produced for that world -- same columns, same
    expressions ("Map ID" is the env's seed: the reference seeds its world with `map_id`).  Returns the rows in completion
    order; `row["_env"]` / `row["_episode"]` say which env and which of its episodes a row belongs to."""
    import torch
    from .vec_env import Drone2DVecEnv
    if params.gaze_method == "NoControl":
        params.drone_view_range = 360                            # experiment.py:28-29
    seeds = np.asarray(seeds if seeds is not None else params.map_id + np.arange(num_envs), dtype=np.int64)
    env = Drone2DVecEnv(params, num_envs, seeds=seeds, device=device, auto_reset=True,
                        oxford=params.gaze_method == "Oxford")
    act = torch.empty(num_envs, dtype=torch.float64, device=env.device)
    played = np.zeros(num_envs, dtype=np.int64)
    rows = []
    p = params
    for _ in range(max_steps):
        _, _, done, _ = env.step(env.plan_gaze(p.gaze_method, act))
        idx = torch.nonzero(done).flatten()
        if idx.numel() == 0:
            continue
        # everything a row needs is still in place right after the step that reported done (the reset is lazy)
        for i, row in _done_rows(env, p, idx, seeds):
            if played[i] >= episodes:
                continue
            row["_env"], row["_episode"] = i, int(played[i])
            rows.append(row)
            played[i] += 1
        if (played >= episodes).all():
            break
    env.close()
    return rows


def _done_rows(env, p, idx, seeds):
    """(env, CSV row) for every env in `idx` (a CUDA index tensor of envs that just reported done): the row
    `Experiment.run` produces for that episode, read from the buffers right after the step that reported done."""
    b = env.buffer
    g = lambda name: b(name)[idx].cpu().numpy()
    steps, sm, col = g("steps"), g("state_machine"), g("collision_flag")
    frz, dead, cnt, tot = g("freezing_flag"), g("dead_lock_flag"), g("tracker_buffer_count"), g("tracker_buffer_ts")
    disc = (b("belief")[idx] != 0).sum((1, 2)).cpu().numpy()
    out = []
    for k, i in enumerate(idx.cpu().numpy().tolist()):
        # 'Agent tracked time': the reference sums len(ts) * 0.1 per archived tracker (experiment.py:74, 94) and the float sum
        # depends on how the total splits over the trackers; the device keeps the count and the total only, so the column
        # is the reference's value up to that rounding (<= a few ulp; compared at 1e-9 against reference rows in the tests)
        n = int(cnt[k])
        base, rem = divmod(int(tot[k]), n) if n else (0, 0)
        tracking_time = float(np.array([(base + (1 if j < rem else 0)) * 0.1 for j in range(n)]).sum())
        row = dict(zip(CSV_COLUMNS, [
            p.gaze_method, p.planner, p.motion_profile, int(seeds[i]), p.agent_radius, p.agent_number, p.pillar_number,
            p.agent_max_speed, p.drone_max_speed, p.var_cam, p.init_position, p.target_list[0], int(steps[k]) * p.dt,
            int(disc[k]), n, tracking_time / n if n else float("nan"),
            1 if sm[k] == state_machine["GOAL_REACHED"] else 0, 1 if col[k] == 1 else 0, 1 if col[k] == 2 else 0,
            int(frz[k]), int(dead[k]), int(sm[k])]))
        out.append((i, row))
    return out


def run_seed_sweep(params, seeds, num_envs, max_steps=1000000, device="cuda:0"):
    """A seed sweep (one reference experiment row per `(config, map_id)`, the map_id being the seed) streamed through a
    fixed batch of `num_envs` envs whose worlds are generated on the GPU: when an env reports done its row is read and
    the env is reseeded lazily with the next seed, so it starts that world at its next step.  Any number of seeds, one
    handle of `num_envs` envs.  Returns one row per entry of `seeds`, in that order; a row equals the one
    `run_batched_rows` produces for that seed (on maps with static agents, up to the group-velocity rounding of device
    worlds, DESIGN.md section 2).  `max_steps` bounds the number of batch steps (RuntimeError when reached)."""
    import torch
    from .vec_env import Drone2DVecEnv
    if params.gaze_method == "NoControl":
        params.drone_view_range = 360                            # experiment.py:28-29
    seeds = np.asarray(seeds, dtype=np.int64).reshape(-1)
    S = len(seeds)
    if S == 0:
        return []
    B = min(int(num_envs), S)
    env = Drone2DVecEnv(params, B, seeds=seeds[:B], device=device, auto_reset=True, oxford=params.gaze_method == "Oxford",
                        world_gen="device")
    act = torch.empty(B, dtype=torch.float64, device=env.device)
    job = np.arange(B)                  # index into `seeds` of the episode each env is playing (-1: idle)
    nxt = B
    rows = [None] * S
    left = S
    try:
        for _ in range(max_steps):
            _, _, done, _ = env.step(env.plan_gaze(params.gaze_method, act))
            idx = torch.nonzero(done).flatten()
            if idx.numel() == 0:
                continue
            envs, new = [], []
            for i, row in _done_rows(env, params, idx, env.seeds):
                if job[i] < 0:
                    continue
                rows[job[i]] = row
                left -= 1
                if nxt < S:
                    job[i] = nxt
                    envs.append(i)
                    new.append(seeds[nxt])
                    nxt += 1
                else:
                    job[i] = -1
            if envs:
                env.reseed(envs, new, lazy=True)
            if left == 0:
                break
        else:
            raise RuntimeError("run_seed_sweep: %d of %d seeds unfinished after %d steps" % (left, S, max_steps))
        torch.cuda.current_stream(env.device).synchronize()
        env.check_worlds()
    finally:
        env.close()
    return rows
