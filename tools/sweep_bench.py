"""Seed-sweep throughput and the per-step cost of the episode log (and of log + world generation under a seed queue).

    python tools/sweep_bench.py [--seeds-per-env 3] [--envs2 4096] [--envs4 4096] [--reps 3] [--out DIR]

1. Rows per second of experiment.run_seed_sweep (episode log + device seed queue, chunks replayed from a CUDA graph)
   against the host-synchronising loop it replaced (kept below as the baseline: read `done` after every step, copy the
   finished envs' buffers to the host, reseed lazily), alternated in the same process.  Both must give the same rows.
   Workloads: BASELINE config 2 geometry (empty_map, 10 agents radius 15, speed 20, NoMove) with LookAhead gaze, and config 4
   (obstacle_map, 10 agents radius 10, speed 20, Primitive planner + Oxford gaze).
2. Added time per step: CUDA events around graph replays of K plain steps (config 2, constant action) with no log, with the
   log, and with log + queue, at 4096 and 65536 envs.
The GPU name and power limit are read in the same run.  Needs a CUDA device (no CPU fallback)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                      # the device name from torch below still says what ran
        return "nvidia-smi unavailable (%s)" % e


def params(cfg, **kw):
    from gym_drone2d_activeperception_b200.params import Params
    if cfg == 2:
        base = dict(planner="NoMove", static_map="maps/empty_map.npy", agent_number=10, agent_radius=15, agent_max_speed=20,
                    gaze_method="LookAhead")
    else:
        base = dict(planner="Primitive", static_map="maps/obstacle_map.npy", agent_number=10, agent_radius=10,
                    agent_max_speed=20, gaze_method="Oxford")
    base.update(kw)
    return Params(debug=False, **base)


def baseline_sweep(p, seeds, num_envs, device="cuda:0"):
    """The previous run_seed_sweep: one host round trip (and a Python loop over the finished envs) per step."""
    import torch
    from gym_drone2d_activeperception_b200.experiment import CSV_COLUMNS
    from gym_drone2d_activeperception_b200.params import state_machine
    from gym_drone2d_activeperception_b200.vec_env import Drone2DVecEnv
    S = len(seeds)
    B = min(num_envs, S)
    env = Drone2DVecEnv(p, B, seeds=seeds[:B], device=device, auto_reset=True, oxford=p.gaze_method == "Oxford",
                        world_gen="device")
    act = torch.empty(B, dtype=torch.float64, device=env.device)
    job, nxt, rows, left = np.arange(B), B, [None] * S, S
    b = env.buffer
    while left:
        _, _, done, _ = env.step(env.plan_gaze(p.gaze_method, act))
        idx = torch.nonzero(done).flatten()
        if idx.numel() == 0:
            continue
        g = lambda name: b(name)[idx].cpu().numpy()
        steps, sm, col = g("steps"), g("state_machine"), g("collision_flag")
        frz, dead, cnt, tot = g("freezing_flag"), g("dead_lock_flag"), g("tracker_buffer_count"), g("tracker_buffer_ts")
        disc = (b("belief")[idx] != 0).sum((1, 2)).cpu().numpy()
        envs, new = [], []
        for k, i in enumerate(idx.cpu().numpy().tolist()):
            n = int(cnt[k])
            base, rem = divmod(int(tot[k]), n) if n else (0, 0)
            tt = float(np.array([(base + (1 if j < rem else 0)) * 0.1 for j in range(n)]).sum())
            row = dict(zip(CSV_COLUMNS, [
                p.gaze_method, p.planner, p.motion_profile, int(env.seeds[i]), p.agent_radius, p.agent_number,
                p.pillar_number, p.agent_max_speed, p.drone_max_speed, p.var_cam, p.init_position, p.target_list[0],
                int(steps[k]) * p.dt, int(disc[k]), n, tt / n if n else float("nan"),
                1 if sm[k] == state_machine["GOAL_REACHED"] else 0, 1 if col[k] == 1 else 0, 1 if col[k] == 2 else 0,
                int(frz[k]), int(dead[k]), int(sm[k])]))
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
    torch.cuda.synchronize()
    env.close()
    return rows


def same_rows(a, b):
    if len(a) != len(b):
        return False
    for x, y in zip(a, b):
        for k in x:
            if not (x[k] == y[k] or (isinstance(y[k], float) and y[k] != y[k] and x[k] != x[k])):
                return False
    return True


def sweep_rates(cfg, B, per_env, reps):
    import torch
    from gym_drone2d_activeperception_b200.experiment import run_seed_sweep
    seeds = 1 + np.arange(B * per_env, dtype=np.int64)
    out = {"config": cfg, "envs": B, "seeds": len(seeds), "new_rows_per_s": [], "baseline_rows_per_s": []}
    rows = {}
    run_seed_sweep(params(cfg), seeds[:2 * B], B)           # untimed: first launches, graph capture path, module loads
    baseline_sweep(params(cfg), seeds[:2 * B], B)
    for r in range(reps):
        for name in ("new", "baseline"):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            got = run_seed_sweep(params(cfg), seeds, B) if name == "new" else baseline_sweep(params(cfg), seeds, B)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            out[name + "_rows_per_s"].append(len(seeds) / dt)
            rows[name] = got
    out["rows_equal"] = same_rows(rows["new"], rows["baseline"])
    return out


def step_cost(B, K, reps):
    """Per-step device time of K-step graphs: plain, + episode log, + log and seed queue (config 2, constant action)."""
    import torch
    from gym_drone2d_activeperception_b200.vec_env import Drone2DVecEnv
    res = {"envs": B, "graph_steps": K}
    for mode in ("plain", "log", "log+queue"):
        env = Drone2DVecEnv(params(2), B, seeds=np.arange(B), world_gen="device")
        if mode != "plain":
            env.enable_episode_log(B * K)
        if mode == "log+queue":
            env.set_seed_queue(10 ** 6 + np.arange(2 * 10 ** 6, dtype=np.int64))
        act = torch.full((B,), 1.0 / 3, dtype=torch.float64, device=env.device)
        for _ in range(4):
            env.step(act)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(K):
                env.step(act)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ms, episodes = 0.0, 0
        for r in range(reps + 1):
            ev[0].record()
            g.replay()
            ev[1].record()
            torch.cuda.synchronize()
            if r:                                   # the first replay is warm-up
                ms += ev[0].elapsed_time(ev[1])
            if mode != "plain":
                recs, dropped = env.read_episodes()
                assert dropped == 0
                episodes += len(recs) if r else 0
        res[mode + "_us_per_step"] = 1e3 * ms / (reps * K)
        if mode != "plain":
            res[mode + "_episodes_per_step"] = episodes / (reps * K)
        env.close()
    res["log_added_us_per_step"] = res["log_us_per_step"] - res["plain_us_per_step"]
    res["log_queue_added_us_per_step"] = res["log+queue_us_per_step"] - res["plain_us_per_step"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seeds-per-env", type=int, default=3)
    ap.add_argument("--envs2", type=int, default=4096)
    ap.add_argument("--envs4", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--graph-steps", type=int, default=64)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("sweep_bench: needs a CUDA device")
    res = {"gpu": gpu_info(), "device": torch.cuda.get_device_name(0), "sweeps": [], "step_cost": []}
    for B in (4096, 65536):
        res["step_cost"].append(step_cost(B, a.graph_steps, 10))
        print(json.dumps(res["step_cost"][-1]), flush=True)
    for cfg, B in ((2, a.envs2), (4, a.envs4)):
        res["sweeps"].append(sweep_rates(cfg, B, a.seeds_per_env, a.reps))
        print(json.dumps(res["sweeps"][-1]), flush=True)
    print(json.dumps(res))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "sweep_bench.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
