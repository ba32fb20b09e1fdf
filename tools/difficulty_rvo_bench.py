"""Time the survivability difficulty metrics of RVO worlds on the GPU.

    python tools/difficulty_rvo_bench.py [--out DIR] [--worlds 65536] [--old-worlds 1024] [--min-ms 100]

1. `metrics.difficulty` on --worlds RVO device worlds (N = 10 agents, 4 pillars, T = 24 / 12, the 64-position grid): one
   scratch handle of all worlds (one eager chunk of 240 x (step + grid_hits)), and a handle of a quarter of them (an eager
   chunk, then three replays of the captured graph).  Each is a host clock around work that ends in a device synchronise.
2. The route that existed before: `global_survivability` (one env per world and position) + `survivability` on the first
   --old-worlds seeds, timed the same way and compared with (1) on those seeds.
3. Kernel time: CUDA events around back-to-back calls lasting at least --min-ms on the full handle -- `grid_hits` with
   and without collision_state, and one RVO `step` (d2d_rvo_kernel + the NoMove step kernel) for scale.
The card's name, power limit and maximum SM clock are read in the same run.  Needs a CUDA device (no CPU fallback)."""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools.difficulty_bench import gpu_info, time_calls  # noqa: E402


def params():
    from gym_drone2d_activeperception_b200.params import Params
    return Params(debug=False, planner="NoMove", gaze_method="NoControl", motion_profile="RVO", agent_number=10,
                  agent_radius=15, agent_max_speed=20, pillar_number=4)


def timed(torch, fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return r, time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for difficulty_rvo_bench.json")
    ap.add_argument("--worlds", type=int, default=65536)
    ap.add_argument("--old-worlds", type=int, default=1024)
    ap.add_argument("--min-ms", type=float, default=100.0)
    args = ap.parse_args()
    import torch
    from gym_drone2d_activeperception_b200 import metrics
    from gym_drone2d_activeperception_b200.vec_env import Drone2DVecEnv
    if not torch.cuda.is_available():
        raise SystemExit("difficulty_rvo_bench needs a CUDA device")
    info = gpu_info()
    print(info)
    rows = []
    p = params()
    S = args.worlds
    seeds = np.arange(S)

    def row(r):
        rows.append(r)
        print(json.dumps(r), flush=True)

    # ---- 1. metrics.difficulty, RVO device worlds
    metrics.difficulty(p, seeds[:64], num_envs=16)         # one-time set-up (module load, graph path) outside the timing
    new = None
    for B in (S, S // 4):
        ts = []
        for _ in range(2):
            r, dt = timed(torch, lambda: metrics.difficulty(p, seeds, num_envs=B))
            ts.append(dt)
            new = new or r
        row({"case": "metrics.difficulty, %d RVO device worlds, num_envs %d, N = 10, 4 pillars, T = 24 / 12, 64 positions"
                     % (S, B), "seconds": [round(x, 3) for x in ts], "us_per_world": round(min(ts) / S * 1e6, 2)})

    # ---- 2. the step-kernel route on a subset
    n = args.old_worlds
    sub = seeds[:n]
    metrics.survivability(p, sub[:4])
    ts, same = [], None
    for _ in range(2):
        (cs, (st, _)), dt = timed(torch, lambda: (metrics.global_survivability(p, sub), metrics.survivability(p, sub)))
        ts.append(dt)
    same = {"global_survival_time": bool(np.array_equal(new["global_survival_time"][:n], metrics.mean_survival_time(cs))),
            "survivability_positions_differing": int((new["survivability"][:n] != st).sum())}
    row({"case": "global_survivability + survivability, %d RVO host worlds (%d envs)" % (n, n * 64),
         "seconds": [round(x, 3) for x in ts], "us_per_world": round(min(ts) / n * 1e6, 2)})
    row({"case": "outputs of both routes on the %d shared worlds" % n, **same})

    # ---- 3. kernel time on the full handle
    grid = (20, 20, 60, 8, 8)
    n_slots, table = metrics.global_slots(24, 0.1, 240)
    env = Drone2DVecEnv(p, S, device="cuda:0", auto_reset=False, trackers=False, oxford=False, owl=False,
                        world_gen="device")
    zero = torch.zeros(S, dtype=torch.float64, device="cuda:0")
    out = (torch.empty((S, 8, 8), dtype=torch.int16, device="cuda"), torch.empty((S, 8, 8), dtype=torch.uint8, device="cuda"),
           torch.empty((S, 8, 8, n_slots), dtype=torch.uint8, device="cuda"))
    env.step(zero)
    env.grid_hits(1, grid, slots=table, n_slots=n_slots, collision_state=True, out=out)
    for with_cs in (False, True):
        o = out if with_cs else out[:2]
        ms = time_calls(torch, lambda: env.grid_hits(2, grid, slots=table, n_slots=n_slots, collision_state=with_cs, out=o),
                        args.min_ms)
        row({"case": "grid_hits kernel, %d envs, N = %d, 64 positions%s" % (S, env.num_agents,
                                                                           ", collision_state" if with_cs else ""),
             "ms_per_call": round(ms, 4)})
    ms = time_calls(torch, lambda: env.step(zero), args.min_ms)
    row({"case": "RVO step (d2d_rvo_kernel + NoMove step kernel), %d envs, N = %d" % (S, env.num_agents),
         "ms_per_call": round(ms, 4)})
    env.close()
    res = {"gpu": info, "rows": rows}
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "difficulty_rvo_bench.json"), "w") as f:
            json.dump(res, f, indent=1)
    if not same["global_survival_time"]:
        raise SystemExit("outputs differ: %s" % same)


if __name__ == "__main__":
    main()
