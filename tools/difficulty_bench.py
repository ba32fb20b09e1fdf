"""Time the survivability difficulty metrics on the GPU.

    python tools/difficulty_bench.py [--out DIR] [--seeds 4096] [--min-ms 100]

1. Seeds per second: `metrics.difficulty` (device worlds, one d2d_difficulty call per chunk) against the step-kernel path
   `global_survivability` + `survivability` + `obstacle_density` (host worlds) on the same seeds, alternated twice in this
   process; each is a host clock around work that ends in a device synchronise.  The outputs are compared.
2. Kernel time: CUDA events around back-to-back `difficulty` calls lasting at least --min-ms, on 65 536 device worlds,
   240 agent steps (T = 24), the 64-position grid, with and without collision_state, for N = 10 agents on the empty map
   and N = 142 on random_map_0 (20 random agents + its 122 static-map agents).
The card's name, power limit and maximum SM clock are read in the same run.  Needs a CUDA device (no CPU fallback)."""
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
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:
        return "nvidia-smi unavailable (%s)" % e


def params(n142=False):
    from gym_drone2d_activeperception_b200.params import Params
    if n142:
        return Params(debug=False, planner="NoMove", gaze_method="NoControl", static_map="maps/random_map_0.npy",
                      agent_number=20, agent_radius=10, agent_max_speed=20)
    return Params(debug=False, planner="NoMove", gaze_method="NoControl", agent_number=10, agent_radius=15,
                  agent_max_speed=20)


def time_calls(torch, fn, min_ms):
    """Mean ms per call of fn() over back-to-back calls lasting >= min_ms (CUDA events), after a warm-up."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    n = 1
    while True:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        b.synchronize()
        ms = a.elapsed_time(b)
        if ms >= min_ms:
            return ms / n
        n = max(n * 2, int(n * 1.2 * min_ms / max(ms, 1e-3)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for difficulty_bench.json")
    ap.add_argument("--seeds", type=int, default=4096)
    ap.add_argument("--min-ms", type=float, default=100.0)
    args = ap.parse_args()
    import torch
    from gym_drone2d_activeperception_b200 import metrics
    from gym_drone2d_activeperception_b200.vec_env import Drone2DVecEnv
    if not torch.cuda.is_available():
        raise SystemExit("difficulty_bench needs a CUDA device")
    info = gpu_info()
    print(info)
    rows = []

    # ---- 1. seeds per second, the two paths alternated
    p = params()
    seeds = np.arange(args.seeds)
    metrics.difficulty(p, seeds[:64])                     # one-time set-up of both paths outside the timing
    metrics.survivability(p, seeds[:4])
    times = {"difficulty": [], "step kernels": []}
    for _ in range(2):
        t0 = time.perf_counter()
        new = metrics.difficulty(p, seeds)
        times["difficulty"].append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        cs = metrics.global_survivability(p, seeds)
        st, mean = metrics.survivability(p, seeds)
        dens = metrics.obstacle_density(p, seeds)
        torch.cuda.synchronize()
        times["step kernels"].append(time.perf_counter() - t0)
    same = {"survivability": bool(np.array_equal(new["survivability"], st)),
            "mean_survivability": bool(np.array_equal(new["mean_survivability"], mean)),
            "global_survival_time": bool(np.array_equal(new["global_survival_time"], metrics.mean_survival_time(cs))),
            "density": bool(np.array_equal(new["density"], dens))}
    for k, v in times.items():
        rows.append({"case": "%s, %d seeds, N = 10, T = 24 / 12, 64 positions" % (k, len(seeds)),
                     "seconds": [round(x, 3) for x in v], "seeds_per_s": round(len(seeds) / min(v), 1)})
        print(json.dumps(rows[-1]))
    rows.append({"case": "outputs equal", **same})
    print(json.dumps(rows[-1]))

    # ---- 2. kernel time, 65 536 worlds
    B = 65536
    grid = (20, 20, 60, 8, 8)
    n_slots, table = metrics.global_slots(24, 0.1, 240)
    for n142 in (False, True):
        env = Drone2DVecEnv(params(n142), B, device="cuda:0", auto_reset=False, trackers=False, world_gen="device")
        fh = torch.empty((B, 8, 8), dtype=torch.int16, device="cuda")
        sh = torch.empty((B, 8, 8), dtype=torch.uint8, device="cuda")
        cs = torch.empty((B, 8, 8, n_slots), dtype=torch.uint8, device="cuda")
        for with_cs in (False, True):
            out = (fh, sh, cs) if with_cs else (fh, sh)
            ms = time_calls(torch, lambda: env.difficulty(240, grid, slots=table, n_slots=n_slots, collision_state=with_cs,
                                                          out=out), args.min_ms)
            nbytes = sum(t.numel() * t.element_size() for t in out)
            rows.append({"case": "kernel, %d worlds, N = %d, 240 steps, 64 positions%s"
                                 % (B, env.num_agents, ", collision_state" if with_cs else ""),
                         "ms_per_call": round(ms, 3), "worlds_per_s": round(B / (ms * 1e-3)),
                         "agent_steps_per_s": round(B * env.num_agents * 240 / (ms * 1e-3)), "bytes_written": nbytes})
            print(json.dumps(rows[-1]))
        env.close()
    res = {"gpu": info, "rows": rows}
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "difficulty_bench.json"), "w") as f:
            json.dump(res, f, indent=1)
    if not all(same.values()):
        raise SystemExit("outputs differ: %s" % same)


if __name__ == "__main__":
    main()
