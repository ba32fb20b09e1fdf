"""Time of world generation on the GPU (d2d_generate_worlds) against the host's world.generate_worlds.

    python tools/worldgen_bench.py [--reps 5] [--host-sample 256] [--out DIR]

For 65 536 config-3 worlds (random_map_0, N = 142) and 131 072 config-5 worlds (shaped_obstacle_map, N = 96): the device
time of one generation call (CUDA events around an eager reseed of every env: the generation kernel plus the reset
kernel), the median over --reps calls after one warm-up, and the host time per world on a sample of seeds.  Prints one
JSON line; writes it to DIR/worldgen_bench.json with --out.  The host sample is checked against the device worlds."""
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
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              stdout=subprocess.PIPE, text=True, timeout=30).stdout.strip()
    except Exception:
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--host-sample", type=int, default=256)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from gym_drone2d_activeperception_b200 import Params
    from gym_drone2d_activeperception_b200.vec_env import Drone2DVecEnv
    from gym_drone2d_activeperception_b200.world import generate_worlds
    cases = [("config3_random_map_0", 65536, dict(static_map="maps/random_map_0.npy")),
             ("config5_shaped_obstacle_map", 131072, dict(static_map="maps/shaped_obstacle_map.npy"))]
    res = {"gpu": gpu_info(), "cases": []}
    for name, B, kw in cases:
        p = Params(debug=False, planner="NoMove", **kw)
        env = Drone2DVecEnv(p, B, seeds=np.arange(B), world_gen="device")
        envs = np.arange(B)
        times = []
        for r in range(a.reps + 1):
            seeds = (r + 1) * B + envs
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            env.reseed(envs, seeds)
            ev1.record()
            torch.cuda.synchronize()
            env.check_worlds()
            if r:
                times.append(ev0.elapsed_time(ev1))
        # host: the same seeds, on a sample
        sample = seeds[:a.host_sample]
        t = time.perf_counter()
        host = generate_worlds(p, sample)
        host_ms = (time.perf_counter() - t) * 1e3 / len(sample)
        dev_pos = env.buffer("agent_pos0")[:len(sample)].cpu().numpy()
        same = bool(np.array_equal(dev_pos, host["agent_pos"]))
        ms = float(np.median(times))
        res["cases"].append(dict(name=name, envs=B, num_agents=env.num_agents, device_ms_median=ms,
                                 device_ms_all=[float(x) for x in times], device_us_per_world=ms * 1e3 / B,
                                 host_ms_per_world=host_ms, host_s_for_all=host_ms * B / 1e3,
                                 speedup_vs_one_host_core=host_ms * B / ms, sample_positions_equal=same))
        env.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "worldgen_bench.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
