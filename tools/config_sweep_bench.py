"""Config sweeps: a product of difficulty axes run as one handle per config against one handle per batch group.

    python tools/config_sweep_bench.py [--seeds 12] [--reps 1] [--out DIR]

540 configs on the empty map: 5 agent speeds x 4 pillar counts x 3 initial positions x 3 agent radii x 3 agent numbers,
which experiment.batch_groups splits into 9 groups (radius x number).  Two workloads, each timed as the per-config loop
and as the grouped call, alternated in this process after an untimed warm-up of both on a few configs, and checked equal:
1. experiment rows, Primitive planner + LookAhead gaze, `--seeds` seeds per config: `[run_seed_sweep(c, seeds, S)]`
   against `run_config_sweep(configs, seeds, 60 * S)` (every pair of a group in one batch);
2. metrics.difficulty over the same configs and seeds: one call per config against one call with the list.
The GPU name and power limit are read in the same run.  Prints one JSON line per workload and a summary line; writes the
summary to DIR/config_sweep_bench.json with --out.  Needs a CUDA device (no CPU fallback)."""
import argparse
import itertools
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                      # the device name from torch below still says what ran
        return "nvidia-smi unavailable (%s)" % e


def configs():
    from gym_drone2d_activeperception_b200.params import Params
    out = []
    for speed, pillars, init, radius, number in itertools.product((10, 20, 30, 40, 50), (0, 2, 4, 6),
                                                                  ([50, 50], [100, 50], [50, 100]), (5, 10, 15),
                                                                  (5, 10, 15)):
        out.append(Params(debug=False, planner="Primitive", gaze_method="LookAhead", static_map="maps/empty_map.npy",
                          agent_max_speed=speed, pillar_number=pillars, init_pos=init, agent_radius=radius,
                          agent_number=number))
    return out


def same_rows(a, b):
    for x, y in zip(a, b):
        for k in y:
            if not (x[k] == y[k] or (isinstance(y[k], float) and math.isnan(y[k]) and math.isnan(x[k]))):
                return False
    return len(a) == len(b)


def timed(fn):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seeds", type=int, default=12)
    ap.add_argument("--reps", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("config_sweep_bench: needs a CUDA device")
    from gym_drone2d_activeperception_b200 import metrics
    from gym_drone2d_activeperception_b200.experiment import batch_groups, run_config_sweep, run_seed_sweep
    seeds = 1 + np.arange(a.seeds, dtype=np.int64)
    S = len(seeds)
    groups = batch_groups(configs())
    B = max(len(g) for g in groups) * S
    res = {"gpu": gpu_info(), "device": torch.cuda.get_device_name(0), "configs": len(configs()), "groups": len(groups),
           "seeds_per_config": S, "workloads": []}
    work = {
        "rows": (lambda cs: [run_seed_sweep(c, seeds, S) for c in cs], lambda cs: run_config_sweep(cs, seeds, B),
                 lambda x, y: all(same_rows(p, q) for p, q in zip(x, y)) and len(x) == len(y)),
        "difficulty": (lambda cs: [metrics.difficulty(c, seeds) for c in cs], lambda cs: metrics.difficulty(cs, seeds),
                       lambda x, y: all(np.array_equal(np.stack([r[k] for r in x]), y[k]) for k in y)),
    }
    for name, (per_config, grouped, equal) in work.items():
        warm = configs()[:2] + configs()[-2:]
        per_config(warm)                          # untimed: module loads, first launches, graph capture paths
        grouped(warm)
        out = {"workload": name, "per_config_s": [], "grouped_s": []}
        for _ in range(a.reps):
            t, x = timed(lambda: per_config(configs()))
            out["per_config_s"].append(t)
            t, y = timed(lambda: grouped(configs()))
            out["grouped_s"].append(t)
            assert equal(x, y), name
        out["equal"] = True
        out["speedup"] = float(np.median(out["per_config_s"]) / np.median(out["grouped_s"]))
        res["workloads"].append(out)
        print(json.dumps(out), flush=True)
    print(json.dumps(res))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "config_sweep_bench.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
