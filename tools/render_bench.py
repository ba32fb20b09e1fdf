"""Time d2d_render (Drone2DVecEnv.render) on the GPU.

    python tools/render_bench.py [--out DIR] [--min-ms 100]

Cases: all 4096 envs of config 2 at 1, 2 and 4 pixels per cell; 65 536 config-4 envs at 1; 16 envs at 10; and the time a
16-env render at 4 adds, per step, to a captured 64-step config-4 (Primitive + Oxford) graph.  Each timing is CUDA events
around back-to-back calls lasting at least --min-ms after a warm-up.  Reported per case: us per call, output bytes per call
over that time, and the share of the data sheet's 7.7 TB/s HBM bandwidth that rate is.  The card's name, power limit and
maximum SM clock are read in the same run.  Needs a CUDA device (no CPU fallback)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

HBM_BYTES_PER_S = 7.7e12


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:
        return "nvidia-smi unavailable (%s)" % e


def params(cfg):
    from gym_drone2d_activeperception_b200.params import Params
    if cfg == 2:
        return Params(debug=False, planner="NoMove", static_map="maps/empty_map.npy", agent_number=10, agent_radius=15,
                      agent_max_speed=20, gaze_method="LookAhead")
    return Params(debug=False, planner="Primitive", static_map="maps/obstacle_map.npy", agent_number=10, agent_radius=10,
                  agent_max_speed=20, gaze_method="Oxford")


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


def row(name, ms, nbytes):
    us = ms * 1e3
    rate = nbytes / (ms * 1e-3)
    return {"case": name, "us_per_call": round(us, 2), "bytes_per_call": int(nbytes), "GB_per_s": round(rate / 1e9, 1),
            "hbm_share": round(rate / HBM_BYTES_PER_S, 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for render_bench.json")
    ap.add_argument("--min-ms", type=float, default=100.0)
    args = ap.parse_args()
    import torch
    from gym_drone2d_activeperception_b200.vec_env import Drone2DVecEnv
    if not torch.cuda.is_available():
        raise SystemExit("render_bench needs a CUDA device")
    info = gpu_info()
    print(info)
    print("torch device:", torch.cuda.get_device_name(0))
    rows = []
    env2 = Drone2DVecEnv(params(2), 4096, world_gen="device")
    for _ in range(20):
        env2.step(env2.plan_gaze("LookAhead"))
    for ppc in (1, 2, 4):
        out = torch.empty((4096, 50 * ppc, 50 * ppc, 3), dtype=torch.uint8, device="cuda")
        ms = time_calls(torch, lambda: env2.render(None, ppc, out=out), args.min_ms)
        rows.append(row("config 2, 4096 envs, ppc %d" % ppc, ms, out.numel()))
        print(json.dumps(rows[-1]))
        if ppc == 4:        # where the time goes: the same call with fewer layers (0: the store path alone)
            for name, layers in (("cells only", 3), ("all but the view wedge", 127 & ~4), ("no layers (white)", 0)):
                ms = time_calls(torch, lambda: env2.render(None, ppc, layers=layers, out=out), args.min_ms)
                rows.append(row("config 2, 4096 envs, ppc %d, %s" % (ppc, name), ms, out.numel()))
                print(json.dumps(rows[-1]))
        del out
    env2.close()

    env4 = Drone2DVecEnv(params(4), 65536, world_gen="device")
    a = env4.plan_oxford()
    for _ in range(20):
        env4.step_plan_oxford(a, a)
    out = torch.empty((65536, 50, 50, 3), dtype=torch.uint8, device="cuda")
    ms = time_calls(torch, lambda: env4.render(None, 1, out=out), args.min_ms)
    rows.append(row("config 4, 65536 envs, ppc 1", ms, out.numel()))
    print(json.dumps(rows[-1]))
    del out
    pick = list(np.random.RandomState(0).choice(65536, 16, replace=False))
    out = torch.empty((16, 500, 500, 3), dtype=torch.uint8, device="cuda")
    ms = time_calls(torch, lambda: env4.render(pick, 10, out=out), args.min_ms)
    rows.append(row("config 4, 16 listed envs, ppc 10", ms, out.numel()))
    print(json.dumps(rows[-1]))
    del out

    # added time per step: a captured 64-step graph with and without a 16-env ppc-4 render per step, replays alternated
    K = 64
    frames = torch.empty((K, 16, 200, 200, 3), dtype=torch.uint8, device="cuda")
    graphs = {}
    for with_render in (False, True):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for t in range(K):
                env4.step_plan_oxford(a, a)
                if with_render:
                    env4.render(pick, 4, out=frames[t])
        graphs[with_render] = g
    for g in graphs.values():
        g.replay()
    torch.cuda.synchronize()
    per = {False: [], True: []}
    for _ in range(3):
        for w, g in graphs.items():
            per[w].append(time_calls(torch, g.replay, args.min_ms) / K)
    base, rend = float(np.median(per[False])), float(np.median(per[True]))
    added = {"case": "16 envs ppc 4 inside a captured 64-step config-4 graph (65536 envs, Primitive + Oxford)",
             "step_us": round(base * 1e3, 1), "step_with_render_us": round(rend * 1e3, 1),
             "added_us_per_step": round((rend - base) * 1e3, 1), "bytes_per_render": 16 * 200 * 200 * 3}
    rows.append(added)
    print(json.dumps(added))
    env4.close()
    res = {"gpu": info, "rows": rows}
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "render_bench.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
