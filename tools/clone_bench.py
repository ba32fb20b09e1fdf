"""Bandwidth of the per-env state copies (d2d_clone_envs, d2d_save_state, d2d_load_state) on BASELINE configs 2 and 4.

    python tools/clone_bench.py [--calls 30] [--warmup 5]

For each config: a 36 864-env handle (worlds tiled from 128 seeds, 10 steps taken so the state is populated), 4096 source
envs each cloned 8x into envs 4096..36863 (32 768 copies, one launch), then the same 32 768 envs saved into a packed
buffer and loaded back.  Each call is timed alone between two CUDA events; the median over --calls calls after --warmup
calls is reported.  Algorithmic bytes = 2 x bytes_per_env x copies (every state byte read once and written once).  Prints
one JSON line.  Writes nothing."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12      # HGX B200 data sheet, one GPU (a card limited below 1000 W may not reach it)
L2_BYTES = 126 << 20
CONFIGS = {
    2: dict(planner="NoMove", static_map="maps/empty_map.npy", agent_number=10, agent_radius=15, agent_max_speed=20, map_id=1),
    4: dict(planner="Primitive", gaze_method="Oxford", static_map="maps/obstacle_map.npy", agent_number=10, agent_radius=10,
            agent_max_speed=20, map_id=1),
}
B, SOURCES, FANOUT = 36864, 4096, 8


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return {"name": name, "power_limit_and_max_sm_clock": out}


def timed(fn, calls, warmup):
    import torch
    for _ in range(warmup):
        fn()
    ms = []
    for _ in range(calls):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return float(np.median(ms)), ms


def run_config(cid, calls, warmup):
    import torch
    from gym_drone2d_activeperception_b200 import Params, generate_worlds
    from gym_drone2d_activeperception_b200.vec_env import Drone2DVecEnv
    p = Params(debug=False, **CONFIGS[cid])
    uniq = generate_worlds(p, 1 + np.arange(128))
    worlds = {k: np.ascontiguousarray(np.concatenate([v] * (B // 128))) for k, v in uniq.items()}
    oxford = cid == 4
    env = Drone2DVecEnv(p, B, worlds=worlds, device="cuda:0", auto_reset=True, oxford=oxford)
    table = torch.as_tensor(np.arange(-80, 80, 80 / 3) / 80, device="cuda:0")
    a = env.plan_oxford() if oxford else None
    g = torch.Generator().manual_seed(0)
    for t in range(10):
        if oxford:
            a = env.step_plan_oxford(a, out=a)
        else:
            env.step(table[torch.randint(0, 6, (B,), generator=g).to("cuda:0")])
    torch.cuda.synchronize()
    nbytes, fp = env.state_layout()
    src = np.ascontiguousarray(np.tile(np.arange(SOURCES), FANOUT), dtype=np.int32)
    dst = np.ascontiguousarray(np.arange(SOURCES, B), dtype=np.int32)
    count = len(dst)
    algo = 2 * nbytes * count
    n0 = env.launch_count()
    env.clone_envs(src, dst)
    assert env.launch_count() == n0 + 1
    for n in ("belief", "env_records", "local_map", "tracker_sigma"):        # the copies are exact
        t = env.buffer(n)
        assert torch.equal(t[torch.as_tensor(dst, device="cuda:0").long()], t[torch.as_tensor(src, device="cuda:0").long()]), n
    clone_ms, _ = timed(lambda: env.clone_envs(src, dst), calls, warmup)
    saved = env.save_state(dst)
    state = saved["state"]
    lib, h = env._lib, env._h
    import ctypes as C
    dptr = dst.ctypes.data_as(C.c_void_p)

    def save():
        rc = lib.d2d_save_state(h, dptr, count, C.c_void_p(state.data_ptr()), env._stream())
        assert rc == 0

    def load():
        rc = lib.d2d_load_state(h, dptr, count, C.c_void_p(state.data_ptr()), C.c_uint64(fp), env._stream())
        assert rc == 0
    save_ms, _ = timed(save, calls, warmup)
    load_ms, _ = timed(load, calls, warmup)
    env.close()

    def rate(ms):
        gbs = algo / (ms * 1e-3) / 1e9
        return {"median_ms": round(ms, 4), "GB_per_s": round(gbs, 1), "of_hbm_bandwidth": round(gbs * 1e9 / HBM_BYTES_PER_S, 3)}
    return {
        "config": cid, "agents_per_env": env.num_agents, "envs": B, "copies": count,
        "bytes_per_env": nbytes, "algorithmic_bytes": algo,
        "working_set": "%.0f MB of state read and written per call, above the %d MB L2; the %d source rows (%.0f MB) are "
                       "each read %dx by the clone and may be served from L2 after the first read"
                       % (algo / 1e6, L2_BYTES >> 20, SOURCES, SOURCES * nbytes / 1e6, FANOUT),
        "clone": rate(clone_ms), "save": rate(save_ms), "load": rate(load_ms),
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--calls", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("clone_bench.py measures the GPU kernel: no CUDA device found")
    out = {"bench": "per-env state copies", "card": card(), "hbm_bytes_per_s_datasheet": HBM_BYTES_PER_S,
           "timing": "CUDA events around each call, median of %d after %d warm-up calls" % (args.calls, args.warmup),
           "results": [run_config(c, args.calls, args.warmup) for c in (2, 4)]}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
