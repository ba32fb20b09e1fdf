#!/usr/bin/env python
"""bench.py -- env-steps/s (and rays/s) of the batched drone2d hot path on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 2|3|4|5] [--envs B]

A "step" is one pass of Drone2DEnv2.step over one batch of synthetic (seeded) environments.  The headline workload is
BASELINE.json configs[1]: empty_map.npy, 4096 envs per GPU, 10 agents, perception + dynamics (NoMove planner, Kalman
trackers on as in the reference).  For N > 1 launch with torchrun (one rank per GPU, weak scaling: every rank steps its own
batch; the only collective of the path is one NCCL all-reduce of the episode statistics).

Prints ONE JSON line (rank 0).
  value      whole-job env-steps/s with inputs resident in HBM.  The timed region is exactly K = --steps steps of every env:
             the K steps of all replicas are captured once as a CUDA graph (NoMove + scripted gaze: one d2d_rollout call
             per replica; otherwise K step launches per replica) and the graph is replayed once between a CUDA-event pair on
             the launch stream, barrier + synchronize around it.  The job's figure is the MAX over ranks; every rank's
             figure is in `per_rank`.  A short K gives a short, noisier region.  The L2 is kept cold by data size: R
             independent replicas of the batch are stepped in turn so that >= 256 MiB of state is touched between two visits
             of a replica.  The e2e legs and `per_step_events` also run K steps each.
  e2e        the same metric through d2d_step_host with pinned HOST buffers, host<->device traffic inside the timed region:
             headline = zero-copy mirror transport (d2d_bind_host_mirror), `e2e.full_copy` = plain copies of the whole
             observation every step.
  roofline   algorithmic bytes (SURVEY.md 8d: 2406 + 104*N per env-step) / measured step time vs the measured HBM copy peak.
  workloads  the other BASELINE configs at their own batch sizes in the same run (config 3: Primitive planner, config 4:
             Primitive + Oxford, config 5: 96 agents, and one point of the config-5 ray / FOV sweep), each with value, e2e,
             roofline and per-rank figures.
  shard_invariant (N > 1)  every rank also steps a 64-env slice of its neighbour's shard; the state hashes agree.
  cpu_baseline   the oracle port of the reference path (oracle/drone2d_oracle.c) on the host cores, bounded sample.

--dump-outputs DIR writes what the headline path returned to its caller at the last of its K timed steps, for every env
of every replica (observation, done, reward, the `info` arrays; the fused Oxford call also the next actions), as
DIR/<name>.npy, float32 or float64, under 64 MiB: above that a fixed seeded sample of envs, whose indices are in
DIR/env_index.npy.  Before that step every env has run exactly W warm-up, the burn-in and the K timed steps from seeded
worlds and actions, so with the same arguments two builds can be compared output for output.  With several ranks the
files hold rank 0's shard.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

CONFIGS = {
    # BASELINE.json configs[1..4] (SURVEY.md 8d parameters)
    2: dict(name="configs[1]: empty_map.npy, 4096 envs/GPU, 10 agents, perception+dynamics (NoMove)", envs=4096,
            params=dict(planner="NoMove", static_map="maps/empty_map.npy", agent_number=10, agent_radius=15,
                        agent_max_speed=20, map_id=1)),
    3: dict(name="configs[2]: random_map_0.npy, 65536 envs/GPU, 20 agents radius 15, Primitive planner checks on device",
            envs=65536,
            params=dict(planner="Primitive", static_map="maps/random_map_0.npy", agent_number=20, agent_radius=15,
                        agent_max_speed=40, map_id=1)),
    4: dict(name="configs[3]: obstacle_map.npy, 65536 envs/GPU, 10 agents speed 20, Primitive planner + Oxford gaze scoring",
            envs=65536, gaze="Oxford",
            params=dict(planner="Primitive", static_map="maps/obstacle_map.npy", agent_number=10, agent_radius=10,
                        agent_max_speed=20, map_id=1)),
    5: dict(name="configs[4]: shaped_obstacle_map.npy, 131072 envs/GPU, 50 agents", envs=131072,
            params=dict(planner="NoMove", static_map="maps/shaped_obstacle_map.npy", agent_number=50, agent_radius=10,
                        agent_max_speed=40, map_id=1)),
}
METRIC = "env-steps/sec"
D2D_STATE_BYTES = 2560 + 400 + 128            # read per env and step: belief grid, ground-truth rows, env record
L2_NOTE = "inputs larger than L2: replicas of the batch stepped round robin, >= 256 MiB of state touched between two " \
          "visits of a replica (L2 = 126 MB); batches above that size need one replica"


# ------------------------------------------------------------------------------------------ workload description
def make_cfg(config_id, planner=None, gaze=None, view_range=0, strip_width=10, motion_profile=None, envs=0):
    base = CONFIGS[config_id]
    cfg = dict(base, params=dict(base["params"]), config_id=config_id, strip_width=strip_width)
    cfg["gaze"] = gaze or base.get("gaze", "scripted")
    if planner and planner != base["params"]["planner"]:
        cfg["params"]["planner"] = planner
        cfg["name"] += " [planner=%s]" % planner
    if motion_profile and motion_profile != "CVM":
        cfg["params"]["motion_profile"] = motion_profile
        cfg["name"] += " [motion_profile=%s]" % motion_profile
    if view_range:
        cfg["params"]["drone_view_range"] = view_range
        cfg["name"] += " [view_range=%d]" % view_range
    if strip_width != 10:
        cfg["name"] += " [strip_width=%d]" % strip_width
    if cfg["gaze"] == "Oxford":
        cfg["params"]["gaze_method"] = "Oxford"
        if base.get("gaze") != "Oxford":
            cfg["name"] += " [gaze=Oxford on device]"
    if envs:
        cfg["envs"] = envs
    return cfg


def n_rays_of(cfg):
    return -(-500 // cfg["strip_width"])            # ceil(map_size[0] / strip_width), utils.py:587


def n_agents_of(cfg):
    from gym_drone2d_activeperception_b200 import Params, count_agents, load_static_map
    p = Params(debug=False, **cfg["params"])
    return count_agents(p, load_static_map(p.static_map))


def public_config(cfg, n_gpus):
    """The `config` object of the JSON line: identical for both arms (--impl ours / reference) of the same workload."""
    return {"workload": cfg["name"], "envs_per_gpu": cfg["envs"], "agents_per_env": n_agents_of(cfg),
            "rays_per_env_step": n_rays_of(cfg), "planner": cfg["params"]["planner"], "gaze": cfg["gaze"],
            "trackers": True, "auto_reset": True, "l2": L2_NOTE, "parallelism": "env-sharded x%d" % n_gpus}


DUMP_BYTES = 60 << 20                           # array data; with the .npy headers the files stay under 64 MiB


def caller_outputs(envs, next_actions=None):
    """What a caller of the step receives from every replica in `envs` (observation, reward, done, info; the fused Oxford
    call also the next actions, one tensor per replica) as host arrays: float64, int32 and int64 buffers as float64, the
    8-bit and float32 ones as float32 (both exact).  Rows are envs, replica r's env i at row r * B + i; when the rows are
    above DUMP_BYTES a fixed seeded sample of them is kept, named by `env_index`."""
    import torch

    def named(e, nxt):
        obs, info = e._obs(), e.info
        out = [("local_map", obs["local_map"]), ("yaw_angle", obs["yaw_angle"]), ("reward", e.reward), ("done", e.buffer("done"))]
        out += sorted(info.items())
        if nxt is not None:
            out.append(("next_actions", nxt))
        return out
    wide = (torch.float64, torch.int32, torch.int64)
    B = envs[0].num_envs
    per_env = 8 + sum((8 if t.dtype in wide else 4) * (t.numel() // B) for _, t in named(envs[0], None if next_actions is None
                                                                                          else next_actions[0]))
    total = B * len(envs)
    n = min(total, DUMP_BYTES // per_env)
    rows = np.arange(total) if n == total else np.sort(np.random.RandomState(0).choice(total, n, replace=False))
    parts = {}
    for r, e in enumerate(envs):
        local = rows[(rows >= r * B) & (rows < (r + 1) * B)] - r * B
        idx = torch.as_tensor(local, device=e.device)
        for name, t in named(e, None if next_actions is None else next_actions[r]):
            t = t.index_select(0, idx)
            parts.setdefault(name, []).append(t.to(torch.float64 if t.dtype in wide else torch.float32).cpu().numpy())
    out = {"env_index": rows.astype(np.float64)}
    out.update({name: np.concatenate(p) for name, p in parts.items()})
    return out


def write_dump(directory, arrays):
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def _gen_chunk(args):
    from gym_drone2d_activeperception_b200 import Params, generate_worlds
    pk, seeds = args
    return generate_worlds(Params(debug=False, **pk), seeds)


def make_worlds(pk, seeds, unique=None, max_procs=32):
    """Host-side world generation (seeded, the reference's own procedure).  `unique` caps the number of distinct
    worlds (tiled to the batch) to bound set-up time for the very large configs; the default keeps every env unique."""
    import multiprocessing as mp
    seeds = np.asarray(seeds)
    B = len(seeds)
    gen = seeds if unique is None or unique >= B else seeds[:unique]
    nproc = max(1, min(len(os.sched_getaffinity(0)), max_procs, len(gen) // 64))
    chunks = np.array_split(gen, nproc)
    if nproc > 1:
        with mp.get_context("fork").Pool(nproc) as pool:
            parts = pool.map(_gen_chunk, [(pk, c) for c in chunks])
    else:
        parts = [_gen_chunk((pk, gen))]
    w = {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}
    if len(gen) < B:
        reps = (B + len(gen) - 1) // len(gen)
        w = {k: np.concatenate([v] * reps)[:B] for k, v in w.items()}
    return w


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu_index, self.rows, self.proc, self.mark = gpu_index, [], None, 0

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=2)
        rows = self.rows[self.mark:] if len(self.rows) - self.mark >= 3 else self.rows
        sm = [float(r[1]) for r in rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm),
                "window": "the timed graph replays of the headline workload plus back-to-back steps for 1.5 s right after "
                          "(reasons: whole run)"}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def algorithmic_bytes(n_agents):
    return 2406 + 104 * n_agents          # SURVEY.md 8(d); tracker / Oxford-state traffic deliberately NOT counted


# ------------------------------------------------------------------------------------------ CPU arm (oracle port)
def cpu_port_run(pk, n_envs, steps, threads, seed0=1, oxford=False):
    """Times the oracle port of the reference path on the host: n_envs envs x steps steps over `threads` threads
    (ctypes releases the GIL), with the batched env's auto-reset rule.  Returns (env-steps/s, seconds)."""
    import oracle
    from gym_drone2d_activeperception_b200 import Params
    p = Params(debug=False, **pk)
    worlds = make_worlds(pk, seed0 + np.arange(n_envs))
    op = oracle.make_params(dt=p.dt, map_scale=p.map_scale, map_size=p.map_size, agent_radius=p.agent_radius,
                            drone_max_acceleration=p.drone_max_acceleration, drone_radius=p.drone_radius,
                            drone_max_yaw_speed=p.drone_max_yaw_speed, drone_view_depth=p.drone_view_depth,
                            drone_view_range=p.drone_view_range, max_flight_time=p.max_flight_time, var_cam=p.var_cam,
                            drone_max_speed=p.drone_max_speed, planner=p.planner)
    envs = [oracle.OracleEnv(op, worlds["agent_pos"][i], worlds["agent_pref"][i], worlds["agent_radius"][i],
                             worlds["gt_grid"][i], worlds["tracker_radius"][i], drone=worlds["drone_pose"][i],
                             targets=p.target_list) for i in range(n_envs)]
    if p.motion_profile == "RVO":
        for i, e in enumerate(envs):
            e.set_rvo(worlds["agent_vel"][i], worlds["obstacles"][i])
    ob = oracle.OracleBatch(envs, threads=threads)
    table = np.arange(-80, 80, 80 / 3) / 80
    rng = np.random.RandomState(0)
    policy = "Oxford" if oxford else "scripted"
    ob.run(2, None if oxford else table[rng.randint(0, 6, (2, n_envs))], policy=policy)        # warm-up
    acts = None if oxford else table[rng.randint(0, 6, (steps, n_envs))]
    t0 = time.perf_counter()
    ob.run(steps, acts, policy=policy)
    dt = time.perf_counter() - t0
    ob.close()
    return n_envs * steps / dt, dt


def run_reference(args, cfg):
    """--impl reference: the reference's CPU implementation of the path (oracle port; the Python reference cannot
    travel to the GPU box), all host threads, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    oracle.build()
    cores = len(os.sched_getaffinity(0))
    n_envs = min(4096, cfg["envs"])
    steps_per = 200
    vals = []
    t_all = time.perf_counter()
    pk = {k: v for k, v in cfg["params"].items() if k != "gaze_method"}
    for it in range(args.warmup + args.steps):
        v, dt = cpu_port_run(pk, n_envs, steps_per, cores, seed0=1 + it, oxford=cfg["gaze"] == "Oxford")
        if it >= args.warmup:
            vals.append((n_envs * steps_per, dt))
        if time.perf_counter() - t_all > 150 and len(vals) >= 1:
            break
    tot_steps = sum(v[0] for v in vals)
    tot_t = sum(v[1] for v in vals)
    value = tot_steps / tot_t
    n_rays = n_rays_of(cfg)
    sample = "%d envs x %d steps per bench step (auto-reset on), %d bench steps, %d threads" % (n_envs, steps_per, len(vals), cores)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": args.gpus,
            "steps": len(vals), "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / max(1, len(vals)),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": public_config(cfg, args.gpus),
            "rays_per_sec": value * n_rays,
            "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


_JSON_OUT = None


def _claim_stdout():
    """stdout carries exactly ONE line, the JSON result: everything else that libraries print there (NCCL's version banner
    under torchrun, for one) is sent to stderr by re-pointing fd 1; the JSON line goes to the saved descriptor."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


# ------------------------------------------------------------------------------------------ GPU arm: one workload
class Ctx(object):
    """Per-process context: rank / device / collectives (through the package's distributed helpers)."""

    def __init__(self, args):
        import torch
        from gym_drone2d_activeperception_b200 import distributed as D
        self.rank, self.local_rank, self.world = D.rank_world()
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        D.init_process_group("nccl", device=self.dev)
        self.D = D
        self.args = args

    def barrier(self):
        import torch
        import torch.distributed as dist
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def gather_rows(self, row):
        """all-gather of one small float64 row per rank -> [world, len(row)] numpy"""
        import torch
        import torch.distributed as dist
        t = torch.tensor([row], dtype=torch.float64, device=self.dev)
        if self.world == 1:
            return t.cpu().numpy()
        out = [torch.zeros_like(t) for _ in range(self.world)]
        dist.all_gather(out, t)
        return torch.cat(out).cpu().numpy()


def measure(ctx, cfg, worlds, t_world, unique, headline):
    """Times one workload on this rank's GPU and reduces over ranks; returns the result dict (meaningful on every rank)."""
    import torch
    from gym_drone2d_activeperception_b200 import Params
    from gym_drone2d_activeperception_b200.vec_env import Drone2DVecEnv
    args, dev, world, rank = ctx.args, ctx.dev, ctx.world, ctx.rank
    B, pk = cfg["envs"], cfg["params"]
    p = Params(debug=False, **pk)
    use_ox = cfg["gaze"] == "Oxford"
    seeds = ctx.D.shard_seeds(pk["map_id"], B, rank)

    def make_env():
        return Drone2DVecEnv(p, B, seeds=seeds, worlds=worlds, device=dev, auto_reset=True, trackers=True, oxford=use_ox,
                             envs_per_block=args.envs_per_block, strip_width=cfg["strip_width"])
    env = make_env()
    n_rays = int(env.cfg.n_rays)
    N = env.num_agents
    K, W = args.steps, args.warmup
    # Cold-L2 rule: consecutive timed steps must not find their inputs in the 126 MB L2.  The timed region steps R
    # independent replicas of the batch round robin (same config, same worlds, own state and own action stream), R chosen
    # so that the state touched between two visits of a replica is >= 256 MiB; big batches (R = 1) already exceed L2.
    touched = B * (D2D_STATE_BYTES + 56 * N)       # + agents (40 B) and tracker flags / hit mask per agent; = ncu's DRAM read
    R = 1 if args.no_flush else max(1, min(64, -(-(256 << 20) // touched)))
    envs = [env] + [make_env() for _ in range(R - 1)]
    ox_out = torch.empty(B, dtype=torch.float64, device=dev)

    # Oxford on the device: one step = Oxford.plan + env.step, through d2d_step_plan_oxford (the step's A* searches beside the
    # gaze scoring of the envs that did not plan); --no-fused-oxford: the two calls d2d_plan_oxford + d2d_step
    fused_ox = use_ox and pk["planner"] == "Primitive" and not args.no_fused_oxford
    ox_next = {}

    def do_step(a, e=None):
        e = env if e is None else e
        if fused_ox:
            if e not in ox_next:
                ox_next[e] = e.plan_oxford(torch.empty(B, dtype=torch.float64, device=dev))
            e.step_plan_oxford(ox_next[e], out=ox_next[e])
        elif use_ox:
            e.step(e.plan_oxford(ox_out))
        else:
            e.step(a)
    table = torch.as_tensor(np.arange(-80, 80, 80 / 3) / 80, device=dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    actions = table[torch.randint(0, 6, (K + W, B), device=dev, generator=gen)].contiguous()
    burn = args.burn_in if headline else min(args.burn_in, 300)

    for e in envs:                                  # eager warm-up: W steps of every replica
        for t in range(W):
            do_step(actions[t], e)
    # burn-in (untimed): episodes last up to 800 steps, so the mix of fresh / explored / tracking envs -- and with it the
    # cost of a step -- only becomes stationary after about a thousand steps (SURVEY 8d: 1000 steps with auto-reset)
    for t in range(burn):
        for e in envs:
            do_step(actions[t % (K + W)], e)
    ctx.barrier()
    side = torch.cuda.Stream(device=dev)
    sampler = None
    if headline:
        sampler = ClockSampler(ctx.local_rank if "CUDA_VISIBLE_DEVICES" not in os.environ else
                               int(os.environ["CUDA_VISIBLE_DEVICES"].split(",")[ctx.local_rank]))
        sampler.start()
        sampler.mark = len(sampler.rows)

    def timed_replay(g):
        """One replay of `g` between a CUDA-event pair, barrier + synchronize around it; returns (ms, wall s)."""
        q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ctx.barrier()
        w0 = time.perf_counter()
        q0.record(); g.replay(); q1.record()
        ctx.barrier()
        return float(q0.elapsed_time(q1)), time.perf_counter() - w0

    # ---- K steps of every env as K launches per replica (one d2d_step per step), replicas interleaved step by step;
    #      captured as one CUDA graph, replayed once: the timed region holds exactly these K steps of every env
    rollout_ok = pk["planner"] == "NoMove" and not use_ox and pk.get("motion_profile", "CVM") != "RVO" and args.envs_per_block <= 0
    graph = torch.cuda.CUDAGraph()
    l0 = sum(e.launch_count() for e in envs)
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            for t in range(K):
                for e in envs:
                    do_step(actions[W + t], e)
    launches = (sum(e.launch_count() for e in envs) - l0) // R     # kernel nodes of the graph per replica
    dump = None
    if rollout_ok:
        ms_graph, wall = None, None               # timed after the headline below (a second K steps of every env)
    else:
        ms_graph, wall = timed_replay(graph)
        if headline and args.dump_outputs and rank == 0:
            dump = caller_outputs(envs, [ox_next.get(e) for e in envs] if fused_ox else None)

    # ---- the same K steps as ONE launch per replica (d2d_rollout): every warp walks its env through the K steps with the
    #      env's working set resident on chip -- the device-resident form of a scripted-gaze run (experiment.py:65-70).
    #      The R calls are captured as one CUDA graph after a W-step warm-up call per replica and replayed once.
    rollout = None
    if rollout_ok:
        for e in envs:
            e.rollout(actions[:W].contiguous())
        act_k = actions[W:W + K].contiguous()
        rgraph = torch.cuda.CUDAGraph()
        r0 = sum(e.launch_count() for e in envs)
        with torch.cuda.stream(side):
            with torch.cuda.graph(rgraph, stream=side):
                for e in envs:
                    e.rollout(act_k)
        r_launches = sum(e.launch_count() for e in envs) - r0
        r_ms, wall = timed_replay(rgraph)
        rollout = {"ms": r_ms / (K * R), "launches": int(r_launches), "region_ms": r_ms,
                   "resident": int(r_launches) == R}     # above two waves of warps d2d_rollout issues K per-step launches
        del rgraph
        if headline and args.dump_outputs and rank == 0:
            dump = caller_outputs(envs)
        ms_graph, _ = timed_replay(graph)
    ms_launch = ms_graph / (K * R)

    per_step = None
    if headline:
        # secondary: the same step timed one launch at a time (CUDA events around every step, 256 MiB L2 flush in between,
        # untimed): includes ~3-4 us of event / launch gap per step; kept for the per-step distribution
        Kp = K
        flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
        pe0 = [torch.cuda.Event(enable_timing=True) for _ in range(Kp)]
        pe1 = [torch.cuda.Event(enable_timing=True) for _ in range(Kp)]
        for t in range(Kp):
            flush.fill_(t & 0xFF)
            pe0[t].record()
            do_step(actions[W + t])
            pe1[t].record()
        ctx.barrier()
        step_ms = np.array([a.elapsed_time(b) for a, b in zip(pe0, pe1)])
        del flush
        per_step = {"what": "same step, one launch at a time: CUDA events around every step, 256 MiB L2 flush (untimed) in "
                            "between; includes the event / launch gap of each step",
                    "steps": int(Kp), "ms_min_med_max": [float(step_ms.min()), float(np.median(step_ms)), float(step_ms.max())],
                    "value": world * B / (float(np.mean(step_ms)) * 1e-3)}

    # ---- end to end through the C ABI with pinned host buffers (wall clock, synchronise per step)
    a_host = actions.cpu().pin_memory()
    lm_host = torch.empty((B, 1, 33, 33), dtype=torch.uint8).pin_memory()
    yaw_host = torch.empty((B,), dtype=torch.float32).pin_memory()
    done_host = torch.empty((B,), dtype=torch.uint8).pin_memory()
    a_rows = [a_host[t] for t in range(K + W)]       # views of the pinned action buffer, one per step
    stage = env.buffer("actions_staging")
    Ke = K

    def e2e_step_host(t):
        if use_ox:      # the policy runs on the device: its actions never leave the GPU, the observation still does
            env.plan_oxford(stage)
            env.step_host(None, lm_host, yaw_host, done_host)
        else:
            env.step_host(a_rows[t % (K + W)], lm_host, yaw_host, done_host)
    stepper = [e2e_step_host]
    warm = [True]
    e2e_bound_s = None

    def e2e_loop():
        step = stepper[0]
        warm[0] = True
        for t in range(3):
            step(t)
        warm[0] = False
        ctx.barrier()
        st0 = env.stats()
        t0 = time.perf_counter()
        for t in range(Ke):
            step(t)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        ctx.barrier()
        return dt, env.stats() - st0

    # (a) plain copies: every step moves the whole observation tensor device -> host
    e2e_copy_s, _ = e2e_loop()
    # (b) the library's zero-copy mirror (d2d_bind_host_mirror): the kernels store the observation bytes that change
    #     straight into the pinned host buffers; the step call copies nothing back
    e2e_mirror_s = None
    if args.e2e_full_copy:
        e2e_s, mirror_bytes = e2e_copy_s, None
    else:
        env.bind_host_mirror(lm_host, yaw_host, done_host)
        e2e_mirror_s, dst = e2e_loop()
        mirror_bytes = float(dst[14]) / Ke
        assert torch.equal(lm_host, env.buffer("local_map").cpu()) and torch.equal(done_host, env.buffer("done").cpu())
        env.bind_host_mirror(None, None, None)
        # (c) the bound form of the same call (d2d_bind_host_io + d2d_step_bound): host buffers given once, the caller
        #     rewrites the pinned action buffer in place (a 8*B-byte host memcpy, inside the timed region), one C call per
        #     step; with the NoMove planner the step kernel signals completion through a pinned flag the host polls.
        #     This is the headline e2e.
        import ctypes
        a_bound = torch.zeros(B, dtype=torch.float64).pin_memory()
        env.bind_host_io(None if use_ox else a_bound, lm_host, yaw_host, done_host)
        dstp, nbytes = a_bound.data_ptr(), B * 8
        srcs = [r.data_ptr() for r in a_rows]

        if fused_ox:
            env.plan_oxford(stage)              # primes the first step; every call below leaves the next step's actions there
            torch.cuda.synchronize()

        def e2e_step_bound(t):
            if fused_ox:
                env.step_bound_plan_oxford()
                return
            if use_ox:
                env.plan_oxford(stage)
            else:
                ctypes.memmove(dstp, srcs[t % (K + W)], nbytes)
            env.step_bound()

        def e2e_step_pipelined(t):
            # the timed loop runs t = 0 .. Ke-1 after a 3-step warm-up: the warm-up's last step and the run's last step do not
            # pre-launch (the loop's barrier / statistics calls follow them)
            ctypes.memmove(dstp, srcs[t % (K + W)], nbytes)
            env.step_pipelined(prelaunch_next=not (t == Ke - 1 or (t == 2 and warm[0])))
        stepper[0] = e2e_step_bound
        e2e_bound_s, _ = e2e_loop()
        if not use_ox and pk["planner"] == "NoMove":
            stepper[0] = e2e_step_pipelined
        e2e_s, dst = e2e_loop()
        mirror_bytes = float(dst[14]) / Ke
        assert torch.equal(lm_host, env.buffer("local_map").cpu()) and torch.equal(done_host, env.buffer("done").cpu())
        env.bind_host_io(None, None, None, None)
    clocks = None
    if headline:
        # clock / throttle sampling needs a loaded window: keep stepping back to back (untimed, same kernel) for ~1.5 s
        t_probe = time.perf_counter()
        while time.perf_counter() - t_probe < 1.5:
            graph.replay()
            torch.cuda.synchronize()
        clocks = sampler.stop()

    # ---- over ranks: the max; every rank's figures are reported
    rows = ctx.gather_rows([ms_launch, 0.0, 0.0, e2e_s * 1e3 / Ke, e2e_copy_s * 1e3 / Ke,
                            (e2e_mirror_s if e2e_mirror_s is not None else e2e_copy_s) * 1e3 / Ke,
                            (e2e_bound_s if e2e_bound_s is not None else e2e_copy_s) * 1e3 / Ke,
                            rollout["ms"] if rollout else ms_launch])
    ms_launch_per_step = float(rows[:, 0].max())     # K single-step launches
    # headline: the K steps through the fastest device-resident entry point that executes exactly these K steps
    ms_step = float(rows[:, 7].max())
    e2e_ms, e2e_copy_ms, e2e_mirror_ms = float(rows[:, 3].max()), float(rows[:, 4].max()), float(rows[:, 5].max())
    e2e_bound_ms = float(rows[:, 6].max())
    # the one collective of the path: all-reduce of the episode statistics
    stats = ctx.D.allreduce_stats(sum(np.asarray(e.stats(), dtype=np.int64) for e in envs), device=dev)
    value = world * B / (ms_step * 1e-3)
    e2e = world * B / (e2e_ms * 1e-3)

    peak, peak_src = measured_peak()
    if rollout and rollout["resident"]:
        kernel_name = "d2d_rollout_warp_kernel (K steps per launch, env state resident on chip)"
    elif rollout:
        kernel_name = "d2d_step_fused_warp_kernel (d2d_rollout above two waves of warps: 1 launch/step)"
    elif pk["planner"] == "NoMove":
        kernel_name = "d2d_step_fused_warp_kernel (1 launch/step)"
    else:
        kernel_name = "d2d_step_prim_warp_kernel + d2d_plan_small_kernel (+ d2d_plan_kernel for its overflow list) + d2d_step_post_list_kernel" + \
                      (" + d2d_oxford_kernel" if use_ox else "") + (" beside the A* kernels (d2d_step_plan_oxford)" if fused_ox else "") + \
                      " (whole step timed)"
    achieved = algorithmic_bytes(N) * B / (ms_step * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", ("traffic_rollout_config%d.json" if (rollout and rollout["resident"]) else
                                            "traffic_config%d.json") % cfg["config_id"])
    if os.path.isfile(tpath) and pk["planner"] == "NoMove" and n_rays == 50 and "view_range" not in cfg["name"]:
        try:
            traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    res = {
        "value": value, "unit": "env-steps/s", "ms_per_step": ms_step, "rays_per_sec": value * n_rays,
        "config": public_config(cfg, world),
        "method": {"timing": (("K = %d steps of every env as ONE d2d_rollout call per replica (%s; R = %d calls captured as one "
                              "CUDA graph); " % (
                                  K, "one resident launch" if rollout["resident"] else "K per-step launches: batch above two waves",
                                  R)) if rollout else
                              ("K = %d steps of every env as K step launches per replica, replicas interleaved step by step, "
                               "captured as one CUDA graph; " % K)) +
                             "the graph replayed once between a CUDA-event pair on the launch stream, barrier + synchronize "
                             "around it; ms per step = region / (K x R); over ranks the max",
                   "timed_steps_per_env": K, "graph_replays": 1,
                   "timed_region_ms_this_rank": rollout["region_ms"] if rollout else ms_launch * K * R, "wall_s_timed_region": wall,
                   "replicas": R, "state_touched_between_visits_mb": round(R * touched / 1e6, 1),
                   "l2": "no rotation (--no-flush): state stays L2-resident" if args.no_flush else L2_NOTE,
                   "burn_in_steps_per_replica": burn, "unique_worlds_per_gpu": int(unique), "world_gen_s": round(t_world, 2),
                   "envs_per_block": int(env.cfg.envs_per_block)},
        "per_rank": [{"rank": r, "ms_per_step": float(rows[r, 7]), "single_step_launch_ms": float(rows[r, 0]),
                      "e2e_ms_per_step": float(rows[r, 3])} for r in range(world)],
        "e2e": {"value": e2e, "unit": "env-steps/s", "h2d_bytes_per_step": 0 if use_ox else B * 8,
                "d2h_bytes_per_step": B * (1089 + 4 + 1) if mirror_bytes is None else int(round(B * 5 + mirror_bytes)),
                "steps": Ke,
                "transport": "cudaMemcpyAsync of the whole observation every step" if mirror_bytes is None else
                             "d2d_bind_host_io: pinned action buffer rewritten by the caller every step (memcpy inside the timed "
                             "region) and read by the kernels in place; kernels store changed observation bytes + yaw + done "
                             "straight into the pinned host buffers (bytes counted on the device, mean per step, this rank); " +
                             ("d2d_step_bound_plan_oxford (Oxford on the device: the actions never leave the GPU; the step's A* searches "
                              "beside the gaze scoring), stream synchronised per step" if fused_ox else
                              "d2d_step_bound, stream synchronised per step" if (use_ox or pk["planner"] != "NoMove") else
                              "d2d_step_pipelined: at <= 4116 envs ONE resident kernel serves the whole run (env state stays on chip; "
                              "a courier block pulls each step's actions out of the pinned buffer once the host has stamped the step; "
                              "everything but the yaw update runs before that gate; completion is a pinned word the host polls); "
                              "larger batches: the next step's kernel is pre-launched behind the current one and waits at the same "
                              "gate.  Every call returns this step's observation before the next actions are written"),
                "bound_sync": {"value": world * B / (e2e_bound_ms * 1e-3),
                               "what": "d2d_step_bound per step (bound buffers, stream synchronised every step, nothing pre-launched)"},
                "mirror_step_host": {"value": world * B / (e2e_mirror_ms * 1e-3),
                                     "what": "d2d_step_host per step with the zero-copy mirror bound (round-1 headline path)"},
                "full_copy": {"value": world * B / (e2e_copy_ms * 1e-3), "d2h_bytes_per_step": B * (1089 + 4 + 1),
                              "what": "d2d_step_host per step, whole observation copied device -> host every step"}},
        "gpu_launches": int(rollout["launches"] // R) if rollout else int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "peak_source": peak_src, "bytes_per_env_step": algorithmic_bytes(N),
                     "kernel": kernel_name, "kernel_ms": ms_step},
        "episode_stats": {n: int(v) for n, v in zip(
            ["env_steps", "episodes", "success", "static_collision", "dynamic_collision", "freezing", "dead_lock",
             "flight_steps", "grid_discovered", "agents_tracked", "tracked_steps", "plans", "plan_failures", "replans"],
            stats.tolist()[:14])},
    }
    if pk["planner"] == "Primitive":
        res["episode_stats"]["plan_overflows"] = int(stats.tolist()[15])     # searches redone by the large A* kernel
    if rollout:
        res["single_step_launches"] = {
            "value": world * B / (ms_launch_per_step * 1e-3), "ms_per_step": ms_launch_per_step, "gpu_launches": int(launches),
            "what": "K more steps of every env as K d2d_step launches per replica (one fused kernel per step, captured as one "
                    "CUDA graph, replayed once): the per-step entry point a device-side policy calls",
            "roofline_frac": algorithmic_bytes(N) * B / (ms_launch_per_step * 1e-3) / 1e9 / peak}
        res["gpu_launches_note"] = "launches per K steps of ONE replica of the batch (the timed region steps all R replicas)"
    if per_step is not None:
        res["per_step_events"] = per_step
    if clocks is not None:
        res["clocks"] = clocks
    if dump is not None:
        res["dump"] = dump
    del graph
    for e in envs:
        e.close()
    torch.cuda.empty_cache()
    return res


def shard_invariance(ctx, cfg, steps=48, n=64):
    """N > 1: a given global env must evolve identically whichever GPU runs it.  Every rank steps the first `n` envs of its
    own shard and the first `n` envs of its right neighbour's shard (worlds regenerated here from the global seeds, actions
    a function of (global env, t)); the state hashes are all-gathered and compared."""
    import torch
    from gym_drone2d_activeperception_b200 import Params, generate_worlds
    from gym_drone2d_activeperception_b200.vec_env import Drone2DVecEnv
    if ctx.world == 1:
        return None
    pk, B = cfg["params"], cfg["envs"]
    p = Params(debug=False, **pk)
    table = np.arange(-80, 80, 80 / 3) / 80

    def run(owner):
        seeds = ctx.D.shard_seeds(pk["map_id"], B, owner)[:n]
        env = Drone2DVecEnv(p, n, seeds=seeds, worlds=generate_worlds(p, seeds), device=ctx.dev, auto_reset=True)
        g = owner * B + np.arange(n)
        for t in range(steps):
            env.step(torch.as_tensor(table[(g * 7 + t * 13) % 6], device=ctx.dev))
        torch.cuda.synchronize()
        hsh = hashlib.sha256()
        for name in ("belief", "local_map", "agent_pos", "agent_pref", "drone_yaw", "done", "steps", "tracker_mu", "hit"):
            hsh.update(env.buffer(name).contiguous().cpu().numpy().tobytes())
        env.close()
        return float(int.from_bytes(hsh.digest()[:6], "little"))         # 48 bits: exact in a float64
    own, nb = run(ctx.rank), run((ctx.rank + 1) % ctx.world)
    rows = ctx.gather_rows([own, nb])
    return bool(all(rows[r, 1] == rows[(r + 1) % ctx.world, 0] for r in range(ctx.world)))


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument("--envs", type=int, default=0, help="envs per GPU (default: the config's)")
    ap.add_argument("--envs-per-block", type=int, default=0)
    ap.add_argument("--unique-worlds", type=int, default=0, help="cap distinct generated worlds (0 = all unique up to 16384)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-workloads", action="store_true", help="headline workload only (skip the `workloads` list)")
    ap.add_argument("--burn-in", type=int, default=1000, help="untimed steps per replica before the timed region")
    ap.add_argument("--no-flush", action="store_true", help="do not rotate replicas (state stays in L2; reported)")
    ap.add_argument("--strip-width", type=int, default=10, help="ray strip width: rays = ceil(500 / strip_width) (config 5 sweep: 10/5/2)")
    ap.add_argument("--view-range", type=int, default=0, help="drone_view_range in degrees (config 5 sweep: 90/180/360)")
    ap.add_argument("--planner", default=None, choices=["NoMove", "Primitive"], help="override the config's planner")
    ap.add_argument("--motion-profile", default=None, choices=["CVM", "RVO"], help="agent motion profile (default CVM)")
    ap.add_argument("--no-fused-oxford", action="store_true", help="Oxford workloads: d2d_plan_oxford + d2d_step instead of d2d_step_plan_oxford")
    ap.add_argument("--e2e-full-copy", action="store_true", help="e2e leg with plain D2H copies instead of the zero-copy mirror")
    ap.add_argument("--gaze", default=None, choices=["scripted", "Oxford"],
                    help="scripted: random actions from the Oxford action set; Oxford: d2d_plan_oxford every step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the headline path's outputs after its last timed step as DIR/<name>.npy (see the module doc)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    if args.warmup < 3:
        args.warmup = 3
    cfg = make_cfg(args.config, planner=args.planner, gaze=args.gaze, view_range=args.view_range,
                   strip_width=args.strip_width, motion_profile=args.motion_profile, envs=args.envs)
    if args.impl == "reference":
        run_reference(args, cfg)
        return

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # the default run (BASELINE config 2 headline, no overrides) also measures the other BASELINE configs
    default_run = args.config == 2 and not (args.planner or args.gaze or args.view_range or args.motion_profile or
                                           args.envs or args.strip_width != 10)
    extra = []
    if default_run and not args.no_workloads:
        extra = [make_cfg(3), make_cfg(4), make_cfg(5), make_cfg(5, view_range=360, strip_width=2)]
    # worlds of every workload are generated before CUDA is touched (fork-based pool)
    procs = max(2, len(os.sched_getaffinity(0)) // max(1, world))
    gen = []
    for c in [cfg] + extra:
        B = c["envs"]
        unique = args.unique_worlds or min(B, 16384 if c is cfg else 8192)
        t0 = time.perf_counter()
        seeds = c["params"]["map_id"] + rank * B + np.arange(B)
        gen.append((c, make_worlds(c["params"], seeds, unique=unique, max_procs=procs), time.perf_counter() - t0, unique))
        log("worlds for", c["name"], "in %.1f s" % gen[-1][2])

    import torch.distributed as dist
    ctx = Ctx(args)
    line = dump = None
    workloads = []
    for i, (c, worlds, t_world, unique) in enumerate(gen):
        t0 = time.perf_counter()
        res = measure(ctx, c, worlds, t_world, unique, headline=(i == 0))
        log("%s: %.1f M env-steps/s, e2e %.1f M (%.1f s)" % (c["name"], res["value"] / 1e6, res["e2e"]["value"] / 1e6,
                                                            time.perf_counter() - t0))
        gen[i] = None                                # release the host arrays of this workload
        if i == 0:
            dump = res.pop("dump", None)
            line = res
        else:
            workloads.append(res)
    inv = shard_invariance(ctx, cfg)

    if rank == 0:
        out = {"metric": METRIC, "value": line["value"], "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": line["ms_per_step"], "higher_is_better": True, "scaling": "weak",
               "vs_baseline": None, "dtype": "f64", "data": "synthetic"}
        out.update({k: v for k, v in line.items() if k not in out})
        if inv is not None:
            out["shard_invariant"] = inv
        if workloads:
            out["workloads"] = workloads
        if not args.no_cpu_baseline and world == 1:
            import oracle
            oracle.build()
            cores = len(os.sched_getaffinity(0))
            # bounded sample of the same workload, sized for ~10 s of CPU work from a short calibration run
            pk = cfg["params"]
            n_envs = min(cfg["envs"], 4096)
            use_ox = cfg["gaze"] == "Oxford"
            v0, dt0 = cpu_port_run(pk, n_envs, 20, cores, oxford=use_ox)
            steps_c = int(min(20000, max(50, 25.0 * v0 / n_envs)))   # the 20-step calibration under-reads the rate ~2x
            v, dt = cpu_port_run(pk, n_envs, steps_c, cores, oxford=use_ox)
            out["cpu_baseline"] = {"value": v, "unit": "env-steps/s", "cores": cores, "kind": "port",
                                   "sample": "%d envs x %d steps of the same workload, auto-reset on (%.1f s)" % (n_envs, steps_c, dt)}
        if dump is not None:
            write_dump(args.dump_outputs, dump)
            log("outputs of the headline path (%d envs) written to %s" % (len(dump["env_index"]), args.dump_outputs))
        emit(out)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
