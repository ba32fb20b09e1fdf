"""Per-phase timeline of the last step of d2d_rollout launches (BASELINE config 2) from a -DD2D_WARP_PROF build of the library
given as the only argument (%globaltimer stamps of every warp: step start, before the ray phase, after it, after the
leader / observation part, step end).  GPU box only:  python tools/rollout_phase_prof.py <path to libdrone2d.so>"""
import os, sys
sys.path.insert(0, os.getcwd())
import numpy as np
from gym_drone2d_activeperception_b200 import _native
_native.LIB_PATH = sys.argv[1]
import torch, bench
from gym_drone2d_activeperception_b200 import Params
from gym_drone2d_activeperception_b200.vec_env import Drone2DVecEnv
cfg = bench.CONFIGS[2]; B, pk = cfg["envs"], cfg["params"]
worlds = bench.make_worlds(pk, pk["map_id"] + np.arange(B))
env = Drone2DVecEnv(Params(debug=False, **pk), B, worlds=worlds, device="cuda:0", auto_reset=True)
table = torch.as_tensor(np.arange(-80, 80, 80 / 3) / 80, device="cuda:0")
g = torch.Generator(device="cuda:0"); g.manual_seed(1)
for _ in range(5):
    env.rollout(table[torch.randint(0, 6, (200, B), device="cuda:0", generator=g)].contiguous())
torch.cuda.synchronize()
prof = env.buffer("warp_prof")
d = {k: [] for k in ("agents+setup 0-1", "rays 1-2", "trackers+leader+obs 2-4", "tail 4-3", "step 0-3")}
for _ in range(20):
    env.rollout(table[torch.randint(0, 6, (50, B), device="cuda:0", generator=g)].contiguous())
    torch.cuda.synchronize()
    p = prof.cpu().numpy().astype(np.int64)
    t0, t1, t2, t3, t4 = p[:, 0], p[:, 1], p[:, 2], p[:, 3], p[:, 4]
    d["agents+setup 0-1"].append(t1 - t0); d["rays 1-2"].append(t2 - t1); d["trackers+leader+obs 2-4"].append(t4 - t2)
    d["tail 4-3"].append(t3 - t4); d["step 0-3"].append(t3 - t0)
print("lib", os.path.basename(os.path.dirname(sys.argv[1])), "B", B, "(last step of 20 launches x 4096 warps, ns per warp)")
for k, v in d.items():
    v = np.concatenate(v)
    print("  %-26s mean %8.1f  p50 %8.1f  p90 %8.1f  max %8.1f" % (k, v.mean(), np.median(v), np.percentile(v, 90), v.max()))
env.close()
