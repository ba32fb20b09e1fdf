"""`Drone2DEnv2`: single-environment facade with the reference's exact class / attribute names
(envs/drone_v2.py:10-305), backed by a B=1 `Drone2DVecEnv` on the GPU.  It exists so that code written against the
reference -- `experiment.py`'s run loop, the gaze policies reading `env.info`, metric scripts poking `env.drone.x` --
runs unchanged; throughput work should use `Drone2DVecEnv` directly.

Proxies read device state lazily (one small D2H copy per attribute access) and never cache across steps.
"""
import types

import numpy as np
import torch

from .params import state_machine as STATE_MACHINE
from .vec_env import Drone2DVecEnv, trajectory_waypoints


class _GridMapProxy(object):
    """`drone.map` / `env.map_gt` (OccupancyGridMap, utils.py:494-548)."""

    def __init__(self, env, which):
        self._env, self._which = env, which
        p = env.params
        self.dim = list(p.map_size)
        self.x_scale = self.y_scale = p.map_scale
        self.width, self.height = p.map_size[0] // p.map_scale, p.map_size[1] // p.map_scale

    @property
    def grid_map(self):
        if self._which == "belief":
            return self._env._vec.buffer("belief")[0].cpu().numpy()
        v = self._env._vec
        rows = v.buffer("gt_rows")[0].cpu().numpy().astype(np.uint64)
        bits = (rows[:, None] >> np.arange(self.height, dtype=np.uint64)[None, :]) & np.uint64(1)
        g = np.where(bits == 1, 1, 2).astype(np.uint8)        # OCCUPIED / UNOCCUPIED
        # DYNAMIC_OCCUPIED marks (value 3).  The step kernels never compute them -- nothing on the hot path reads them
        # (perception, collision and observation test `== 1`) -- so the view is synthesised here from the agent state:
        pos = v.buffer("agent_pos")[0].cpu().numpy().reshape(-1, 2)
        rad = v.buffer("agent_radius")[0].cpu().numpy().reshape(-1)
        if int(v.buffer("steps")[0].item()) == 0:
            # right after __init__ / reset(): init_obstacles marks every cell whose CENTRE lies in an agent disc, border
            # cells included (utils.py:520-525)
            cx = self.x_scale * (np.arange(self.width) + 0.5)
            cy = self.y_scale * (np.arange(self.height) + 0.5)
            for (ax, ay), r in zip(pos, rad):
                g[((cx[:, None] - ax) ** 2 + (cy[None, :] - ay) ** 2) <= r ** 2] = 3
            return g
        # after a step: update_dynamic_grid (utils.py:527-540) stamps a (2*(r // scale) + 1)^2 box of cells around every
        # agent's cell, except on OCCUPIED cells; last step's marks were demoted to UNOCCUPIED first
        for (ax, ay), r in zip(pos, rad):
            ux, uy = int(r // self.x_scale), int(r // self.y_scale)
            pi, pj = int(ax // self.x_scale), int(ay // self.y_scale)
            i0, i1 = max(pi - ux, 0), min(pi + ux + 1, self.width)
            j0, j1 = max(pj - uy, 0), min(pj + uy + 1, self.height)
            if i1 > i0 and j1 > j0:
                box = g[i0:i1, j0:j1]
                box[box != 1] = 3
        return g

    def get_grid(self, x, y):                                 # utils.py:545-548
        if x >= self.dim[0] or x < 0 or y >= self.dim[1] or y < 0:
            return 1
        return self.grid_map[int(x // self.x_scale), int(y // self.y_scale)]


class _TrackerProxy(object):
    def __init__(self, env, i):
        self._env, self._i = env, i

    @property
    def active(self):
        return bool(self._env._vec.buffer("tracker_active")[0, self._i].item())

    @property
    def radius(self):
        return float(self._env._vec.buffer("tracker_radius")[0, self._i].item())

    @property
    def mu_upds(self):
        return [self._env._vec.buffer("tracker_mu")[0, self._i].cpu().numpy().reshape(4, 1)]

    @property
    def Sigma_upds(self):
        return [self._env._vec.buffer("tracker_sigma")[0, self._i].cpu().numpy()]

    @property
    def ts(self):
        return [float(k) for k in range(int(self._env._vec.buffer("tracker_ts")[0, self._i].item()))]

    def estimate_pos(self, t):                                # utils.py:220-223
        mu = self.mu_upds[-1]
        return mu[:2, 0] + t * mu[2:, 0]


class _BufferedTracker(object):
    def __init__(self, n):
        self.ts = [float(k) for k in range(n)]


class _DroneProxy(object):
    """`env.drone` (Drone2D, utils.py:714-784): x / y / yaw are readable AND writable like the reference's attributes."""

    def __init__(self, env):
        self._env = env
        p = env.params
        self.yaw_range, self.yaw_depth, self.radius, self.dt, self.params = p.drone_view_range, p.drone_view_depth, \
            p.drone_radius, p.dt, p
        self.map = _GridMapProxy(env, "belief")
        self.trackers = [_TrackerProxy(env, i) for i in range(env._vec.num_agents)]

    def _get(self, name):
        return float(self._env._vec.buffer(name)[0].item())

    def _set_pose(self, x=None, y=None, yaw=None):
        pose = [self.x if x is None else x, self.y if y is None else y, self.yaw if yaw is None else yaw]
        self._env._vec.set_drone_pose(np.array([pose], dtype=np.float64))

    x = property(lambda self: self._get("drone_x"), lambda self, v: self._set_pose(x=v))
    y = property(lambda self: self._get("drone_y"), lambda self, v: self._set_pose(y=v))
    yaw = property(lambda self: self._get("drone_yaw"), lambda self, v: self._set_pose(yaw=v))

    @property
    def velocity(self):
        return np.array([self._get("drone_vx"), self._get("drone_vy")])

    @property
    def acceleration(self):
        return np.zeros(2)

    def get_local_map(self):
        return self._env._vec.buffer("local_map")[0, 0].cpu().numpy()


class _TrajectoryProxy(object):
    """`planner.trajectory` (Trajectory2D, utils.py:280-298), expanded on demand from the stored A* segments."""

    def __init__(self, env):
        self._env = env

    def _expand(self):
        v = self._env._vec
        return trajectory_waypoints(v.cfg, v.buffer("traj_coeff")[0].cpu().numpy(), int(v.buffer("traj_nseg")[0].item()),
                                    int(v.buffer("traj_cursor")[0].item()))

    @property
    def positions(self):
        return list(self._expand()[0])

    @property
    def velocities(self):
        return list(self._expand()[1])

    @property
    def accelerations(self):
        return [np.array([0, 0]) for _ in range(len(self))]

    def __len__(self):
        v = self._env._vec
        return int(v.buffer("traj_nseg")[0].item()) * v.cfg.n_way - int(v.buffer("traj_cursor")[0].item())


class _AgentProxy(object):
    def __init__(self, env, i):
        self._env, self._i = env, i

    @property
    def position(self):
        return self._env._vec.buffer("agent_pos")[0, self._i].cpu().numpy()

    @property
    def pref_velocity(self):
        return self._env._vec.buffer("agent_pref")[0, self._i].cpu().numpy()

    @property
    def velocity(self):
        # CVM: velocity IS pref_velocity (drone_v2.py:178); RVO: the velocity RVO_update chose (drone_v2.py:169-173)
        if self._env._vec.cfg.motion_profile == 1:
            return self._env._vec.buffer("agent_vel")[0, self._i].cpu().numpy()
        return self.pref_velocity

    @property
    def radius(self):
        return float(self._env._vec.buffer("agent_radius")[0, self._i].item())


class _PlannerProxy(object):
    def __init__(self, env):
        self._env = env
        self.trajectory = _TrajectoryProxy(env)

    @property
    def target(self):
        v = self._env._vec
        return np.array([v.buffer("target_x")[0].item(), v.buffer("target_y")[0].item(), 0.0, 0.0])


class Drone2DEnv2(object):
    """Drop-in for `envs.drone_v2.Drone2DEnv2(params)`."""

    def __init__(self, params, device="cuda:0"):
        self.params = params
        self.dt = params.dt
        self.max_steps = params.max_flight_time / params.dt
        self.target_list = [list(t) for t in params.target_list]
        from .world import generate_worlds
        worlds = generate_worlds(params, [params.map_id])
        self._vec = Drone2DVecEnv(params, 1, seeds=[params.map_id], device=device, auto_reset=False, worlds=worlds,
                                  oxford=getattr(params, "gaze_method", "") == "Oxford",
                                  owl=getattr(params, "gaze_method", "") == "Owl")
        self.drone = _DroneProxy(self)
        self.planner = _PlannerProxy(self)
        self.agents = [_AgentProxy(self, i) for i in range(self._vec.num_agents)]
        self.map_gt = _GridMapProxy(self, "gt")
        # circular pillars [x, y, rad] of init_obstacles_random_size (drone_v2.py:14-27); empty unless pillar_number > 0
        self.obstacles = [list(o) for o in np.asarray(self._pillars(params), dtype=np.float64).reshape(-1, 3)]
        L = self._vec.local_map_size
        box = types.SimpleNamespace
        self.action_space = box(low=np.array([-1.0]), high=np.array([1.0]), shape=(1,))
        self.observation_space = box(spaces={"yaw_angle": box(shape=(1,), dtype=np.float32),
                                             "local_map": box(shape=(1, L, L), dtype=np.float32),
                                             "swep_map": box(shape=(1, L, L), dtype=np.float32)})
        self._a = torch.zeros(1, dtype=torch.float64, device=self._vec.device)

    @staticmethod
    def _pillars(params):
        from .world import generate_world, load_static_map
        if getattr(params, "pillar_number", 0) <= 0:
            return np.zeros((0, 3))
        return generate_world(params, int(params.map_id), load_static_map(params.static_map))["obstacles"]

    # ---- reference attributes
    @property
    def steps(self):
        return int(self._vec.buffer("steps")[0].item())

    @property
    def state_machine(self):
        return int(self._vec.buffer("state_machine")[0].item())

    @property
    def fail_count(self):
        return int(self._vec.buffer("fail_count")[0].item())

    @property
    def tracker_buffer(self):
        cnt = int(self._vec.buffer("tracker_buffer_count")[0].item())
        tot = int(self._vec.buffer("tracker_buffer_ts")[0].item())
        if cnt == 0:
            return []
        base, rem = divmod(tot, cnt)      # only len() and the sum of len(ts) are observable (experiment.py:74-91)
        return [_BufferedTracker(base + (1 if i < rem else 0)) for i in range(cnt)]

    @property
    def info(self):                       # drone_v2.py:238-250
        v = self._vec
        return {"drone": self.drone, "trajectory": self.planner.trajectory, "state_machine": self.state_machine,
                "target": self.planner.target, "collision_flag": int(v.buffer("collision_flag")[0].item()),
                "dead_lock_flag": int(v.buffer("dead_lock_flag")[0].item()),
                "freezing_flag": int(v.buffer("freezing_flag")[0].item()), "flight_time": self.steps * self.dt,
                "tracker_buffer": self.tracker_buffer}

    # ---- gym protocol
    def reset(self):
        self._vec.reset()
        return {}                         # the reference returns {} (drone_v2.py:261)

    def step(self, a):
        self._a.fill_(float(a))
        obs, _, done, _ = self._vec.step(self._a)
        lm = obs["local_map"][0].cpu().numpy()
        state = {"local_map": lm, "swep_map": lm.copy(), "yaw_angle": obs["yaw_angle"][0].cpu().numpy()}
        return state, 0, bool(done[0].item()), self.info

    # ---- state snapshots (ALE cloneState / restoreState, MuJoCo get_state / set_state)
    def get_state(self):
        """A snapshot of the whole env -- live state and reset snapshot -- as returned by Drone2DVecEnv.save_state."""
        return self._vec.save_state([0])

    def set_state(self, s):
        """Restores a snapshot of `get_state` (of this env or of one with the same params); later steps repeat bit for bit."""
        self._vec.load_state(s, [0])

    def render(self, mode="human"):
        """mode="rgb_array": the env's frame as numpy uint8 [500, 500, 3] (10 pixels per cell, every layer), drawn on the
        device (Drone2DVecEnv.render).  There is no pygame window."""
        if mode == "rgb_array":
            return self._vec.render([0], pixels_per_cell=10)[0].cpu().numpy()
        raise NotImplementedError("render(mode=%r): there is no pygame window on the B200 path; use mode=\"rgb_array\" "
                                  "(see DESIGN.md §7)" % (mode,))

    def close(self):
        self._vec.close()


_REGISTRY = {"gym-2d-perception-v2": Drone2DEnv2}


def make(env_id, params=None, **kw):
    """gym.make('gym-2d-perception-v2', params=params) (envs/__init__.py:5-8, experiment.py:31)."""
    return _REGISTRY[env_id](params=params, **kw)
