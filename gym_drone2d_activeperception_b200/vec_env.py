"""`Drone2DVecEnv`: the batched drop-in for the reference's `Drone2DEnv2` (envs/drone_v2.py:10-305).

Same protocol as the reference env -- `reset()`, `step(a) -> (obs, reward, done, info)`, observation keys
`local_map` / `swep_map` / `yaw_angle`, reward identically 0 (drone_v2.py:257) -- with a leading batch axis and
all arrays living on the GPU as torch tensors that alias the CUDA library's arena (no copies).  Every step is
executed by hand-written sm_100a kernels behind the C ABI of include/drone2d.h; there is no CPU fallback.
"""
import ctypes as C
import math

import numpy as np
import torch

from . import _native
from .params import Params
from .world import count_agents, generate_worlds, load_static_map, world_key, world_source

_TORCH_DTYPES = {0: (torch.uint8, "|u1"), 1: (torch.int8, "|i1"), 2: (torch.int32, "<i4"), 3: (torch.int64, "<i8"),
                 4: (torch.float32, "<f4"), 5: (torch.float64, "<f8")}


class _DevView(object):
    """Zero-copy description of a device buffer for torch.as_tensor (CUDA array interface v2)."""

    def __init__(self, ptr, shape, strides_elems, typestr, itemsize):
        self.__cuda_array_interface__ = {
            "shape": tuple(int(s) for s in shape),
            "typestr": typestr,
            "data": (int(ptr), False),
            "version": 2,
            "strides": tuple(int(s) * itemsize for s in strides_elems),
        }


def oxford_cos_threshold(view_range_deg):
    """c* = min{c : np.arccos(c) <= radians(view_range/2)} by bisection over doubles using the ARRAY np.arccos
    (the loop Oxford.get_view_map runs, yaw_planner.py:78).  The device then tests `c >= c*` (SURVEY §7.3-10)."""
    ang = math.radians(view_range_deg / 2)

    def ok(c):
        return bool(np.arccos(np.full(9, c))[0] <= ang)

    lo, hi = -1.0, 1.0
    if ok(lo):
        return -1.0
    while True:
        mid = lo + (hi - lo) / 2
        if mid == lo or mid == hi:
            return hi
        if ok(mid):
            hi = mid
        else:
            lo = mid


def make_config(params, num_envs, num_agents, device_index, auto_reset=True, trackers=True, oxford=False,
                envs_per_block=0, strip_width=10, owl=False):
    """Fills d2d_config from a reference-style Params object; lookup tables use the reference's numpy expressions."""
    cfg = _native.D2DConfig()
    cfg.struct_size = C.sizeof(_native.D2DConfig)
    cfg.device = device_index
    cfg.num_envs = num_envs
    cfg.num_agents = num_agents
    if params.planner not in ("NoMove", "Primitive", "Jerk_Primitive"):
        raise ValueError("planner %r is not supported (NoMove, Primitive, Jerk_Primitive)" % (params.planner,))
    if params.motion_profile not in ("CVM", "RVO"):
        raise ValueError("motion_profile %r is not supported (CVM, RVO)" % (params.motion_profile,))
    cfg.motion_profile = {"CVM": 0, "RVO": 1}[params.motion_profile]
    cfg.planner = {"NoMove": 0, "Primitive": 1, "Jerk_Primitive": 2}[params.planner]
    cfg.trackers = 1 if trackers else 0
    cfg.auto_reset = 1 if auto_reset else 0
    cfg.oxford = (_native.POLICY_OXFORD if oxford else 0) | (_native.POLICY_OWL if owl else 0)
    cfg.envs_per_block = envs_per_block
    cfg.n_rays = math.ceil(params.map_size[0] / strip_width)            # utils.py:587
    cfg.dt, cfg.map_scale = params.dt, params.map_scale
    cfg.map_w, cfg.map_h = params.map_size
    cfg.agent_radius = params.agent_radius
    cfg.drone_max_acceleration = params.drone_max_acceleration
    cfg.drone_radius = params.drone_radius
    cfg.drone_max_yaw_speed = params.drone_max_yaw_speed
    cfg.drone_view_depth = params.drone_view_depth
    cfg.drone_view_range = params.drone_view_range
    cfg.max_flight_time = params.max_flight_time
    cfg.var_cam = params.var_cam
    cfg.drone_max_speed = params.drone_max_speed
    cfg.ox_cos_thresh = oxford_cos_threshold(params.drone_view_range)
    tl = params.target_list
    if len(tl) > _native.MAX_TARGETS:
        raise ValueError("at most %d targets" % _native.MAX_TARGETS)
    cfg.n_targets = len(tl)
    for i, t in enumerate(tl):
        cfg.targets[i][0], cfg.targets[i][1] = float(t[0]), float(t[1])
    # Primitive.__init__ traj_planner.py:98-104
    if params.drone_max_speed <= 40:
        u = np.arange(-params.drone_max_acceleration, params.drone_max_acceleration, 0.4 * params.drone_max_speed - 5)
    else:
        u = np.arange(-params.drone_max_acceleration, params.drone_max_acceleration, 4)
    pdt = 2
    sample_num = params.drone_max_speed * pdt // params.map_scale
    ts = np.arange(0, pdt, pdt / sample_num)                             # traj_planner.py:180
    tw = np.arange(pdt, 0, -params.dt)                                   # traj_planner.py:212
    if len(u) > _native.MAX_U or len(ts) > _native.MAX_SAMP or len(tw) > _native.MAX_WAY:
        raise ValueError("planner tables too large")
    cfg.n_u, cfg.n_samp, cfg.n_way = len(u), len(ts), len(tw)
    for i, v in enumerate(u):
        cfg.u_space[i] = float(v)
    for i, t in enumerate(ts):
        cfg.t_samp[i], cfg.t_samp2[i] = float(t), float(t ** 2)
    for i, t in enumerate(tw):
        cfg.t_way[i], cfg.t_way2[i], cfg.t_way_x2[i] = float(t), float(t ** 2), float(2 * t)
    vy = np.arange(-params.drone_max_yaw_speed, params.drone_max_yaw_speed, params.drone_max_yaw_speed / 3)
    cfg.n_yaw = len(vy)                                                  # yaw_planner.py:65
    for i, v in enumerate(vy):
        cfg.v_yaw_space[i] = float(v)
    # Owl.__init__ yaw_planner.py:153-167
    ou = np.arange(-params.drone_max_yaw_speed, params.drone_max_yaw_speed, params.drone_max_yaw_speed / 10)
    if len(ou) > _native.MAX_OWL_U:
        raise ValueError("Owl u_space too large")
    cfg.n_owl_u = len(ou)
    for i, v in enumerate(ou):
        cfg.owl_u_space[i] = float(v)
    cfg.owl_repeat = max(0, int(0.8 // params.dt) - 1)                   # yaw_planner.py:220
    return cfg


def config_difference(a, b):
    """The name of the first d2d_config field in which `a` and `b` differ (compared byte for byte), or None."""
    for f in _native.D2DConfig._fields_:
        d = getattr(_native.D2DConfig, f[0])
        if C.string_at(C.addressof(a) + d.offset, d.size) != C.string_at(C.addressof(b) + d.offset, d.size):
            return f[0]
    return None


class Drone2DVecEnv(object):
    """Batched `Drone2DEnv2`.

    params    : reference-style `Params` (ours or the reference's own object; only attributes are read)
    num_envs  : B environments on this GPU
    seeds     : per-env RNG seeds (default `params.map_id + arange(B)`; the reference seeds with map_id)
    worlds    : optional pre-generated worlds (dict of arrays as returned by world.generate_worlds)
    auto_reset: an env that returned done=True is re-initialised (same seed => same world, exactly what the
                reference's reset() does) at the start of its next step; the terminal observation is returned.
    world_gen : "host" (default) builds the worlds with world.generate_worlds and uploads them; "device" generates them
                on the GPU (d2d_generate_worlds), identical except for the documented group-velocity rounding (DESIGN.md
                section 2).  `reseed` needs neither.  Cannot be combined with `worlds`.
    world_sources, sources : world_gen="device" only: the handle's table of world sources (`set_world_sources`, a list of
                Params that share this handle's config) and the source of each env's initial world (default 0), so the
                initial worlds can come from many configurations; `seeds` then holds world keys (world.world_key).
    """

    metadata = {"render.modes": ["rgb_array"]}

    def __init__(self, params, num_envs, seeds=None, device="cuda:0", auto_reset=True, trackers=True, oxford=None,
                 envs_per_block=0, strip_width=10, worlds=None, owl=None, jerk_tie_orders=None, world_gen="host",
                 world_sources=None, sources=None):
        if world_gen not in ("host", "device"):
            raise ValueError("world_gen must be 'host' or 'device', got %r" % (world_gen,))
        if world_gen == "device" and worlds is not None:
            raise ValueError("world_gen='device' generates the worlds itself: do not pass `worlds`")
        if world_gen != "device" and (world_sources is not None or sources is not None):
            raise ValueError("world_sources / sources need world_gen='device'")
        if sources is not None and world_sources is None:
            raise ValueError("sources index a table of world sources: pass world_sources too")
        if not torch.cuda.is_available():
            raise _native.Drone2DNativeError("CUDA device required: Drone2DVecEnv has no CPU path")
        self.params = params
        self.num_envs = int(num_envs)
        self.device = torch.device(device)
        self._dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self._lib = _native.load()
        self._smap = load_static_map(params.static_map)
        self.num_agents = count_agents(params, self._smap)
        if oxford is None:
            oxford = getattr(params, "gaze_method", "") == "Oxford"
        if owl is None:
            owl = getattr(params, "gaze_method", "") == "Owl"
        self._cfg_kw = dict(auto_reset=auto_reset, trackers=trackers, oxford=oxford, envs_per_block=envs_per_block,
                            strip_width=strip_width, owl=owl)
        self.cfg = make_config(params, self.num_envs, self.num_agents, self._dev_index, **self._cfg_kw)
        self._h = C.c_void_p()
        rc = self._lib.d2d_create(C.byref(self.cfg), C.byref(self._h))
        if rc != 0:
            msg = self._lib.d2d_last_error(None)
            raise _native.Drone2DNativeError("d2d_create failed (%d): %s" % (rc, msg.decode() if msg else "?"))
        if self.cfg.planner == 2:       # Jerk_Primitive: per-heading tables evaluated with the reference's numpy expressions
            from . import jerk
            self._jerk_tables = jerk.make_tables(params, jerk_tie_orders)
            self._check(self._lib.d2d_set_jerk_tables(self._h, C.byref(self._jerk_tables)), "d2d_set_jerk_tables")
        # a copy: reseed / clone_envs / load_state rewrite entries, and must not write into the caller's array
        self.seeds = np.array(seeds if seeds is not None else params.map_id + np.arange(self.num_envs), dtype=np.int64)
        self._world_sources = None
        self._log_capacity, self._queue_set = 0, False
        if world_gen == "device":
            if world_sources is not None:
                self.set_world_sources(world_sources)
            self.reseed(np.arange(self.num_envs), self.seeds, sources=sources)
            torch.cuda.current_stream(self.device).synchronize()
            self.check_worlds()
        else:
            if worlds is None:
                worlds = generate_worlds(params, self.seeds, self._smap)
            self.set_worlds(worlds)
        self._views = {}
        self._mirror, self._mirror_ptrs = None, (None, None, None)
        self.local_map_size = 4 * (params.drone_view_depth // params.map_scale) + 1
        self.reward = self.buffer("reward")
        self._zero_actions = torch.zeros(self.num_envs, dtype=torch.float64, device=self.device)

    # ------------------------------------------------------------------ plumbing
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _check(self, rc, what):
        _native.check(self._h, rc, what)

    def set_worlds(self, worlds, first_env=0):
        w = {k: np.ascontiguousarray(v) for k, v in worlds.items()}
        count = w["drone_pose"].shape[0]
        n = self.num_agents
        assert w["agent_radius"].shape == (count, n), (w["agent_radius"].shape, count, n)

        def p(a, dt):
            a = np.ascontiguousarray(a, dtype=dt)
            return a, a.ctypes.data_as(C.c_void_p)

        keep = [p(w["agent_pos"], np.float64), p(w["agent_pref"], np.float64), p(w["agent_radius"], np.float64),
                p(w["tracker_radius"], np.float64), p(w["gt_grid"], np.uint8), p(w["drone_pose"], np.float64)]
        self._check(self._lib.d2d_set_world(self._h, first_env, count, *[k[1] for k in keep]), "d2d_set_world")
        if self.cfg.motion_profile == 1:      # RVO: initial velocities + circular obstacles (d2d_set_rvo)
            if "agent_vel" not in w or "obstacles" not in w:
                raise ValueError("motion_profile 'RVO' needs worlds with 'agent_vel' and 'obstacles' (world.generate_worlds)")
            obs = np.ascontiguousarray(w["obstacles"], dtype=np.float64).reshape(count, -1, 3)
            if obs.shape[1] > 16:
                raise ValueError("motion_profile 'RVO': at most 16 circular obstacles (pillar_number) per env")
            nobs = np.full(count, obs.shape[1], dtype=np.int32)
            rv = [p(w["agent_vel"], np.float64), p(obs, np.float64), p(nobs, np.int32)]
            self._check(self._lib.d2d_set_rvo(self._h, first_env, count, rv[0][1], rv[1][1], rv[2][1], int(obs.shape[1])),
                        "d2d_set_rvo")
        if "rng_key" in w:      # legacy np.random stream state (only consumed when var_cam != 0)
            rk = [p(w["rng_key"], np.uint32), p(w["rng_pos"], np.int32), p(w["rng_has_gauss"], np.int32),
                  p(w["rng_gauss"], np.float64)]
            self._check(self._lib.d2d_set_rng(self._h, first_env, count, *[k[1] for k in rk]), "d2d_set_rng")

    def set_world_sources(self, configs):
        """The handle's table of world sources (d2d_set_world_sources): `configs[k]` (a Params) is source k of the world
        keys `reseed(..., sources=)` and `set_seed_queue(..., sources=)` take.  Every config must give this handle's
        d2d_config field for field (make_config: agent_radius, num_agents, drone and planner parameters, targets, view
        range, ...); they may differ in what only shapes the world -- the static map, agent_number within the same agent
        count, pillar_number, agent_max_speed, init_pos.  ValueError names the first field that differs.  Replaces the
        table; until the first call the handle's own params are source 0."""
        configs = list(configs)
        if not 1 <= len(configs) <= _native.WORLD_MAX_SOURCES:
            raise ValueError("set_world_sources: %d configs (1..%d)" % (len(configs), _native.WORLD_MAX_SOURCES))
        srcs = (_native.D2DWorldSource * len(configs))()
        for k, p in enumerate(configs):
            smap = load_static_map(p.static_map)
            field = config_difference(self.cfg, make_config(p, self.num_envs, count_agents(p, smap), self._dev_index,
                                                            **self._cfg_kw))
            if field is not None:
                raise ValueError("set_world_sources: config %d differs from the handle's config in %r" % (k, field))
            srcs[k] = world_source(p, smap)
        self._upload_sources(configs, srcs)

    def _upload_sources(self, configs, srcs):
        self._check(self._lib.d2d_set_world_sources(self._h, srcs, len(configs)), "d2d_set_world_sources")
        self._world_sources = list(configs)

    def _default_sources(self):
        """The handle's own params as source 0, as the handle was created (no config comparison)."""
        if self._world_sources is None:
            self._upload_sources([self.params], (_native.D2DWorldSource * 1)(world_source(self.params, self._smap)))

    def _keys(self, what, seeds, sources, n):
        """`seeds` (sources=None: seeds or keys as given) or world_key(sources, seeds) as a contiguous int64 array of n."""
        sd = np.asarray(seeds).reshape(-1)
        if sd.size and sd.dtype.kind not in "iu":
            raise ValueError("seeds must be integers, got %s" % sd.dtype)
        if sources is not None:
            src = np.asarray(sources).reshape(-1)
            if src.size != sd.size:
                raise ValueError("%s: %d sources for %d seeds" % (what, src.size, sd.size))
            sd = world_key(src, sd)
        sd = np.ascontiguousarray(sd, dtype=np.int64)
        if n is not None and sd.size != n:
            raise ValueError("%s: %d seeds for %d envs" % (what, sd.size, n))
        return sd

    def reseed(self, envs, seeds, lazy=False, sources=None):
        """Gives envs[i] the world of seeds[i], generated on the GPU (d2d_generate_worlds, one launch, asynchronous):
        lazy=False resets those envs now, as `reset` does; lazy=True marks them, and each starts its new world at its next
        step -- the path auto-reset takes after done, so the terminal outputs of an env that just reported done stay
        readable until then.  Afterwards `seeds[e]` is the seed of the world env e resets into.  Seeds must lie in
        [0, 2**32), as np.random.RandomState requires.  With `sources` (indices into the table of `set_world_sources`) env
        envs[i] gets the world of seed seeds[i] built from source sources[i] (d2d_generate_worlds_keyed), and `seeds[e]`
        holds its world key.  A seed whose world cannot be built is reported by the next call or by `check_worlds`."""
        idx = self._env_indices(envs)
        sd = self._keys("reseed", seeds, sources, idx.size)
        self._default_sources()
        flags = _native.WORLD_LAZY if lazy else _native.WORLD_EAGER
        fn, name = ((self._lib.d2d_generate_worlds, "d2d_generate_worlds") if sources is None else
                    (self._lib.d2d_generate_worlds_keyed, "d2d_generate_worlds_keyed"))
        self._check(fn(self._h, idx.ctypes.data_as(C.c_void_p), sd.ctypes.data_as(C.c_void_p), int(idx.size), flags,
                       self._stream()), name)
        self.seeds[idx] = sd
        self._set_world_seeds(idx, sd)

    def check_worlds(self):
        """Raises if an earlier `reseed` met a seed whose world cannot be built (call after synchronising the stream)."""
        if self._world_sources is not None:
            self._check(self._lib.d2d_generate_worlds(self._h, None, None, 0, _native.WORLD_EAGER, self._stream()),
                        "d2d_generate_worlds")

    def buffer(self, name):
        """Torch tensor aliasing the named arena buffer (see DESIGN.md / d2d_get_buffer)."""
        # "oxford_last_time_observed" is materialised from the compact policy state on every request (never cached)
        cacheable = name != "oxford_last_time_observed"
        t = self._views.get(name) if (cacheable and hasattr(self, "_views")) else None
        if t is not None:
            return t
        info = _native.D2DBufferInfo()
        self._check(self._lib.d2d_get_buffer(self._h, name.encode(), C.byref(info)), "d2d_get_buffer(%s)" % name)
        tdt, typestr = _TORCH_DTYPES[info.dtype]
        shape = [info.shape[i] for i in range(info.ndim)]
        strides = [info.strides[i] for i in range(info.ndim)]
        if 0 in shape:
            t = torch.empty(shape, dtype=tdt, device=self.device)
        else:
            view = _DevView(info.dev_ptr, shape, strides, typestr, torch.empty((), dtype=tdt).element_size())
            t = torch.as_tensor(view, device=self.device)
        if cacheable and hasattr(self, "_views"):
            self._views[name] = t
        return t

    # ------------------------------------------------------------------ gym-style API
    def _obs(self):
        lm = self.buffer("local_map")
        # the reference returns the same crop under both keys (drone_v2.py:252-253)
        return {"local_map": lm, "swep_map": lm, "yaw_angle": self.buffer("yaw_angle")}

    def reset(self, mask=None, lazy=False):
        """reset() of the reference re-runs __init__ (drone_v2.py:259-261) and returns {}; here the initial observation
        is returned (zeros + initial yaw).  mask: optional bool/uint8 CUDA tensor [B] selecting envs.  lazy=True only marks
        the envs (d2d_request_reset): they are re-initialised inside their next step, like an env that returned done under
        auto_reset; the observation tensors keep their content until then."""
        mptr = None
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            mptr = C.c_void_p(mask.data_ptr())
        if lazy:
            self._check(self._lib.d2d_request_reset(self._h, mptr, self._stream()), "d2d_request_reset")
        else:
            self._check(self._lib.d2d_reset(self._h, mptr, self._stream()), "d2d_reset")
        return self._obs()

    def step(self, actions):
        """actions: float64 CUDA tensor [B] (or [B,1]) in [-1, 1] (action_space Box(-1,1,(1,)), drone_v2.py:120).
        Returns (obs, reward, done, info): reward is the constant-zero tensor, done a uint8 tensor [B]."""
        if not torch.is_tensor(actions):
            actions = torch.as_tensor(np.asarray(actions, dtype=np.float64), device=self.device)
        a = actions.to(device=self.device, dtype=torch.float64).reshape(-1).contiguous()
        if a.numel() != self.num_envs:
            raise ValueError("expected %d actions, got %d" % (self.num_envs, a.numel()))
        self._check(self._lib.d2d_step(self._h, C.c_void_p(a.data_ptr()), self._stream()), "d2d_step")
        return self._obs(), self.reward, self.buffer("done"), self.info

    def rollout(self, actions):
        """K consecutive steps in ONE launch (d2d_rollout): `actions` is a float64 CUDA tensor [K, B] (row t = the actions of
        step t) or [B] with `steps` implied 1.  Every warp walks its env through the K steps with the env's state resident on
        chip; all buffers and statistics end up bit-identical to K `step` calls, the per-step outputs hold the last step's
        values.  NoMove planner / CVM profile only (other configurations raise).  Returns what the last `step` would."""
        a = actions.to(device=self.device, dtype=torch.float64)
        if a.dim() == 1:
            a = a.reshape(1, -1)
        a = a.reshape(a.shape[0], -1).contiguous()
        if a.shape[1] != self.num_envs:
            raise ValueError("expected [K, %d] actions, got %s" % (self.num_envs, tuple(a.shape)))
        self._check(self._lib.d2d_rollout(self._h, C.c_void_p(a.data_ptr()), int(a.shape[0]), int(a.shape[1]), self._stream()),
                    "d2d_rollout")
        return self._obs(), self.reward, self.buffer("done"), self.info

    def step_host(self, actions_host, local_map_host=None, yaw_host=None, done_host=None):
        """Same step through HOST buffers (pinned torch tensors or numpy arrays): actions to the device (pinned memory is
        read by the kernels in place), step, observation back on the host.  Output buffers that are the bound mirror
        (`bind_host_mirror`) cost nothing here: their pointers are cached and the library copies nothing."""
        def ptr(x):
            if x is None:
                return None
            return x.data_ptr() if torch.is_tensor(x) else x.ctypes.data
        m = self._mirror
        if m is not None and local_map_host is m[0] and yaw_host is m[1] and done_host is m[2]:
            lp, yp, dp = self._mirror_ptrs
        else:
            lp, yp, dp = ptr(local_map_host), ptr(yaw_host), ptr(done_host)
        rc = self._lib.d2d_step_host(self._h, ptr(actions_host), lp, yp, dp,
                                     torch.cuda.current_stream(self.device).cuda_stream)
        if rc != 0:
            self._check(rc, "d2d_step_host")

    def bind_host_mirror(self, local_map_host=None, yaw_host=None, done_host=None):
        """Zero-copy observation mirror (d2d_bind_host_mirror): the step kernels repeat every observation store into these
        PINNED host tensors, so `step_host` called with the same tensors copies nothing back -- only the cells a step
        changes cross PCIe.  The tensors are persistent state (read-only for the caller); all None unbinds."""
        for x in (local_map_host, yaw_host, done_host):
            if x is not None and not (torch.is_tensor(x) and x.is_pinned() and x.is_contiguous()):
                raise ValueError("bind_host_mirror needs contiguous pinned torch tensors (tensor.pin_memory())")
        def ptr(x):
            return None if x is None else C.c_void_p(x.data_ptr())
        self._check(self._lib.d2d_bind_host_mirror(self._h, ptr(local_map_host), ptr(yaw_host), ptr(done_host)),
                    "d2d_bind_host_mirror")
        self._mirror = (local_map_host, yaw_host, done_host)      # keep the buffers alive while bound
        self._mirror_ptrs = tuple(None if x is None else x.data_ptr() for x in self._mirror)

    def bind_host_io(self, actions_host=None, local_map_host=None, yaw_host=None, done_host=None):
        """Bound form of `step_host` (d2d_bind_host_io): all PINNED host tensors are given once -- the caller rewrites
        `actions_host` in place before every step and reads the three observation tensors after it -- and a step is then
        `step_bound()` or `step_pipelined()`, one C call without per-step pointer marshalling.  actions_host=None: the
        actions come from the device buffer "actions_staging".  All None unbinds."""
        for x in (actions_host, local_map_host, yaw_host, done_host):
            if x is not None and not (torch.is_tensor(x) and x.is_pinned() and x.is_contiguous()):
                raise ValueError("bind_host_io needs contiguous pinned torch tensors (tensor.pin_memory())")
        def ptr(x):
            return None if x is None else C.c_void_p(x.data_ptr())
        self._check(self._lib.d2d_bind_host_io(self._h, ptr(actions_host), ptr(local_map_host), ptr(yaw_host), ptr(done_host),
                                               self._stream()), "d2d_bind_host_io")
        self._io = (actions_host, local_map_host, yaw_host, done_host)      # keep the buffers alive while bound
        self._mirror = (local_map_host, yaw_host, done_host)
        self._mirror_ptrs = tuple(None if x is None else x.data_ptr() for x in self._mirror)
        self._step_bound = self._lib.d2d_step_bound
        self._step_pipelined = self._lib.d2d_step_pipelined
        self._hv = self._h.value

    def step_bound(self):
        """One step through the buffers bound by `bind_host_io`."""
        rc = self._step_bound(self._hv)
        if rc != 0:
            self._check(rc, "d2d_step_bound")

    def step_bound_plan_oxford(self):
        """`step_bound()` with the Oxford policy on the device (d2d_step_bound_plan_oxford): steps with the actions in
        "actions_staging", leaves the observation in the bound host buffers and the next step's actions in the staging buffer.
        Prime the first step with `plan_oxford(env.buffer("actions_staging"))`."""
        self._check(self._lib.d2d_step_bound_plan_oxford(self._h), "d2d_step_bound_plan_oxford")

    def step_pipelined(self, prelaunch_next=True):
        """One step through the bound buffers with the NEXT step's kernel pre-launched (d2d_step_pipelined): the action only
        turns the yaw at the end of a step, so the next step's action-independent work overlaps the caller's handling of this
        observation.  `prelaunch_next=True` promises another `step_pipelined` call; pass False on the last step of a run."""
        rc = self._step_pipelined(self._hv, 1 if prelaunch_next else 0)
        if rc != 0:
            self._check(rc, "d2d_step_pipelined")

    @property
    def info(self):
        """Batched counterpart of `env.info` (drone_v2.py:238-250): tensors aliasing device state."""
        b = self.buffer
        return {
            "drone_x": b("drone_x"), "drone_y": b("drone_y"), "drone_yaw": b("drone_yaw"),
            "drone_vx": b("drone_vx"), "drone_vy": b("drone_vy"),
            "state_machine": b("state_machine"), "target_x": b("target_x"), "target_y": b("target_y"),
            "collision_flag": b("collision_flag"), "dead_lock_flag": b("dead_lock_flag"),
            "freezing_flag": b("freezing_flag"), "steps": b("steps"),
            "belief": b("belief"), "hit": b("hit"),
            "tracker_buffer_count": b("tracker_buffer_count"), "tracker_buffer_ts": b("tracker_buffer_ts"),
        }

    def flight_time(self):
        return self.buffer("steps").to(torch.float64) * self.params.dt

    def set_drone_pose(self, pose):
        """Writes drone x / y / yaw for every env, as the metric scripts do on the reference object
        (script/difficulty_calculator/glob_survivability_calculator.py:36-37).  pose: [B,3] array-like (host)."""
        pose = np.ascontiguousarray(np.asarray(pose, dtype=np.float64).reshape(self.num_envs, 3))
        self._check(self._lib.d2d_set_drone_pose(self._h, pose.ctypes.data_as(C.c_void_p), self._stream()),
                    "d2d_set_drone_pose")

    # ------------------------------------------------------------------ per-env state (clone / save / load)
    @staticmethod
    def _env_indices(x):
        """int sequence, numpy array or CPU tensor -> contiguous int32 numpy array (range checks are the library's)."""
        if torch.is_tensor(x):
            if x.device.type != "cpu":
                raise ValueError("env indices must be a host sequence, numpy array or CPU tensor")
            x = x.numpy()
        a = np.asarray(x).reshape(-1)
        if a.size and a.dtype.kind not in "iu":
            raise ValueError("env indices must be integers, got %s" % a.dtype)
        a = a.astype(np.int64)
        if a.size and (a.min() < -2 ** 31 or a.max() >= 2 ** 31):
            raise _native.Drone2DNativeError("env index out of range")
        return np.ascontiguousarray(a, dtype=np.int32)

    def state_layout(self):
        """(bytes per env of a packed state row, 64-bit layout fingerprint) -- d2d_state_layout."""
        nbytes, fp = C.c_int64(), C.c_uint64()
        self._check(self._lib.d2d_state_layout(self._h, C.byref(nbytes), C.byref(fp)), "d2d_state_layout")
        return int(nbytes.value), int(fp.value)

    def clone_envs(self, src, dst):
        """Env dst[i] becomes an exact copy of env src[i], live state and reset snapshot (d2d_clone_envs, one kernel):
        with the same actions every later step, reset and policy call of dst[i] is bit-identical to src[i]'s.  src may
        repeat an env (fork it into several copies); dst must not, and no env may be in both.  The clone's reset target came
        with it, so `seeds[dst] = seeds[src]`.  Actions kept in "actions_staging" are caller data and are not copied: re-plan
        after a clone when stepping with `step_bound_plan_oxford`."""
        s, d = self._env_indices(src), self._env_indices(dst)
        if s.size != d.size:
            raise ValueError("clone_envs: %d sources for %d destinations" % (s.size, d.size))
        self._check(self._lib.d2d_clone_envs(self._h, s.ctypes.data_as(C.c_void_p), d.ctypes.data_as(C.c_void_p), int(s.size),
                                             self._stream()), "d2d_clone_envs")
        self.seeds[d] = self.seeds[s]
        if self._log_capacity and s.size:
            ws = self.buffer("world_seed")
            ws[torch.as_tensor(d.astype(np.int64), device=self.device)] = ws[torch.as_tensor(s.astype(np.int64), device=self.device)]

    def save_state(self, envs=None):
        """Packs the state of `envs` (default: all) into a uint8 CUDA tensor [count, bytes_per_env] (d2d_save_state).
        Returns {"fingerprint": int, "state": tensor, "seeds": int64 array}; the state tensor may be moved (`.cpu()`,
        `torch.save`, `.to("cuda:k")`) and is loaded with `load_state` into any env with the same fingerprint."""
        nbytes, fp = self.state_layout()
        idx = None if envs is None else self._env_indices(envs)
        count = self.num_envs if idx is None else int(idx.size)
        state = torch.zeros((count, nbytes), dtype=torch.uint8, device=self.device)
        self._check(self._lib.d2d_save_state(self._h, None if idx is None else idx.ctypes.data_as(C.c_void_p), count,
                                             C.c_void_p(state.data_ptr()), self._stream()), "d2d_save_state")
        seeds = self.seeds.copy() if idx is None else self.seeds[idx]
        return {"fingerprint": fp, "state": state, "seeds": np.asarray(seeds, dtype=np.int64)}

    def load_state(self, saved, envs=None):
        """Writes row i of `saved["state"]` into env envs[i] (default: envs 0..count-1) -- d2d_load_state.  The state must
        be a uint8 tensor [count, bytes_per_env] on this env's device; the library rejects a state of another layout
        (fingerprint).  Seeds travel with the state."""
        nbytes, _ = self.state_layout()
        state = saved["state"]
        if not torch.is_tensor(state) or state.dtype != torch.uint8 or state.dim() != 2 or state.shape[1] != nbytes:
            raise ValueError("load_state: expected a uint8 tensor [count, %d]" % nbytes)
        if state.device.type != "cuda" or state.device.index != self._dev_index:
            raise ValueError("load_state: the state is on %s, this env is on cuda:%d (move it with .to())"
                             % (state.device, self._dev_index))
        state = state.contiguous()
        count = int(state.shape[0])
        idx = None if envs is None else self._env_indices(envs)
        if idx is not None and idx.size != count:
            raise ValueError("load_state: %d rows for %d envs" % (count, idx.size))
        self._check(self._lib.d2d_load_state(self._h, None if idx is None else idx.ctypes.data_as(C.c_void_p), count,
                                             C.c_void_p(state.data_ptr()), C.c_uint64(int(saved["fingerprint"])),
                                             self._stream()), "d2d_load_state")
        if saved.get("seeds") is not None:
            envs = np.arange(count) if idx is None else idx
            self.seeds[envs] = np.asarray(saved["seeds"], dtype=np.int64)
            self._set_world_seeds(envs, self.seeds[envs])

    # ------------------------------------------------------------------ episode log + seed queue
    def _set_world_seeds(self, envs, seeds):
        """While the episode log is enabled, "world_seed" follows the seeds of reseed / clone_envs / load_state (a device
        write on the current stream, ordered with the library call it mirrors)."""
        if self._log_capacity and len(envs):
            self.buffer("world_seed")[torch.as_tensor(np.asarray(envs, dtype=np.int64), device=self.device)] = \
                torch.as_tensor(np.asarray(seeds, dtype=np.int64), device=self.device)

    def enable_episode_log(self, capacity):
        """Enables the episode log (d2d_enable_episode_log) with room for `capacity` records between two `read_episodes`
        calls: from now on every step appends, on the device, one record per env that reported done (the fields of the
        reference's experiment row).  `B * steps between reads` never drops a record.  "world_seed" is filled from
        `self.seeds`.  capacity=0 disables the log (and clears a seed queue)."""
        capacity = int(capacity)
        self._check(self._lib.d2d_enable_episode_log(self._h, capacity), "d2d_enable_episode_log")
        for name in ("episode_log", "episode_log_head", "world_seed"):
            self._views.pop(name, None)
        self._log_capacity, self._queue_set = capacity, False
        self._log_out = np.zeros(capacity, dtype=_native.EPISODE_DTYPE)
        if capacity:
            self.buffer("world_seed").copy_(torch.as_tensor(self.seeds, dtype=torch.int64))

    def read_episodes(self):
        """(records, dropped): the records written since the last read as a numpy structured array of dtype
        `_native.EPISODE_DTYPE` in (step, env) order, and how many the full log could not take (d2d_read_episode_log;
        synchronises the current stream).  While a seed queue is set, `self.seeds` is refreshed from "world_seed"."""
        if not self._log_capacity:
            raise _native.Drone2DNativeError("read_episodes: the episode log is not enabled (enable_episode_log)")
        n, dropped = C.c_int64(), C.c_int64()
        self._check(self._lib.d2d_read_episode_log(self._h, self._log_out.ctypes.data_as(C.c_void_p), C.byref(n),
                                                   C.byref(dropped), self._stream()), "d2d_read_episode_log")
        if self._queue_set:
            self.seeds[:] = self.buffer("world_seed").cpu().numpy()
        return self._log_out[:n.value].copy(), int(dropped.value)

    def set_seed_queue(self, seeds, sources=None):
        """Seeds for the envs that finish from now on (d2d_set_seed_queue): in every step each env that reports done takes
        the next one (ascending env order) and starts that world, generated on the device, at its next step; its record
        carries the seed of the world it finished.  When the queue runs out, envs replay their last world.  Needs the episode
        log and auto-reset; the world source is set up here.  With `sources` the queue holds the world keys
        world_key(sources, seeds) (d2d_set_world_queue), and the records and `seeds` carry keys.  An empty sequence clears
        the queue."""
        sd = self._keys("set_seed_queue", seeds, sources, None)
        if self._log_capacity and self.cfg.auto_reset:
            self._default_sources()
        fn, name = ((self._lib.d2d_set_seed_queue, "d2d_set_seed_queue") if sources is None else
                    (self._lib.d2d_set_world_queue, "d2d_set_world_queue"))
        self._check(fn(self._h, sd.ctypes.data_as(C.c_void_p), int(sd.size), self._stream()), name)
        self._queue_set = sd.size > 0

    def plan_oxford(self, out=None):
        """Oxford.plan for every env (yaw_planner.py:81-127): returns float64 CUDA tensor [B] of actions."""
        if out is None:
            out = torch.empty(self.num_envs, dtype=torch.float64, device=self.device)
        self._check(self._lib.d2d_plan_oxford(self._h, C.c_void_p(out.data_ptr()), self._stream()), "d2d_plan_oxford")
        return out

    def step_plan_oxford(self, actions, out=None):
        """`step(actions)` followed by `plan_oxford(out)` as ONE call (d2d_step_plan_oxford): one iteration of the reference's
        `action = policy.plan(info); ...; info = env.step(action)` loop with identical results.  Under the Primitive planner
        the step's A* searches run beside the gaze scoring of the envs that did not plan.  `out` may be `actions` (in place).
        Returns the next actions (float64 CUDA tensor [B]); observation / done are read from the buffers as after step()."""
        a = actions.to(device=self.device, dtype=torch.float64).reshape(-1).contiguous()
        if a.numel() != self.num_envs:
            raise ValueError("expected %d actions, got %d" % (self.num_envs, a.numel()))
        if out is None:
            out = torch.empty(self.num_envs, dtype=torch.float64, device=self.device)
        self._check(self._lib.d2d_step_plan_oxford(self._h, C.c_void_p(a.data_ptr()), C.c_void_p(out.data_ptr()), self._stream()),
                    "d2d_step_plan_oxford")
        return out

    def plan_gaze(self, policy, out=None):
        """NoControl / Rotating / LookAhead / LookGoal / Owl .plan for every env (yaw_planner.py), on the device.
        policy: name or d2d_gaze value.  'Oxford' is routed to plan_oxford().  'Owl' needs the env created with owl=True
        (or params.gaze_method == 'Owl')."""
        if policy == "Oxford":
            return self.plan_oxford(out)
        code = _native.GAZE[policy] if isinstance(policy, str) else int(policy)
        if out is None:
            out = torch.empty(self.num_envs, dtype=torch.float64, device=self.device)
        self._check(self._lib.d2d_plan_gaze(self._h, code, C.c_void_p(out.data_ptr()), self._stream()), "d2d_plan_gaze")
        return out

    # ------------------------------------------------------------------ rendering
    @staticmethod
    def render_layers(layers):
        """"all", an int mask of _native.RENDER_* bits, or an iterable of names ("ground_truth", "belief", "view", "plan",
        "trackers", "agents", "drone") -> int mask."""
        if isinstance(layers, str):
            if layers.lower() == "all":
                return _native.RENDER_ALL
            layers = [layers]
        if isinstance(layers, (int, np.integer)):
            return int(layers)
        mask = 0
        for name in layers:
            key = str(name).lower()
            if key not in _native.RENDER_LAYERS:
                raise ValueError("unknown render layer %r (one of %s)" % (name, ", ".join(_native.RENDER_LAYERS)))
            mask |= _native.RENDER_LAYERS[key]
        return mask

    def render(self, envs=None, pixels_per_cell=2, layers="all", out=None):
        """RGB frames of `envs` drawn on the device (d2d_render, one kernel): uint8 CUDA tensor [count, H, W, 3] with
        H = W = 50 * pixels_per_cell, in the reference's screen layout (column = x, row = y, origin top-left).
        envs: None (all), a step-1 range or an ascending contiguous list (rendered as a range), or any other sequence of
        at most 1024 env indices (repeats allowed).  layers: "all", an int mask or an iterable of layer names
        (`render_layers`).  out: a preallocated contiguous uint8 tensor of that shape on this device -- what a captured
        CUDA graph renders into.  The frames show the arena as it is: an env that just reported done shows its terminal
        state until its next step."""
        ppc = int(pixels_per_cell)
        mask = self.render_layers(layers)
        first, lst = 0, None
        if envs is None:
            count = self.num_envs
        elif isinstance(envs, range) and envs.step == 1:
            first, count = envs.start, max(0, envs.stop - envs.start)
        else:
            idx = self._env_indices(envs)
            count = int(idx.size)
            if count and np.array_equal(idx, np.arange(idx[0], idx[0] + count)):
                first = int(idx[0])
            else:
                if count > _native.RENDER_MAX_LIST:
                    raise ValueError("render: a list of %d envs (at most %d; a larger selection must be a contiguous range)"
                                     % (count, _native.RENDER_MAX_LIST))
                lst = idx
        H = 50 * ppc
        shape = (count, H, H, 3)
        if out is None:
            out = torch.empty(shape, dtype=torch.uint8, device=self.device)
        elif (not torch.is_tensor(out) or out.dtype != torch.uint8 or tuple(out.shape) != shape or not out.is_contiguous()
              or out.device.type != "cuda" or out.device.index != self._dev_index):
            raise ValueError("render: `out` must be a contiguous uint8 tensor %s on cuda:%d" % (shape, self._dev_index))
        self._check(self._lib.d2d_render(self._h, None if lst is None else lst.ctypes.data_as(C.c_void_p), int(first),
                                         int(count), ppc, int(mask), C.c_void_p(out.data_ptr() if count else 0),
                                         self._stream()), "d2d_render")
        return out

    # ------------------------------------------------------------------ difficulty metrics
    def difficulty(self, steps, grid, envs=None, slots=None, n_slots=None, collision_state=False, out=None):
        """Dynamic and static collisions of a drone held at every position of `grid`, over `steps` agent steps from each
        env's reset snapshot (d2d_difficulty, one kernel; CVM handles only).  It reads the snapshot and writes only its
        outputs, so the result does not depend on how far the envs have stepped.
        grid: (x0, y0, step, nx, ny), positions x0 + i * step, y0 + j * step.  envs: None (all) or a step-1 range.
        Returns {"first_hit": int16 [count, nx, ny] (first agent step k = 1..steps after which an agent disc grown by the
        drone radius holds the position; 0: none), "static_hit": uint8 [count, nx, ny] (collision_flag would be 1)} and,
        with collision_state=True, "collision_state": uint8 [count, nx, ny, n_slots], the array of glob_survivability:
        slot slots[k-1] is set when step k has a dynamic and no static hit.  slots: one slot per step (default: step k ->
        slot k-1; shorter tables leave the later steps unrecorded); n_slots defaults to the largest slot + 1.
        out: preallocated contiguous CUDA tensors of those shapes and dtypes, a tuple (first_hit, static_hit[,
        collision_state]) -- what a captured CUDA graph writes into."""
        first, count = 0, self.num_envs
        if envs is not None:
            if not (isinstance(envs, range) and envs.step == 1):
                raise ValueError("difficulty: envs must be None or a step-1 range")
            first, count = envs.start, max(0, envs.stop - envs.start)
        spec, n_slots = difficulty_spec(steps, grid, collision_state, slots, n_slots)
        nx, ny = spec.nx, spec.ny
        shapes = [((count, nx, ny), torch.int16), ((count, nx, ny), torch.uint8)]
        if collision_state:
            shapes.append(((count, nx, ny, n_slots), torch.uint8))
        if out is None:
            out = tuple(torch.empty(s, dtype=d, device=self.device) for s, d in shapes)
        else:
            out = tuple(out)
            if len(out) != len(shapes) or any(
                    not torch.is_tensor(t) or t.dtype != d or tuple(t.shape) != s or not t.is_contiguous() or
                    t.device.type != "cuda" or t.device.index != self._dev_index for t, (s, d) in zip(out, shapes)):
                raise ValueError("difficulty: `out` must be contiguous tensors %s on cuda:%d"
                                 % (", ".join("%s %s" % (d, s) for s, d in shapes), self._dev_index))

        def ptr(t):
            return C.c_void_p(t.data_ptr() if count else 0)
        self._check(self._lib.d2d_difficulty(self._h, C.byref(spec), int(first), int(count), ptr(out[0]), ptr(out[1]),
                                             ptr(out[2]) if collision_state else None, self._stream()), "d2d_difficulty")
        res = {"first_hit": out[0], "static_hit": out[1]}
        if collision_state:
            res["collision_state"] = out[2]
        return res

    def stats(self, reset=False):
        """Episode statistics accumulated on device (int64 [16], names in _native.STAT_NAMES)."""
        out = np.zeros(_native.NUM_STATS, dtype=np.int64)
        self._check(self._lib.d2d_stats(self._h, out.ctypes.data_as(C.c_void_p), 1 if reset else 0, self._stream()),
                    "d2d_stats")
        return out

    def launch_count(self):
        return int(self._lib.d2d_launch_count(self._h))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._views = {}
            self._lib.d2d_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def difficulty_spec(steps, grid, collision_state=False, slots=None, n_slots=None):
    """The d2d_difficulty_spec of `Drone2DVecEnv.difficulty` and its number of collision_state slots (0 without
    collision_state)."""
    x0, y0, step, nx, ny = grid
    spec = _native.D2DDifficultySpec()
    spec.struct_size = C.sizeof(_native.D2DDifficultySpec)
    spec.nx, spec.ny = int(nx), int(ny)
    spec.x0, spec.y0, spec.step = float(x0), float(y0), float(step)
    spec.steps = int(steps)
    if not 1 <= spec.steps <= _native.DIFF_MAX_STEPS:
        raise ValueError("difficulty: steps %d outside 1..%d" % (spec.steps, _native.DIFF_MAX_STEPS))
    if not collision_state:
        return spec, 0
    table = list(range(spec.steps)) if slots is None else [int(s) for s in slots]
    if len(table) > spec.steps:
        raise ValueError("difficulty: %d slots for %d steps" % (len(table), spec.steps))
    if any(s < 0 or s >= _native.DIFF_NO_SLOT for s in table):
        raise ValueError("difficulty: slot indices must lie in [0, %d)" % _native.DIFF_NO_SLOT)
    n = int(n_slots) if n_slots is not None else (max(table) + 1 if table else 0)
    if n < 1:
        raise ValueError("difficulty: collision_state needs at least one slot")
    table += [_native.DIFF_NO_SLOT] * (spec.steps - len(table))
    spec.n_slots = n
    spec.slot[:spec.steps] = table
    return spec, n


def trajectory_waypoints(cfg, coeff, nseg, cursor):
    """Host-side expansion of one env's stored A* segments into the reference's waypoint lists
    (Trajectory2D.positions / .velocities, traj_planner.py:208-217) from `cursor` on.
    coeff: [D2D_MAX_SEGMENTS, 6] array, nseg / cursor ints.  Returns (positions [L,2], velocities [L,2])."""
    import ctypes as _C  # noqa: F401
    n_way = cfg.n_way
    pos, vel = [], []
    for a in range(int(cursor), int(nseg) * n_way):
        seg, ws = divmod(a, n_way)
        ti = n_way - 1 - ws
        t, t2, tt = cfg.t_way[ti], cfg.t_way2[ti], cfg.t_way_x2[ti]
        c = coeff[seg]
        # np.array([1, t, t**2]) @ coeff.T on the reference image == fma(t2, h, p + t*v); np.around
        px = np.rint(_fma(t2, c[2], c[0] + t * c[1]))
        py = np.rint(_fma(t2, c[5], c[3] + t * c[4]))
        pos.append((px, py))
        vel.append((c[1] + tt * c[2], c[4] + tt * c[5]))
    return np.array(pos, dtype=np.float64).reshape(-1, 2), np.array(vel, dtype=np.float64).reshape(-1, 2)


_libm = None


def _fma(a, b, c):
    global _libm
    if _libm is None:
        import ctypes.util
        _libm = C.CDLL(ctypes.util.find_library("m") or "libm.so.6")
        _libm.fma.restype = C.c_double
        _libm.fma.argtypes = [C.c_double] * 3
    return _libm.fma(float(a), float(b), float(c))
