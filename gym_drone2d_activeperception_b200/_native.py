"""ctypes binding of libdrone2d.so (include/drone2d.h).  There is NO fallback: if the CUDA library is missing or
a call fails, an exception is raised."""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("D2D_LIB") or os.path.join(HERE, "libdrone2d.so")     # D2D_LIB: an A/B build of the same ABI (tools/)

MAX_TARGETS, MAX_U, MAX_SAMP, MAX_WAY, MAX_YAW = 8, 64, 32, 64, 16
NUM_STATS = 16
GAZE = {"NoControl": 0, "Rotating": 1, "LookAhead": 2, "LookGoal": 3, "Owl": 4}
POLICY_OXFORD, POLICY_OWL, MAX_OWL_U = 1, 2, 32
BELIEF_STRIDE = 2560
STAT_NAMES = ["env_steps", "episodes", "success", "static_collision", "dynamic_collision", "freezing", "dead_lock",
              "flight_steps", "grid_discovered", "agents_tracked", "tracked_steps", "plans", "plan_failures", "replans",
              "mirror_bytes", "plan_overflows"]


class D2DConfig(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int32), ("device", C.c_int32), ("num_envs", C.c_int32), ("num_agents", C.c_int32),
        ("planner", C.c_int32), ("trackers", C.c_int32), ("auto_reset", C.c_int32), ("oxford", C.c_int32),
        ("envs_per_block", C.c_int32), ("n_rays", C.c_int32), ("n_targets", C.c_int32),
        ("n_u", C.c_int32), ("n_samp", C.c_int32), ("n_way", C.c_int32), ("n_yaw", C.c_int32), ("motion_profile", C.c_int32),
        ("dt", C.c_double), ("map_scale", C.c_double), ("map_w", C.c_double), ("map_h", C.c_double),
        ("agent_radius", C.c_double),
        ("drone_max_acceleration", C.c_double), ("drone_radius", C.c_double), ("drone_max_yaw_speed", C.c_double),
        ("drone_view_depth", C.c_double), ("drone_view_range", C.c_double), ("max_flight_time", C.c_double),
        ("var_cam", C.c_double), ("drone_max_speed", C.c_double), ("ox_cos_thresh", C.c_double),
        ("targets", (C.c_double * 2) * MAX_TARGETS),
        ("u_space", C.c_double * MAX_U),
        ("t_samp", C.c_double * MAX_SAMP), ("t_samp2", C.c_double * MAX_SAMP),
        ("t_way", C.c_double * MAX_WAY), ("t_way2", C.c_double * MAX_WAY), ("t_way_x2", C.c_double * MAX_WAY),
        ("v_yaw_space", C.c_double * MAX_YAW),
        ("n_owl_u", C.c_int32), ("owl_repeat", C.c_int32), ("owl_u_space", C.c_double * MAX_OWL_U),
    ]


JERK_H, JERK_MAXT = 72, 40


class D2DJerkTables(C.Structure):
    _fields_ = [
        ("dx", C.c_double * JERK_H), ("dy", C.c_double * JERK_H),
        ("T", C.c_double * JERK_H), ("Tp", (C.c_double * 4) * JERK_H),
        ("times", C.c_int32 * JERK_H),
        ("tt", (C.c_double * JERK_MAXT) * JERK_H), ("ttp", ((C.c_double * 4) * JERK_MAXT) * JERK_H),
        ("tie_order", (C.c_uint8 * JERK_H) * 144),
    ]


WORLD_MAX_RANDOM, WORLD_MAX_PILLARS, WORLD_GROUPS = 256, 64, 100
WORLD_EAGER, WORLD_LAZY = 1, 2
WORLD_MAX_SOURCES = 4096                # world sources of one handle (d2d_set_world_sources); key = source * 2**32 + seed

# d2d_render: frame layers (drone2d.h D2D_RENDER_*), drawn back to front in this order
RENDER_MAX_PPC, RENDER_MAX_LIST = 10, 1024
RENDER_GROUND_TRUTH, RENDER_BELIEF, RENDER_VIEW, RENDER_PLAN = 1, 2, 4, 8
RENDER_TRACKERS, RENDER_AGENTS, RENDER_DRONE, RENDER_ALL = 16, 32, 64, 127
RENDER_LAYERS = {"ground_truth": RENDER_GROUND_TRUTH, "belief": RENDER_BELIEF, "view": RENDER_VIEW, "plan": RENDER_PLAN,
                 "trackers": RENDER_TRACKERS, "agents": RENDER_AGENTS, "drone": RENDER_DRONE}


# d2d_difficulty: position grid and step limits, and the slot-table entry of a step that collision_state does not record
DIFF_MAX_POS, DIFF_MAX_STEPS, DIFF_NO_SLOT = 1024, 1024, 0xFFFF


class D2DDifficultySpec(C.Structure):
    _fields_ = [("struct_size", C.c_int32), ("nx", C.c_int32), ("ny", C.c_int32),
                ("x0", C.c_double), ("y0", C.c_double), ("step", C.c_double),
                ("steps", C.c_int32), ("n_slots", C.c_int32), ("slot", C.c_uint16 * DIFF_MAX_STEPS)]


class D2DWorldSource(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int32), ("agent_number", C.c_int32), ("pillar_number", C.c_int32), ("pad_", C.c_int32),
        ("agent_radius", C.c_double), ("agent_max_speed", C.c_double), ("drone_radius", C.c_double),
        ("init_x", C.c_double), ("init_y", C.c_double), ("map_w", C.c_double), ("map_h", C.c_double),
        ("headings", (C.c_double * 2) * WORLD_MAX_RANDOM),
        ("static_map", (C.c_uint8 * 50) * 50),
    ]


class D2DEpisodeRecord(C.Structure):
    """d2d_episode_record (drone2d.h): one finished episode of the episode log."""
    _fields_ = [("seed", C.c_int64), ("step", C.c_int64), ("tracked_steps", C.c_int64), ("env", C.c_int32),
                ("steps", C.c_int32), ("grid_discovered", C.c_int32), ("trackers", C.c_int32),
                ("state_machine", C.c_uint8), ("collision_flag", C.c_uint8), ("freezing_flag", C.c_uint8),
                ("dead_lock_flag", C.c_uint8), ("reserved", C.c_int32)]


# the same record as a numpy structured dtype (what Drone2DVecEnv.read_episodes returns)
EPISODE_DTYPE = np.dtype({"names": [f[0] for f in D2DEpisodeRecord._fields_],
                          "formats": ["<i8", "<i8", "<i8", "<i4", "<i4", "<i4", "<i4", "u1", "u1", "u1", "u1", "<i4"],
                          "offsets": [getattr(D2DEpisodeRecord, f[0]).offset for f in D2DEpisodeRecord._fields_],
                          "itemsize": C.sizeof(D2DEpisodeRecord)})


class D2DBufferInfo(C.Structure):
    _fields_ = [("dev_ptr", C.c_void_p), ("nbytes", C.c_int64), ("dtype", C.c_int32), ("ndim", C.c_int32),
                ("shape", C.c_int64 * 4), ("strides", C.c_int64 * 4)]


EXPORTS = ["d2d_version", "d2d_last_error", "d2d_create", "d2d_destroy", "d2d_set_world", "d2d_set_rng", "d2d_set_rvo", "d2d_set_jerk_tables", "d2d_reset", "d2d_request_reset", "d2d_step", "d2d_rollout",
           "d2d_step_host", "d2d_bind_host_mirror", "d2d_bind_host_io", "d2d_step_bound", "d2d_step_pipelined", "d2d_plan_oxford", "d2d_step_plan_oxford", "d2d_step_bound_plan_oxford", "d2d_plan_gaze", "d2d_set_drone_pose", "d2d_get_buffer", "d2d_stats",
           "d2d_launch_count", "d2d_clone_envs", "d2d_state_layout", "d2d_save_state", "d2d_load_state",
           "d2d_set_world_source", "d2d_generate_worlds", "d2d_enable_episode_log", "d2d_read_episode_log",
           "d2d_set_seed_queue", "d2d_render", "d2d_difficulty", "d2d_set_world_sources", "d2d_generate_worlds_keyed",
           "d2d_set_world_queue", "d2d_grid_hits"]

_lib = None


class Drone2DNativeError(RuntimeError):
    pass


def load():
    """Loads libdrone2d.so; raises if it has not been built (python -m gym_drone2d_activeperception_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise Drone2DNativeError(
            "libdrone2d.so not found at %s -- build it with `python -m gym_drone2d_activeperception_b200.build` "
            "(there is no CPU fallback)" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    L.d2d_version.restype = C.c_int
    L.d2d_last_error.restype = C.c_char_p
    L.d2d_last_error.argtypes = [vp]
    L.d2d_create.argtypes = [C.POINTER(D2DConfig), C.POINTER(vp)]
    L.d2d_destroy.argtypes = [vp]
    L.d2d_set_world.argtypes = [vp, C.c_int32, C.c_int32, vp, vp, vp, vp, vp, vp]
    L.d2d_set_rng.argtypes = [vp, C.c_int32, C.c_int32, vp, vp, vp, vp]
    L.d2d_set_rvo.argtypes = [vp, C.c_int32, C.c_int32, vp, vp, vp, C.c_int32]
    L.d2d_set_jerk_tables.argtypes = [vp, C.POINTER(D2DJerkTables)]
    L.d2d_reset.argtypes = [vp, vp, vp]
    L.d2d_request_reset.argtypes = [vp, vp, vp]
    L.d2d_step.argtypes = [vp, vp, vp]
    L.d2d_rollout.argtypes = [vp, vp, C.c_int32, C.c_int64, vp]
    L.d2d_step_host.argtypes = [vp, vp, vp, vp, vp, vp]
    L.d2d_bind_host_mirror.argtypes = [vp, vp, vp, vp]
    L.d2d_bind_host_io.argtypes = [vp, vp, vp, vp, vp, vp]
    L.d2d_step_bound.argtypes = [vp]
    L.d2d_step_pipelined.argtypes = [vp, C.c_int32]
    L.d2d_plan_oxford.argtypes = [vp, vp, vp]
    L.d2d_step_plan_oxford.argtypes = [vp, vp, vp, vp]
    L.d2d_step_bound_plan_oxford.argtypes = [vp]
    L.d2d_plan_gaze.argtypes = [vp, C.c_int32, vp, vp]
    L.d2d_set_drone_pose.argtypes = [vp, vp, vp]
    L.d2d_get_buffer.argtypes = [vp, C.c_char_p, C.POINTER(D2DBufferInfo)]
    L.d2d_stats.argtypes = [vp, vp, C.c_int32, vp]
    L.d2d_launch_count.argtypes = [vp]
    L.d2d_launch_count.restype = C.c_int64
    L.d2d_clone_envs.argtypes = [vp, vp, vp, C.c_int32, vp]
    L.d2d_state_layout.argtypes = [vp, C.POINTER(C.c_int64), C.POINTER(C.c_uint64)]
    L.d2d_save_state.argtypes = [vp, vp, C.c_int32, vp, vp]
    L.d2d_load_state.argtypes = [vp, vp, C.c_int32, vp, C.c_uint64, vp]
    L.d2d_set_world_source.argtypes = [vp, C.POINTER(D2DWorldSource)]
    L.d2d_generate_worlds.argtypes = [vp, vp, vp, C.c_int32, C.c_int32, vp]
    L.d2d_enable_episode_log.argtypes = [vp, C.c_int64]
    L.d2d_read_episode_log.argtypes = [vp, vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64), vp]
    L.d2d_set_seed_queue.argtypes = [vp, vp, C.c_int64, vp]
    L.d2d_set_world_sources.argtypes = [vp, vp, C.c_int32]
    L.d2d_generate_worlds_keyed.argtypes = [vp, vp, vp, C.c_int32, C.c_int32, vp]
    L.d2d_set_world_queue.argtypes = [vp, vp, C.c_int64, vp]
    L.d2d_render.argtypes = [vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, vp, vp]
    L.d2d_difficulty.argtypes = [vp, C.POINTER(D2DDifficultySpec), C.c_int32, C.c_int32, vp, vp, vp, vp]
    L.d2d_grid_hits.argtypes = [vp, C.POINTER(D2DDifficultySpec), C.c_int32, C.c_int32, C.c_int32, vp, vp, vp, vp]
    for name in EXPORTS:
        if name not in ("d2d_version", "d2d_last_error", "d2d_launch_count"):
            getattr(L, name).restype = C.c_int
    _lib = L
    return L


def check(handle, rc, what):
    if rc != 0:
        msg = load().d2d_last_error(handle)
        raise Drone2DNativeError("%s failed (%d): %s" % (what, rc, msg.decode() if msg else "?"))
