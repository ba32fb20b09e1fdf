/*
 * drone2d.h -- C ABI of libdrone2d.so: the B200-native batched replacement for the per-step hot path of
 * smoggy-P/gym-Drone2D-ActivePerception.
 *
 * The reference has no FFI layer; its boundary for this path is the gym 0.21 Env protocol of
 * `Drone2DEnv2` (envs/drone_v2.py:69 __init__, :152 step, :259 reset) plus the `env.info` dict its callers
 * read (experiment.py:69-101, yaw_planner.py:81-127).  Each entry point below names the reference interface
 * it replaces.  All functions return 0 on success or a negative d2d_status; no C++ exception crosses the
 * ABI; d2d_last_error() gives the message.  A handle is bound to one CUDA device and is not thread-safe;
 * distinct handles (one per GPU / process) are independent.  All work is enqueued on the caller's stream
 * (a `cudaStream_t` passed as void*, NULL = legacy default stream); only the *_host variants and d2d_stats
 * synchronise that stream.
 *
 * Memory: the library owns one device arena per handle (state for `num_envs` environments, laid out env-major:
 * per-agent arrays, one belief grid and ground-truth bitmap per env, and one 128-byte record per env with the
 * drone / bookkeeping scalars, so the warp that owns an env streams its state with coalesced / bulk copies).
 * d2d_get_buffer() exposes every state and observation array as a raw device pointer + shape/strides so the
 * host language can wrap them zero-copy (the Python host wraps them as torch tensors).
 */
#ifndef DRONE2D_H
#define DRONE2D_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define D2D_VERSION 100          /* 0.1.0 */
#define D2D_MAX_TARGETS 8
#define D2D_MAX_U 64
#define D2D_MAX_SAMP 32
#define D2D_MAX_WAY 64
#define D2D_MAX_YAW 16
#define D2D_MAX_SEGMENTS 100     /* Primitive.plan stops after 99 expansions (traj_planner.py:149) */
#define D2D_BELIEF_STRIDE 2560   /* bytes per env of the belief grid buffer (50*50 used, 128-B aligned rows) */
#define D2D_NUM_STATS 16

typedef enum d2d_status {
    D2D_OK = 0,
    D2D_ERR_INVALID = -1,        /* bad argument / unsupported configuration */
    D2D_ERR_CUDA = -2,           /* a CUDA runtime call failed (see d2d_last_error) */
    D2D_ERR_NOMEM = -3,
    D2D_ERR_STATE = -4           /* call sequence error, e.g. step before set_world */
} d2d_status;

typedef enum d2d_planner {
    D2D_PLANNER_NOMOVE = 0,      /* traj_planner.py:68-76 */
    D2D_PLANNER_PRIMITIVE = 1,   /* traj_planner.py:80-233 */
    D2D_PLANNER_JERK = 2         /* Jerk_Primitive, traj_planner.py:403-516; needs d2d_set_jerk_tables */
} d2d_planner;

/* params.motion_profile: constant-velocity agents (velocity IS pref_velocity) or reciprocal velocity obstacles */
typedef enum d2d_motion { D2D_MOTION_CVM = 0, D2D_MOTION_RVO = 1 } d2d_motion;

/* gaze policies of yaw_planner.py that d2d_plan_gaze evaluates for every env (Oxford has its own entry point) */
typedef enum d2d_gaze {
    D2D_GAZE_NOCONTROL = 0, D2D_GAZE_ROTATING = 1, D2D_GAZE_LOOKAHEAD = 2, D2D_GAZE_LOOKGOAL = 3,
    D2D_GAZE_OWL = 4             /* stateful (yaw_planner.py:151-222): needs cfg.oxford & D2D_POLICY_OWL */
} d2d_gaze;

/* bits of d2d_config.oxford: which gaze-policy state lives in the arena */
#define D2D_POLICY_OXFORD 1      /* Oxford.last_time_observed_map (yaw_planner.py:49-50) */
#define D2D_POLICY_OWL 2         /* Owl.U_list + the repeated-action queue (yaw_planner.py:160-172) */
#define D2D_MAX_OWL_U 32

typedef enum d2d_dtype { D2D_U8 = 0, D2D_I8 = 1, D2D_I32 = 2, D2D_I64 = 3, D2D_F32 = 4, D2D_F64 = 5 } d2d_dtype;

/* indices into the statistics vector (episode totals, experiment.py:76-101 CSV columns) */
enum {
    D2D_STAT_ENV_STEPS = 0, D2D_STAT_EPISODES, D2D_STAT_SUCCESS, D2D_STAT_STATIC_COLLISION,
    D2D_STAT_DYNAMIC_COLLISION, D2D_STAT_FREEZING, D2D_STAT_DEAD_LOCK, D2D_STAT_FLIGHT_STEPS,
    D2D_STAT_GRID_DISCOVERED, D2D_STAT_AGENTS_TRACKED, D2D_STAT_TRACKED_STEPS, D2D_STAT_PLANS,
    D2D_STAT_PLAN_FAILURES, D2D_STAT_REPLANS,
    D2D_STAT_MIRROR_BYTES,       /* local_map bytes stored into the host mirror (d2d_bind_host_mirror) */
    D2D_STAT_PLAN_OVERFLOWS      /* A* searches that outgrew the small-footprint kernel and were redone by the large one */
};

/* Mirrors the reference `Params` object (utils.py:65-106) plus the batch shape.  The lookup tables are the
 * reference's own numpy expressions, evaluated by the host (traj_planner.py:98-104,180,212; yaw_planner.py:65)
 * so that np.arange's element values are reproduced exactly. */
typedef struct d2d_config {
    int32_t struct_size;             /* sizeof(d2d_config), ABI check */
    int32_t device;                  /* CUDA device ordinal */
    int32_t num_envs;                /* B */
    int32_t num_agents;              /* N = agent_number + nnz(static_map) (drone_v2.py:28-66) */
    int32_t planner;                 /* d2d_planner */
    int32_t trackers;                /* 1: run the Kalman trackers (utils.py:242-275) every step, as the reference does */
    int32_t auto_reset;              /* 1: an env that reported done is re-initialised at the start of its next step */
    int32_t oxford;                  /* D2D_POLICY_* bits: gaze-policy state to allocate (1 = Oxford, as before) */
    int32_t envs_per_block;          /* 0 = library default; tuning knob (4, 8 or 16) */
    int32_t n_rays;                  /* ceil(map_size[0] / strip_width), utils.py:587 */
    int32_t n_targets;
    int32_t n_u, n_samp, n_way, n_yaw;
    int32_t motion_profile;          /* d2d_motion: how the agents move (params.motion_profile, drone_v2.py:169-179) */
    double dt, map_scale, map_w, map_h;
    double agent_radius;             /* params.agent_radius */
    double drone_max_acceleration, drone_radius, drone_max_yaw_speed;
    double drone_view_depth, drone_view_range, max_flight_time, var_cam, drone_max_speed;
    double ox_cos_thresh;            /* min{c : np.arccos(c) <= radians(view_range/2)} (host bisection) */
    double targets[D2D_MAX_TARGETS][2];
    double u_space[D2D_MAX_U];
    double t_samp[D2D_MAX_SAMP], t_samp2[D2D_MAX_SAMP];
    double t_way[D2D_MAX_WAY], t_way2[D2D_MAX_WAY], t_way_x2[D2D_MAX_WAY];
    double v_yaw_space[D2D_MAX_YAW];
    /* Owl (yaw_planner.py:151-172): u_space = np.arange(-max_yaw_speed, max_yaw_speed, max_yaw_speed / 10) evaluated by the
     * host, and how often a chosen action is repeated: int(0.8 // params.dt) - 1 (yaw_planner.py:220-221) */
    int32_t n_owl_u, owl_repeat;
    double owl_u_space[D2D_MAX_OWL_U];
} d2d_config;

/* Jerk_Primitive (traj_planner.py:403-516): constants of the 72 candidate headings np.arange(0, 360, 5), evaluated by the host
 * with the reference's own numpy expressions (np.cos / np.sin of math.radians, numpy-scalar `**`, np.arange, np.floor), and
 * the heading order `cost[:, 0].argsort()` produces for the goal bearings where the cost ties. */
#define D2D_JERK_H 72
#define D2D_JERK_MAXT 40
typedef struct d2d_jerk_tables {
    double dx[D2D_JERK_H], dy[D2D_JERK_H];            /* d * np.cos(radians(theta)), d * np.sin(radians(theta)), d = 30 (:409, 414-415) */
    double T[D2D_JERK_H], Tp[D2D_JERK_H][4];          /* T (:429-432) and T**2 .. T**5 */
    int32_t times[D2D_JERK_H];                        /* int(np.floor(T / dt)) (:434) */
    double tt[D2D_JERK_H][D2D_JERK_MAXT];             /* np.arange(dt, times*dt + dt, dt)[:times] (:438) */
    double ttp[D2D_JERK_H][D2D_JERK_MAXT][4];         /* tt**2 .. tt**5 */
    /* cost[:, 0].argsort() (:478) of the host's numpy for goal bearings phi_h % 360 == 2.5 * m, m = 0..143: the cost is
     * symmetric about the bearing there, pairs of headings tie, and numpy's default argsort is unstable -- the order is
     * recorded from the library.  Any other bearing has distinct costs (ascending order is unique). */
    uint8_t tie_order[144][D2D_JERK_H];
} d2d_jerk_tables;

typedef struct d2d_handle d2d_handle;

typedef struct d2d_buffer_info {
    void *dev_ptr;
    int64_t nbytes;
    int32_t dtype;                   /* d2d_dtype */
    int32_t ndim;
    int64_t shape[4];
    int64_t strides[4];              /* in elements */
} d2d_buffer_info;

int d2d_version(void);
const char *d2d_last_error(const d2d_handle *h);   /* h may be NULL: error of the last failed d2d_create */

/* Replaces Drone2DEnv2.__init__ (drone_v2.py:69-149) minus world generation: allocates the arena. */
int d2d_create(const d2d_config *cfg, d2d_handle **out);
int d2d_destroy(d2d_handle *h);

/* Replaces the state produced by init_obstacles_random_size + OccupancyGridMap.init_obstacles
 * (drone_v2.py:12-66, utils.py:508-525) for envs [first_env, first_env+count): HOST arrays, env-major.
 *   agent_pos, agent_pref : [count][N][2] f64     agent_radius, tracker_radius : [count][N] f64
 *   gt_grid : [count][gw][gh] u8 ground-truth grid (only cells == 1 are occupancy; utils.py:666,770)
 *   drone_pose : [count][3] f64 (x, y, yaw degrees)
 * Stores the data as the per-env reset snapshot and resets those envs (reset() == __init__, drone_v2.py:259). */
int d2d_set_world(d2d_handle *h, int32_t first_env, int32_t count, const double *agent_pos, const double *agent_pref,
                  const double *agent_radius, const double *tracker_radius, const uint8_t *gt_grid,
                  const double *drone_pose);

/* Required once when cfg.planner = D2D_PLANNER_JERK (before the first step): the per-heading tables above (HOST). */
int d2d_set_jerk_tables(d2d_handle *h, const d2d_jerk_tables *tables);

/* State of the reference's global legacy `np.random` stream right after world generation (np.random.seed(map_id),
 * drone_v2.py:80, then the 100 heading draws, :54), as returned by RandomState.get_state(): key [count][624] u32, pos,
 * has_gauss, cached_gaussian per env (HOST).  Needed only when var_cam != 0: the per-step measurement noise
 * `sigma * np.random.randn(2)` (utils.py:605) continues this stream; reset() restores it. */
int d2d_set_rng(d2d_handle *h, int32_t first_env, int32_t count, const uint32_t *key, const int32_t *pos,
                const int32_t *has_gauss, const double *gauss);

/* Needed when cfg.motion_profile = D2D_MOTION_RVO (RVO.RVO_update, utils.py:299-357, called at drone_v2.py:169-175): the
 * agents' initial velocities (drone_v2.py:19 `(0., 0.)` for the random agents, :62 the group velocity for map-cell agents)
 * and the circular obstacles of init_obstacles_random_size (drone_v2.py:14-27), HOST arrays:
 *   agent_vel [count][N][2] f64, obstacles [count][max_obstacles][3] f64 (x, y, rad), num_obstacles [count] i32 (<= 16).
 * Stored as part of the reset snapshot.  The step then runs d2d_rvo_kernel before Agent.step; atan2 / asin / sin / cos of
 * run-time values are CUDA's, so agent state matches the reference to 1e-9 rather than bit for bit under this profile. */
int d2d_set_rvo(d2d_handle *h, int32_t first_env, int32_t count, const double *agent_vel, const double *obstacles,
                const int32_t *num_obstacles, int32_t max_obstacles);

/* Replaces Drone2DEnv2.reset() (drone_v2.py:259-261) for every env whose mask byte is non-zero
 * (mask_dev == NULL: all).  mask_dev is a DEVICE pointer to num_envs bytes. */
int d2d_reset(d2d_handle *h, const uint8_t *mask_dev, void *stream);

/* Lazy form of d2d_reset: marks the selected envs (EnvRec::pending_reset); each is re-initialised from its snapshot at the
 * START of its next step -- the path auto_reset takes for an env that returned done -- inside the step kernel, without the
 * separate reset kernel and without touching the observation until then (a gaze policy called in between sees the env as
 * freshly reset, as it does after done).  After that step the state equals d2d_reset + the same step. */
int d2d_request_reset(d2d_handle *h, const uint8_t *mask_dev, void *stream);

/* Replaces Drone2DEnv2.step(a) (drone_v2.py:152-257) for all envs.  actions_dev: DEVICE [num_envs] f64 in [-1, 1].
 * Results land in the buffers "local_map", "yaw_angle", "done", "collision_flag", ... (d2d_get_buffer). */
int d2d_step(d2d_handle *h, const double *actions_dev, void *stream);

/* K consecutive steps in ONE launch (replaces the `for t in range(K): env.step(a[t])` loop of experiment.py:65-70 when the
 * actions of the K steps are known up front -- scripted / constant gaze -- or were produced on the device).
 * actions_dev: DEVICE f64, action of env e at step t = actions_dev[t * action_stride + e] (action_stride >= num_envs, or 0:
 * the same [num_envs] vector every step).  Every warp walks ITS env through the K steps with the env's working set resident
 * in shared memory (fetched from HBM once, not once per step) and never waits for the other envs between steps.  All buffers
 * and statistics end up bit-identical to K d2d_step calls; the per-step outputs ("done", "local_map", ...) hold the LAST
 * step's values.  Batches above two waves of warps (8288 envs on a 148-SM GPU) are stepped by K per-step launches instead
 * (the per-step kernel's small blocks keep a large batch's SMs busier; same results).  NoMove planner, CVM motion profile,
 * default warp kernels (envs_per_block <= 0) only: everything else returns D2D_ERR_INVALID (those steps consist of several
 * dependent launches; call d2d_step). */
int d2d_rollout(d2d_handle *h, const double *actions_dev, int32_t num_steps, int64_t action_stride, void *stream);

/* Same step with HOST buffers (the call an FFI user makes): gets the actions to the device (pinned memory is read by
 * the kernels directly over PCIe, pageable memory is copied first), steps, copies the observation back and
 * synchronises.  Any output pointer may be NULL.  actions_host == NULL: the actions are taken from the device buffer
 * "actions_staging" (d2d_get_buffer), e.g. written there by d2d_plan_oxford / d2d_plan_gaze.
 *   local_map_host [num_envs][1][L][L] u8, yaw_host [num_envs] f32, done_host [num_envs] u8 */
int d2d_step_host(d2d_handle *h, const double *actions_host, uint8_t *local_map_host, float *yaw_host,
                  uint8_t *done_host, void *stream);

/* Zero-copy observation mirror for d2d_step_host.  The reference hands its caller a NEW observation dict every step
 * (drone_v2.py:251-255); over PCIe that is 1089 B per env per step although a step changes only a few cells of the
 * window.  After this call the step kernels repeat every store to "local_map" / "yaw_angle" / "done" into the given
 * PINNED host buffers (cudaHostAlloc / cudaHostRegister / torch pin_memory; device-mapped, local_map_host 4-byte
 * aligned), so a d2d_step_host call that is passed the same pointers copies nothing back: only changed cells (or a whole
 * window when the drone's cell changed / the env was reset) cross the bus.  The buffers are persistent state: the
 * caller may read them between steps but must not modify them, and must keep them alive until they are unbound
 * (all NULL) or the handle is destroyed.  Any pointer may be NULL (that output is then copied as before).  The first
 * d2d_step_host after a bind, d2d_reset or d2d_set_world refreshes the mirror with one full copy. */
int d2d_bind_host_mirror(d2d_handle *h, uint8_t *local_map_host, float *yaw_host, uint8_t *done_host);

/* Bound form of d2d_step_host for callers that step in a tight loop (a vectorised-env worker): all host buffers and the
 * stream are given ONCE, a step is then d2d_step_bound(h) or d2d_step_pipelined(h, more).
 *   actions_host  PINNED [num_envs] f64 the caller rewrites before every step (read by the kernels in place over PCIe);
 *                 NULL: actions come from the device buffer "actions_staging" (policy on the GPU)
 *   local_map_host / yaw_host / done_host  PINNED, become the zero-copy observation mirror (d2d_bind_host_mirror rules)
 * Binding with all pointers NULL unbinds. */
int d2d_bind_host_io(d2d_handle *h, const double *actions_host, uint8_t *local_map_host, float *yaw_host, uint8_t *done_host,
                     void *stream);

/* One step through the bound buffers: d2d_step_host without per-call pointer resolution. */
int d2d_step_bound(d2d_handle *h);

/* The same step, pipelined.  In Drone2DEnv2.step the action only turns the yaw at the very END of the step (step_yaw,
 * utils.py:741-743, called at drone_v2.py:214); agent motion, ray casting, trackers, collision tests and the done logic
 * never see it.  prelaunch_next != 0 promises that another d2d_step_pipelined call follows; the library then starts the
 * FOLLOWING step before this call returns: everything of it that does not depend on its action runs while the caller is
 * still looking at this step's observation and choosing the next actions, and stops at a gate just before the yaw update.
 * The next d2d_step_pipelined call publishes the actions (the caller has written them into the bound pinned buffer) and
 * opens the gate.  Host-mirror stores of a step are issued only behind its gate, so the observation buffers stay valid
 * until the next call, as with d2d_step_host.  Results are identical to d2d_step_bound.
 *   Batches of at most one wave of warps (4116 envs on a 148-SM B200): ONE resident kernel serves the whole run of calls.
 *     Each env's working set stays in shared memory between steps; a courier block on the one SM that holds no env polls a
 *     stamp word in pinned host memory and pulls the step's actions out of the bound buffer itself, so the host's part of a
 *     step is one store (no launch, no copy, no stream synchronisation); completion of a step is a pinned word the last
 *     block writes after the step's single system-scope fence, and the call polls it.  4117 .. 4144 envs fill every SM: same
 *     kernel, actions delivered by one async copy per step instead of the courier.
 *   Larger batches (up to ~16k envs): one kernel per step, launched behind the current one (the round-1 design).
 *   Planners other than NoMove, the RVO profile, actions taken from "actions_staging" and batches above ~16k envs (whose
 *     step dwarfs the latency being hidden) run synchronously (same results, nothing started ahead).
 * Contract: until the call that passes prelaunch_next = 0 (the last step of a run) every other entry point of this handle
 * returns D2D_ERR_STATE, and the kernel that waits for the next actions OWNS the GPU: work queued on the same device in
 * between (a policy network, a cudaDeviceSynchronize) waits for it.  This entry point is meant for HOST policies; a policy
 * on the GPU calls d2d_step / d2d_rollout with device actions, which needs no host round trip in the first place.  A
 * kernel whose actions never arrive gives up after ~2 s and the next call reports it; d2d_destroy and re-binding release
 * a waiting kernel (it completes its step with action 0). */
int d2d_step_pipelined(d2d_handle *h, int32_t prelaunch_next);

/* Replaces Oxford.plan(env.info) (yaw_planner.py:81-127) for all envs: writes the chosen action per env to
 * actions_out_dev (DEVICE [num_envs] f64) and advances the policy state.  Requires cfg.oxford = 1. */
int d2d_plan_oxford(d2d_handle *h, double *actions_out_dev, void *stream);

/* d2d_step(actions_dev) followed by d2d_plan_oxford(next_actions_dev) -- one iteration of the reference's loop
 * `action = policy.plan(info); _, _, done, info = env.step(action)` (main.py / experiment.py:33-36) as ONE call, with the same
 * results as the two calls.  Under the Primitive planner the A* searches of the step (a latency chain that leaves most of every
 * SM idle) and the completion of the envs that planned run on an internal side stream while `stream` already scores the gaze
 * candidates of the envs whose step was complete without a search; the call returns with both joined on `stream`.
 * next_actions_dev may be actions_dev (in place).  Other planners: the two calls back to back.  Requires cfg.oxford & 1. */
int d2d_step_plan_oxford(d2d_handle *h, const double *actions_dev, double *next_actions_dev, void *stream);

/* d2d_step_bound with the policy on the device: steps with the actions in "actions_staging" (bound with actions_host = NULL),
 * leaves the observation in the bound host buffers and the NEXT step's Oxford actions in "actions_staging"
 * (d2d_step_plan_oxford on the bound stream).  Prime the first step with d2d_plan_oxford(h, staging, stream). */
int d2d_step_bound_plan_oxford(d2d_handle *h);

/* Replaces NoControl / Rotating / LookAhead / LookGoal / Owl .plan(env.info) (yaw_planner.py:10-39, 136-255) for all envs:
 * writes the action per env to actions_out_dev (DEVICE [num_envs] f64).  `policy` is a d2d_gaze value.  Owl is called the
 * way experiment.py:33-34 calls it (the class object is the instance); its state (36 direction-uncertainty bins, the queue
 * of repeated actions) lives in the arena (cfg.oxford & D2D_POLICY_OWL), advances with every call and is re-initialised
 * with the env (a new policy per episode, experiment.py:27-34). */
int d2d_plan_gaze(d2d_handle *h, int32_t policy, double *actions_out_dev, void *stream);

/* Replaces direct writes to env.drone.x / .y / .yaw by the metric scripts
 * (script/difficulty_calculator/glob_survivability_calculator.py:36-37).  pose_host: [num_envs][3] f64 HOST. */
int d2d_set_drone_pose(d2d_handle *h, const double *pose_host, void *stream);

/* Named views of the arena (see DESIGN.md "Data layout"): "local_map", "yaw_angle", "done", "belief", "agent_pos",
 * "agent_pref", "agent_radius", "hit", "drone_x", ... Returns D2D_ERR_INVALID for an unknown name. */
int d2d_get_buffer(d2d_handle *h, const char *name, d2d_buffer_info *out);

/* Episode statistics accumulated on the device since the last call with reset != 0; copies D2D_NUM_STATS int64
 * counters to out_host (synchronises the stream).  The multi-GPU host all-reduces this vector (NCCL). */
int d2d_stats(d2d_handle *h, int64_t *out_host, int32_t reset, void *stream);

/* Per-env state copies, the counterpart of ALE cloneState / restoreState and MuJoCo get_state / set_state: branch an env
 * into copies, checkpoint and replay it, move it to another handle or GPU.  The state of an env is every per-env arena row:
 * the live state AND its reset snapshot (agents and their *0 rows, RVO velocities and obstacles, radii, ground truth,
 * belief, the 128-byte env record verbatim -- pending_reset included --, the step outputs and flags, trackers, trajectory,
 * planner verdicts, the np.random stream with its reset copy, Oxford / Owl policy state, drone acceleration).  Not part of
 * it: global tables, the statistics, the constant reward, scratch a step consumes within itself, and "actions_staging",
 * which holds caller data -- a caller that keeps the next actions there (d2d_step_bound_plan_oxford) must re-plan
 * (d2d_plan_oxford) after a clone or load.
 * d2d_clone_envs, d2d_save_state and d2d_load_state return D2D_ERR_STATE before d2d_set_world and while a pipelined step
 * is in flight, and check every argument before anything is enqueued (a rejected call changes nothing).  Each is ONE kernel
 * launch on `stream`.  Clone and load mark the host observation mirror stale, so the next host step refreshes it with one
 * full copy (as after d2d_reset). */

/* Env dst[i] becomes an exact copy of env src[i] (i < count): live state AND reset snapshot, so every later step,
 * auto/lazy reset and policy call of dst[i] is bit-identical to what src[i] would do with the same actions.
 * src_host / dst_host: HOST int32 arrays, validated before anything is enqueued (0 <= index < num_envs, dst entries
 * distinct, no index in both arrays; src entries may repeat: one env forks into several).  Statistics are not touched.
 * count = 0 does nothing.  One kernel launch. */
int d2d_clone_envs(d2d_handle *h, const int32_t *src_host, const int32_t *dst_host, int32_t count, void *stream);

/* Size of one env's packed state (a multiple of 128 B) and a 64-bit fingerprint of everything that decides the layout
 * or its meaning: d2d_config without num_envs / device / envs_per_block, plus a layout version.  Any handle, any time. */
int d2d_state_layout(const d2d_handle *h, int64_t *bytes_per_env, uint64_t *fingerprint);

/* Packs envs[i] into row i of a DEVICE buffer [count][bytes_per_env] (envs_host NULL: envs 0..count-1; entries may
 * repeat), and back: d2d_load_state writes row i into env envs[i] (entries distinct).  state_dev: device memory of the
 * handle's device, 16-byte aligned (else D2D_ERR_INVALID).  The packed rows can be moved anywhere (host, file, another
 * GPU) and loaded into any handle whose fingerprint matches; a different fingerprint is D2D_ERR_INVALID.  Padding bytes
 * between the fields of a packed row are left as they were. */
int d2d_save_state(d2d_handle *h, const int32_t *envs_host, int32_t count, void *state_dev, void *stream);
int d2d_load_state(d2d_handle *h, const int32_t *envs_host, int32_t count, const void *state_dev,
                   uint64_t fingerprint, void *stream);

/* World generation on the device: the world of a seed, as init_obstacles_random_size + OccupancyGridMap.init_obstacles
 * build it (drone_v2.py:12-66, utils.py:508-525) and world.generate_world restates it, generated by the GPU instead of the
 * host.  d2d_world_source holds the seed-independent inputs; the seed decides the rest through the reference's two
 * streams, Python's `random.Random(seed)` (pillars, agent positions and radii) and `np.random.RandomState(seed)` (the 100
 * group headings, then the measurement noise).  The result is what d2d_set_world / d2d_set_rng / d2d_set_rvo would store
 * for the host-generated world of that seed, bit for bit, except for the static-map group velocities: the reference
 * evaluates agent_max_speed * np.cos / np.sin(direction) with glibc, the device with correctly rounded sin / cos (they
 * differ by 1 ulp in about 0.1 % of the directions; DESIGN.md section 2). */
#define D2D_WORLD_MAX_RANDOM 256      /* random disc agents (params.agent_number) */
#define D2D_WORLD_MAX_PILLARS 64      /* params.pillar_number (at most 16 under the RVO motion profile) */
#define D2D_WORLD_GROUPS 100          /* group ids of the static map: np.random.rand(100) headings (drone_v2.py:54) */
#define D2D_WORLD_EAGER 1             /* reset the envs now, as d2d_reset does */
#define D2D_WORLD_LAZY 2              /* mark the envs (pending_reset): they start the new world at their next step */

typedef struct d2d_world_source {
    int32_t struct_size;              /* sizeof(d2d_world_source), ABI check */
    int32_t agent_number;             /* random disc agents, placed by rejection (drone_v2.py:28-47) */
    int32_t pillar_number;            /* circular obstacles, placed first (drone_v2.py:14-26) */
    int32_t pad_;
    double agent_radius;              /* params.agent_radius; -1: random radii uniform(5, 15) */
    double agent_max_speed;
    double drone_radius;
    double init_x, init_y;            /* params.init_position: the drone's reset pose (yaw 270) */
    double map_w, map_h;              /* params.map_size */
    /* the random agents' preferred velocities -v * [cos, sin](2 pi k / agent_number) as the host's NumPy evaluates them */
    double headings[D2D_WORLD_MAX_RANDOM][2];
    /* the static map (params.static_map), [x][y]: 0 = free, else the group id of the radius-5 agent on that cell, < 100 */
    uint8_t static_map[50][50];
} d2d_world_source;

/* World keys: a world is named by key = source * 2^32 + seed, `source` an index into the handle's table of world sources
 * (d2d_set_world_sources) and `seed` in [0, 2^32).  With source 0 the key is the seed, so a handle with one source sees
 * seeds everywhere a key is stored ("world_seed", d2d_episode_record.seed). */
#define D2D_WORLD_MAX_SOURCES 4096

/* Stores the table of world sources srcs[0, count) (HOST structs, copied), 1 <= count <= D2D_WORLD_MAX_SOURCES; a later
 * call replaces the table.  Every source is checked against the config: the map size, drone_radius and agent_radius must
 * be the config's, agent_number + the non-zero cells of static_map == num_agents, and under RVO pillar_number <= 16.  All
 * or nothing: a rejected call changes nothing and names the index of the first bad source.  The device table grows only:
 * a call with more sources than any earlier one reallocates it and synchronises the device first, so a CUDA graph captured
 * before (its generation kernels hold the table's address) must be captured again; a call that fits also synchronises the
 * device (no d2d_generate_worlds kernel and no seed-queue generation behind a logged step may still read the table) and
 * overwrites the table in place.  Keys queued before (d2d_set_world_queue) are not re-checked. */
int d2d_set_world_sources(d2d_handle *h, const d2d_world_source *srcs, int32_t count);

/* d2d_set_world_sources(h, src, 1). */
int d2d_set_world_source(d2d_handle *h, const d2d_world_source *src);

/* Generates the worlds of seeds_host[i] into envs envs_host[i] (HOST arrays, i < count) in ONE launch on `stream`,
 * asynchronously.  Writes the reset snapshot (agents and their *0 rows, radii, ground truth, the reset pose, the np.random
 * stream when var_cam != 0, the RVO velocities and obstacles) and then, by `flags`:
 *   D2D_WORLD_EAGER  resets the envs as d2d_reset does (a second launch) and marks the host mirror stale;
 *   D2D_WORLD_LAZY   marks them like d2d_request_reset: each starts the new world at its next step.  Under auto_reset this is
 *                    what happens to an env that just reported done; its terminal outputs stay readable until that step,
 *                    and a gaze policy called in between already sees the new initial state.
 * Everything is checked before anything is enqueued (a rejected call changes nothing): envs in [0, num_envs) and distinct,
 * seeds in [0, 2^32) (np.random.RandomState rejects anything else), exactly one flag.  D2D_ERR_STATE before
 * d2d_set_world_source and while a pipelined step is in flight.  Statistics are untouched; the first call counts as
 * d2d_set_world (+ d2d_set_rng / d2d_set_rvo).
 * A seed whose world cannot be built (the reference's rejection loops would never end: more than 65536 rejected draws in a
 * row) is recorded by the kernel; the NEXT call reports it with D2D_ERR_STATE (env, seed and source in d2d_last_error),
 * clears it and does nothing else.  count = 0 enqueues nothing: after synchronising the stream it reports such a failure at once. */
int d2d_generate_worlds(d2d_handle *h, const int32_t *envs_host, const int64_t *seeds_host, int32_t count, int32_t flags,
                        void *stream);

/* d2d_generate_worlds with world keys: envs_host[i] gets the world of seed keys_host[i] & 0xffffffff built from source
 * keys_host[i] >> 32.  A negative key, or one whose source is not in the table, is rejected before anything is enqueued.
 * A world that cannot be built is reported as above, with its env, seed and source. */
int d2d_generate_worlds_keyed(d2d_handle *h, const int32_t *envs_host, const int64_t *keys_host, int32_t count, int32_t flags,
                              void *stream);

/* Episode log: one fixed-size record per (step, env) that reported done -- everything the reference's experiment row
 * (experiment.py:69-101) needs, written on the device by the step that finished the episode, so a driver can step many
 * times between host synchronisations.  The events are exactly those D2D_STAT_EPISODES counts. */
typedef struct d2d_episode_record {   /* 48 bytes */
    int64_t seed;                /* "world_seed"[env] at the step that reported done: the world key (the seed for source 0) */
    int64_t step;                /* index of that step among the steps logged since the log was enabled */
    int64_t tracked_steps;       /* "tracker_buffer_ts" */
    int32_t env;
    int32_t steps;               /* "steps" (flight time = steps * dt) */
    int32_t grid_discovered;     /* belief cells != 0 */
    int32_t trackers;            /* "tracker_buffer_count" */
    uint8_t state_machine, collision_flag, freezing_flag, dead_lock_flag;
    int32_t reserved;
} d2d_episode_record;

/* Enables the episode log with room for `capacity` records (0 disables it and frees its buffers; enabling again
 * reallocates them, so a CUDA graph captured before must be captured again).  Synchronises the device.  The library-owned
 * DEVICE buffers (d2d_get_buffer; D2D_ERR_STATE while the log is disabled):
 *   "episode_log"       [capacity][48] u8 records
 *   "episode_log_head"  int64[4]: records written since the last read, steps logged, seeds handed out by the queue, queue length
 *   "world_seed"        int64 [num_envs], zero when enabled: the key of each env's world (its seed for source 0).  The
 *                       caller writes it with ordinary device writes; the library writes it only from the seed queue.
 *                       Not env state: clone / save / load and the state layout ignore it.
 * While the log is enabled every step entry point (d2d_step, d2d_step_plan_oxford after its side stream has joined,
 * d2d_step_host, d2d_step_bound, d2d_step_bound_plan_oxford) enqueues one more kernel behind the step: it appends a record
 * for every env whose "done" is non-zero, in ascending env order, so the log is in (step, env) order.  The step counter
 * lives on the device, so replays of a captured graph count correctly.  d2d_rollout runs its K steps as K per-step launches
 * (each followed by the log kernel) and d2d_step_pipelined takes its synchronous path.  Resets, clone and load write no
 * records.  A record that finds the log full is not written but counted (the `dropped` of the next read); a capacity of
 * num_envs x (steps between reads) never drops.  With the log disabled (the default) nothing is launched. */
int d2d_enable_episode_log(d2d_handle *h, int64_t capacity);

/* Synchronises `stream`, copies the records written since the last read to out_host (HOST, room for `capacity` records),
 * their number to *count and the number of records the full log could not take to *dropped, then resets the written
 * count (in stream order).  D2D_ERR_STATE when the log is disabled, or when a world of the seed queue could not be built
 * (env, seed and source in d2d_last_error; the failure is cleared, the records stay for the next read). */
int d2d_read_episode_log(d2d_handle *h, d2d_episode_record *out_host, int64_t *count, int64_t *dropped, void *stream);

/* Seed queue: from the next logged step on, every env that reports done takes the next seed of the queue (ascending env
 * order within a step, while seeds remain).  Its record carries the OLD "world_seed"; "world_seed"[env] becomes the new seed
 * and a second kernel behind the log kernel generates that world with D2D_WORLD_LAZY semantics, so the env starts it at its
 * next step (d2d_generate_worlds).  When the queue runs out, finished envs auto-reset into their last world as before.  A
 * world that cannot be built is reported by the next d2d_read_episode_log or d2d_generate_worlds.  No host copy per step:
 * gaze policy, step, log and generation can be captured in a CUDA graph together.
 * seeds_host: HOST int64 [count], each in [0, 2^32); uploaded, the queue cursor is reset in stream order; count = 0 clears
 * the queue.  D2D_ERR_STATE without d2d_set_world_source, without cfg.auto_reset or without an enabled log.  A rejected
 * call changes nothing. */
int d2d_set_seed_queue(d2d_handle *h, const int64_t *seeds_host, int64_t count, void *stream);

/* The seed queue with world keys (d2d_generate_worlds_keyed): keys_host HOST int64 [count], each naming a source of the
 * current table; "world_seed" and the records carry the keys.  The same contract as d2d_set_seed_queue otherwise. */
int d2d_set_world_queue(d2d_handle *h, const int64_t *keys_host, int64_t count, void *stream);

/* Rendering: replaces Drone2DEnv2.render (drone_v2.py:263-303, utils.py:31-64, 550-558, 786-817) with rgb_array frames drawn
 * on the device instead of a pygame window.  Frame of one env: uint8 [H][W][3] RGB, C-contiguous, H = W = 50 * ppc
 * (pixels_per_cell in 1..D2D_RENDER_MAX_PPC; ppc 10 is the reference's 500 x 500 screen), in the screen layout: column =
 * world x, row = world y, origin top-left; cell (i, j) covers rows j*ppc.. and columns i*ppc...  `layers` (D2D_RENDER_*
 * bits) are drawn back to front: ground truth / belief cells, the field of view the step's rays sweep, the planner target and
 * the remaining Primitive waypoints, active tracker rings, agents (red if seen this step, else blue), the drone.  Exact
 * pixel rules and palette: DESIGN.md section 2, "Rendering".
 * Envs: envs_host == NULL renders [first_env, first_env + count); otherwise envs_host[0..count) (HOST int32, repeats
 * allowed, at most D2D_RENDER_MAX_LIST entries), passed by value in the kernel's parameters: either form is ONE kernel
 * launch with no upload, so it can be captured in a CUDA graph beside the step.  frames_dev: DEVICE [count][H][W][3] of
 * the handle's device, any byte alignment.  Every argument is checked before anything is enqueued (a rejected call writes
 * nothing); count = 0 enqueues nothing.  D2D_ERR_STATE before d2d_set_world and while a pipelined step is in flight.
 * The call reads the arena and writes only the frames.  It shows the arena as it is: an env that just reported done shows
 * its terminal state until its next step, an env with a lazy reset or reseed pending shows its old world until then. */
#define D2D_RENDER_MAX_PPC 10
#define D2D_RENDER_MAX_LIST 1024      /* longest env list; larger selections are a contiguous range */
enum { D2D_RENDER_GROUND_TRUTH = 1, D2D_RENDER_BELIEF = 2, D2D_RENDER_VIEW = 4, D2D_RENDER_PLAN = 8,
       D2D_RENDER_TRACKERS = 16, D2D_RENDER_AGENTS = 32, D2D_RENDER_DRONE = 64, D2D_RENDER_ALL = 127 };
int d2d_render(d2d_handle *h, const int32_t *envs_host, int32_t first_env, int32_t count, int32_t pixels_per_cell,
               int32_t layers, uint8_t *frames_dev, void *stream);

/* Difficulty: the survivability metric family of the reference (script/difficulty_calculator/survivability_calculator.py,
 * glob_survivability_calculator.py) evaluated on the device from each env's RESET SNAPSHOT (agent_pos0 / agent_pref0,
 * agent_radius, ground truth).  The kernel steps the agents alone, K = spec->steps times, with the step kernels' CVM
 * Agent.step, and after agent step k = 1..K tests every position p of the grid x = x0 + i * step, y = y0 + j * step
 * (i < nx, j < ny; position index i * ny + j):
 *   dynamic hit  any agent a: norm(agent_a - p) < r_a + drone_radius     (Drone2D.is_collide's agent test)
 *   static hit   one of the five probes of Drone2D.is_collide at p meets an occupied or off-map cell (collision_flag 1)
 * Outputs, DEVICE memory of the handle's device, for envs [first_env, first_env + count):
 *   first_hit       int16 [count][nx*ny]  first step k with a dynamic hit (0: none within `steps`); statics ignored
 *   static_hit      uint8 [count][nx*ny]  1 if the drone at p collides with a static cell
 *   collision_state uint8 [count][nx*ny][n_slots] or NULL: byte [p][slot[k-1]] is OR-ed with (dynamic hit after step k and
 *                   no static hit) -- glob_survivability's array, collision_flag == 2 -- for every k with slot[k-1] !=
 *                   D2D_DIFF_NO_SLOT; every other byte is 0.  NULL requires n_slots == 0 and vice versa.
 * Only CVM handles: under RVO the agents' motion needs d2d_rvo_kernel, and the call returns D2D_ERR_STATE (step the envs
 * and test the grid after every step with d2d_grid_hits below).  The planner does not matter.  The spec travels by value
 * in the kernel parameters: a call is ONE launch with no upload and can be captured in a CUDA graph.  Every argument is checked before
 * anything is enqueued (a rejected call changes nothing); count = 0 enqueues nothing.  The call reads the reset snapshot and
 * writes only the outputs: env state, statistics, the episode log and the host mirror are untouched, and the result does not
 * depend on how far the envs have stepped.  D2D_ERR_STATE before d2d_set_world and while a pipelined step is in flight. */
#define D2D_DIFF_MAX_POS   1024
#define D2D_DIFF_MAX_STEPS 1024
#define D2D_DIFF_NO_SLOT   0xFFFF      /* slot[] entry: step k is not recorded in collision_state */
typedef struct d2d_difficulty_spec {
    int32_t struct_size;                  /* sizeof(d2d_difficulty_spec) */
    int32_t nx, ny;                       /* position grid, nx * ny in 1..D2D_DIFF_MAX_POS */
    double  x0, y0, step;                 /* finite; step > 0 */
    int32_t steps;                        /* K agent steps from the reset snapshot, 1..D2D_DIFF_MAX_STEPS */
    int32_t n_slots;                      /* collision_state slots per position, 0..D2D_DIFF_MAX_STEPS; 0 = not written */
    uint16_t slot[D2D_DIFF_MAX_STEPS];    /* slot of step k (k = 1..steps): < n_slots or D2D_DIFF_NO_SLOT, non-decreasing */
} d2d_difficulty_spec;
int d2d_difficulty(d2d_handle *h, const d2d_difficulty_spec *spec, int32_t first_env, int32_t count, int16_t *first_hit,
                   uint8_t *static_hit, uint8_t *collision_state, void *stream);

/* Grid hits: the outputs of d2d_difficulty built one step at a time from the LIVE agents (agent_pos, agent_radius) instead
 * of the reset snapshot, for every motion profile (CVM and RVO) and any planner.  The caller steps the envs with the step
 * kernels and calls d2d_grid_hits with t = 1, 2, ..., spec->steps after step t; the outputs then equal d2d_difficulty's
 * for agents moved by those steps (under CVM from a reset, exactly d2d_difficulty's).  Call t folds the positions hit now
 * into the outputs:
 *   t == 1          first_hit is set to 1 where hit and 0 elsewhere, and the range's collision_state rows are zero-filled;
 *   t > 1           first_hit is set to t where it is still 0 and the position is hit;
 *   every call      static_hit is written (the same value each time: the ground truth does not move), and for a step with
 *                   slot[t-1] != D2D_DIFF_NO_SLOT byte [p][slot[t-1]] of collision_state is set to 1 at every hit position
 *                   that is not static.
 * Same spec, outputs, range and checks as d2d_difficulty, plus 1 <= t <= spec->steps.  A run's calls must go to one stream
 * (or be otherwise ordered), use the same spec, range and outputs, and see no reset, reseed or world change between t = 1
 * and spec->steps.  Every argument is checked before anything is enqueued (a rejected call changes nothing); count = 0
 * enqueues nothing.  ONE launch with no upload, so a loop of steps and calls can be captured in a CUDA graph.  The call
 * reads the agents and the ground truth and writes only the outputs: env state, statistics, the episode log and the host
 * mirror are untouched.  D2D_ERR_STATE before d2d_set_world and while a pipelined step is in flight. */
int d2d_grid_hits(d2d_handle *h, const d2d_difficulty_spec *spec, int32_t t, int32_t first_env, int32_t count,
                  int16_t *first_hit, uint8_t *static_hit, uint8_t *collision_state, void *stream);

/* Number of kernel launches issued by this handle so far (bench.py's gpu_launches). */
int64_t d2d_launch_count(const d2d_handle *h);

#ifdef __cplusplus
}
#endif
#endif /* DRONE2D_H */
