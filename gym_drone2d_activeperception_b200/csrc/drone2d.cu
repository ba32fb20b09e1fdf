// drone2d.cu -- C-ABI implementation of libdrone2d.so (see include/drone2d.h).
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false -lineinfo -O3 --shared -Xcompiler -fPIC
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <string>
#include <vector>
#include <initializer_list>

#include "d2d_state.cuh"
#include "d2d_math.cuh"
#include "d2d_step.cuh"
#include "d2d_plan.cuh"
#include "d2d_rvo.cuh"
#include "d2d_clone.cuh"
#include "d2d_worldgen.cuh"
#include "d2d_episode.cuh"
#include "d2d_render.cuh"
#include "d2d_difficulty.cuh"

// ------------------------------------------------------------------------------------------ handle
// Per-env state tag of an arena buffer: env e's row of `row_bytes` bytes starts at offset + e * row_stride, in each of
// `planes` planes that lie plane_stride bytes apart.  d2d_clone_envs / d2d_save_state / d2d_load_state copy exactly the
// tagged rows.  planes == 0 (NOT_ENV_STATE): global tables, the statistics, caller data and scratch a step consumes within
// itself.  add_buf takes the tag as a required argument, so every buffer added later must say which it is.
struct EnvRows {
    int64_t row_bytes, row_stride;
    int planes;
    int64_t plane_stride;
};
static const EnvRows NOT_ENV_STATE = {0, 0, 0, 0};
static EnvRows env_rows(int64_t row_bytes, int planes = 1, int64_t plane_stride = 0) {
    return EnvRows{row_bytes, row_bytes, planes, plane_stride};
}

struct BufDesc {
    std::string name;
    size_t offset, nbytes;
    int dtype, ndim;
    int64_t shape[4], strides[4];
    EnvRows rows = NOT_ENV_STATE;
};

struct d2d_handle {
    d2d_config cfg;
    DevP P;
    int B, Bpad, N, NP, HW, E, T;
    unsigned char *arena = nullptr;
    size_t arena_bytes = 0;
    std::vector<BufDesc> bufs;
    double *stage_actions = nullptr;     // device staging for d2d_step_host
    int64_t launches = 0;
    int64_t step_count = 0;
    bool world_set = false;
    bool rng_set = false;
    bool rvo_set = false;
    bool jerk_set = false;
    std::string err;
    size_t smem_step = 0, smem_post = 0;
    int plan_threads = 64;
    OxProgram *ox_prog = nullptr;
    CloneTable state_tab;                 // per-env state rows (EnvRows tags) and their packed layout
    uint64_t state_fingerprint = 0;
    int *clone_idx = nullptr;             // device copy of the index arrays of the last clone / save / load
    size_t clone_idx_bytes = 0;
    std::vector<int32_t> clone_stage;     // host staging of those arrays
    cudaEvent_t clone_ev = nullptr;       // recorded behind the last kernel that read clone_idx
    double *ox_export = nullptr;          // lazily allocated [B][2500] view of last_time_observed
    // world generation (d2d_set_world_sources / d2d_generate_worlds_keyed)
    WgTables *wg_tab = nullptr;           // device table of the seed-independent tables, one per world source
    int32_t wg_count = 0;                 // sources in the table (the valid range of a key's high word)
    int32_t wg_cap = 0;                   // sources wg_tab can hold (grows only)
    int32_t *wg_idx = nullptr;            // device: [count] envs, (8-byte aligned) [count] keys (i64), [num_envs] reset mask
    size_t wg_idx_bytes = 0;
    std::vector<int32_t> wg_stage;        // host staging of those arrays
    cudaEvent_t wg_ev = nullptr;          // recorded behind the last kernel that read wg_idx
    volatile unsigned long long *wg_fault = nullptr;   // pinned, mapped [2]: (1 << 63 | key), env of a world given up
    unsigned long long *wg_fault_dev = nullptr;        // device-visible address of wg_fault
    unsigned int *wg_claim = nullptr;     // device: non-zero once a kernel has claimed wg_fault (first failure wins)
    // episode log and seed queue (d2d_enable_episode_log / d2d_set_world_queue); ep_mem == nullptr: disabled
    unsigned char *ep_mem = nullptr;      // records, head, world_seed, list, gen_env, gen_key, gen_count in one allocation
    EpLog ep = {};
    long long *ep_queue = nullptr;        // device copy of the queue
    int64_t ep_queue_cap = 0;             // keys it can hold
    int64_t ep_qlen = 0;                  // keys of the current queue (0: no queue, no generation launch)
    int ep_blocks = 1;                    // grid of d2d_episode_log_kernel: one block per 32 envs, at most one per SM
    long long ep_qhead[2] = {0, 0};       // host staging of head[2], head[3]
    // zero-copy observation mirror (d2d_bind_host_mirror): host addresses as bound; *_stale: the host copy must be
    // refreshed by a full device->host copy at the next d2d_step_host (after bind / eager reset)
    uint8_t *mir_lm = nullptr; float *mir_yaw = nullptr; uint8_t *mir_done = nullptr;
    bool mir_stale = true;
    size_t smem_pre = 0, smem_plan = 0;
    int plan_small = -1;                 // d2d_plan_small_kernel: -1 not decided yet, 0 off, > 0 grid size (co-resident blocks)
    int plan_sms = 0;                    // SMs of the device (set with plan_small)
    // d2d_step_plan_oxford: the A* searches of a step run on this stream beside the Oxford scoring of the other envs
    cudaStream_t side_stream = nullptr;
    cudaEvent_t side_ev[2] = {nullptr, nullptr};     // [0] step kernel done (fork), [1] planning envs completed (join)
    std::vector<const void *> attr_funcs;   // kernels whose dynamic shared-memory limit this handle has raised
    // bound host path (d2d_bind_host_io)
    bool io_bound = false;
    const double *io_actions_dev = nullptr;      // device-visible address of the caller's pinned action buffer (or staging)
    uint8_t *io_lm = nullptr; float *io_yaw = nullptr; uint8_t *io_done = nullptr;
    cudaStream_t io_stream = nullptr;
    // pipelined stepping (d2d_step_pipelined): gate word + fault word in one pinned, mapped allocation
    volatile unsigned int *gate_host = nullptr;  // pinned: [16] fault word written by a kernel that gave up waiting
    unsigned int *gate_dev = nullptr;            // device-visible address of gate_host
    const double *io_actions_host = nullptr;     // the caller's pinned action buffer (host address)
    cudaStream_t copy_stream = nullptr;          // carries the per-step action copy
    unsigned int pipe_seq = 0;
    bool pipe_inflight = false;                  // the kernel of the NEXT step has been launched and waits at its gate
    int pipe_mode = 0;                           // 1: one pre-launched kernel per step; 2: resident kernel (whole run, B <= one wave)
    double *pipe_pub = nullptr;                  // pinned [B + 1]: the step's actions + stamp word, source of the ONE copy per step
    unsigned long long *pipe_count = nullptr;    // device counter behind DevP::gate_count
    int resident_capacity = -1;                  // envs the resident kernel can hold at once (blocks/SM x SMs x warps/block)
    int resident_blocks = 0;                     // ... and the blocks that are co-resident (one may serve as the courier)
    bool pipe_courier = false;                   // this run's actions are pulled by the kernel's courier block (no copy engine)
    cudaEvent_t pipe_ev[3] = {nullptr, nullptr, nullptr};   // [0], [1]: completion of alternate steps; [2]: sentinels in place
    // D2D_PIPE_DEBUG=1: host-side time of the phases of d2d_step_pipelined, printed by d2d_destroy
    double dbg_launch_ns = 0, dbg_wait_ns = 0, dbg_total_ns = 0; long dbg_n = 0, dbg_polls = 0;
};
#include <time.h>
static inline double now_ns() { timespec t; clock_gettime(CLOCK_MONOTONIC, &t); return t.tv_sec * 1e9 + t.tv_nsec; }

#define D2D_NO_PIPE(h)                                                                                                 \
    do {                                                                                                               \
        if ((h)->pipe_inflight) {                                                                                      \
            (h)->err = "a pipelined step is in flight: finish it with d2d_step_pipelined(h, 0) first";                 \
            return D2D_ERR_STATE;                                                                                      \
        }                                                                                                              \
    } while (0)

// Raises the dynamic shared-memory limit of `func` to 227 KB once per handle.  Per handle, not per process: a handle is
// driven by one thread at a time (drone2d.h), so no state is shared between threads that drive distinct handles.
static int ensure_smem_attr(d2d_handle *h, const void *func, const char *what) {
    for (const void *f : h->attr_funcs) if (f == func) return D2D_OK;
    cudaError_t ce = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (ce != cudaSuccess) { h->err = std::string("cudaFuncSetAttribute(") + what + "): " + cudaGetErrorString(ce); return D2D_ERR_CUDA; }
    h->attr_funcs.push_back(func);
    return D2D_OK;
}

static thread_local std::string g_create_err;

static size_t dtype_size(int dt) {
    switch (dt) {
        case D2D_U8: case D2D_I8: return 1;
        case D2D_I32: case D2D_F32: return 4;
        default: return 8;
    }
}

#define CUDA_TRY(h, call)                                                                          \
    do {                                                                                           \
        cudaError_t _e = (call);                                                                   \
        if (_e != cudaSuccess) {                                                                   \
            (h)->err = std::string(#call) + ": " + cudaGetErrorString(_e);                         \
            return D2D_ERR_CUDA;                                                                   \
        }                                                                                          \
    } while (0)

// registers a buffer of `count` rows x inner dims; returns offset
static size_t add_buf(d2d_handle *h, size_t &cursor, const char *name, int dtype, int ndim,
                      std::initializer_list<int64_t> shape, std::initializer_list<int64_t> strides, size_t alloc_elems,
                      EnvRows rows) {
    BufDesc b;
    b.name = name; b.dtype = dtype; b.ndim = ndim; b.rows = rows;
    for (int i = 0; i < 4; i++) { b.shape[i] = i < ndim ? shape.begin()[i] : 1; b.strides[i] = i < ndim ? strides.begin()[i] : 1; }
    cursor = (cursor + 255) / 256 * 256;
    b.offset = cursor;
    b.nbytes = alloc_elems * dtype_size(dtype);
    cursor += b.nbytes;
    h->bufs.push_back(b);
    return b.offset;
}

// registers a named strided view of bytes that another buffer owns (fields of the per-env EnvRec records)
static void add_view(d2d_handle *h, const char *name, int dtype, int ndim, std::initializer_list<int64_t> shape,
                     std::initializer_list<int64_t> strides, size_t offset, size_t nbytes) {
    BufDesc b;
    b.name = name; b.dtype = dtype; b.ndim = ndim;
    for (int i = 0; i < 4; i++) { b.shape[i] = i < ndim ? shape.begin()[i] : 1; b.strides[i] = i < ndim ? strides.begin()[i] : 1; }
    b.offset = offset; b.nbytes = nbytes;
    h->bufs.push_back(b);
}

extern "C" int d2d_version(void) { return D2D_VERSION; }

extern "C" const char *d2d_last_error(const d2d_handle *h) { return h ? h->err.c_str() : g_create_err.c_str(); }

extern "C" int64_t d2d_launch_count(const d2d_handle *h) { return h ? h->launches : 0; }

// ------------------------------------------------------------------------------------------ reset kernel
// Eager reset (Drone2DEnv2.reset -> __init__, drone_v2.py:259-261, 69-117) of masked envs from the snapshot.
__global__ void d2d_reset_kernel(const DevP P, const uint8_t *__restrict__ mask) {
    const int e = blockIdx.x;
    if (e >= P.B) return;
    if (mask && !mask[e]) return;
    const int tid = threadIdx.x, T = blockDim.x;
    const size_t base = (size_t)e * P.NP;
    for (int k = tid; k < P.N; k += T) {
        P.apos[base + k] = P.apos0[base + k];
        P.apref[base + k] = P.apref0[base + k];
        if (P.motion_rvo) P.avel[base + k] = P.avel0[base + k];
        P.hit[base + k] = 0;
        P.trk_active[base + k] = 0;
        P.trk_radius[base + k] = P.trk_radius0[base + k];
        P.trk_ts[base + k] = 1;
        double *mu = P.trk_mu + (base + k) * 4, *S = P.trk_sigma + (base + k) * 16;
        for (int i = 0; i < 4; i++) mu[i] = 0.0;
        for (int i = 0; i < 16; i++) S[i] = 0.0;
        S[0] = 1.0; S[5] = 1.0; S[10] = 10.0; S[15] = 10.0;
    }
    uint32_t *bel = (uint32_t *)(P.belief + (size_t)e * D2D_BELIEF_STRIDE);
    for (int w = tid; w < D2D_BELIEF_STRIDE / 4; w += T) bel[w] = 0u;
    for (int w = tid; w < D2D_LOCAL_CELLS; w += T) P.local_map[(size_t)e * D2D_LOCAL_CELLS + w] = 0;
    if (P.ox_seen)
        for (int w = tid; w < D2D_OX_SEEN_STRIDE / 2; w += T) ((uint32_t *)(P.ox_seen + (size_t)e * D2D_OX_SEEN_STRIDE))[w] = 0u;
    if (P.owl_U)
        for (int w = tid; w < D2D_OWL_BINS; w += T) P.owl_U[(size_t)e * D2D_OWL_BINS + w] = 0.0;
    if (P.rng_key)
        for (int w = tid; w < 624; w += T) P.rng_key[(size_t)e * 624 + w] = P.rng_key0[(size_t)e * 624 + w];
    if (tid == 0) {
        const double x = P.rec[e].p0x, y = P.rec[e].p0y, yaw = P.rec[e].p0yaw;
        P.rec[e].px = x; P.rec[e].py = y; P.rec[e].yaw = yaw; P.rec[e].vx = 0; P.rec[e].vy = 0;
        P.rec[e].tgx = x; P.rec[e].tgy = y;
        if (P.planner == D2D_PLANNER_JERK) { P.rec[e].tgx = 0.0; P.rec[e].tgy = 0.0; }   // Jerk_Primitive.__init__ :406
        P.drone_acc[e] = double2{0.0, 0.0};
        P.rec[e].steps = 0; P.rec[e].sm = SM_WAIT_FOR_GOAL; P.rec[e].fail = 0; P.rec[e].tcur = 0;
        P.collision[e] = 0; P.dead_lock[e] = 0; P.freezing[e] = 0; P.done[e] = 0; P.rec[e].pending_reset = 0;
        P.rec[e].bufc = 0; P.rec[e].bufts = 0; P.rec[e].tracked = 0;
        P.rec[e].nseg = 0; P.rec[e].cursor = 0; P.need_plan[e] = 0; P.plan_ok[e] = 1; P.replan[e] = 0;
        P.yaw_obs[e] = (float)yaw;
        P.rec[e].ox_fresh = 0; P.rec[e].owl_fresh = 0; P.owl_q[e] = 0; P.owl_u[e] = 0.0; P.tmp_act_cnt[e] = 0; P.tmp_act_ts[e] = 0; P.ox_calls[e] = 0;
        P.rng_pos[e] = P.rng_pos0[e]; P.rng_has[e] = P.rng_has0[e]; P.rng_gauss[e] = P.rng_gauss0[e];
        // local_map was zeroed above, which IS the window of an all-unexplored belief grid at the initial cell
        P.rec[e].obs_ix = d2d_cell(x, P.scale, P.inv_scale); P.rec[e].obs_iy = d2d_cell(y, P.scale, P.inv_scale);
    }
}

__global__ void d2d_set_pose_kernel(const DevP P, const double *__restrict__ pose) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= P.B) return;
    P.rec[e].px = pose[3 * e]; P.rec[e].py = pose[3 * e + 1]; P.rec[e].yaw = pose[3 * e + 2];
    P.rec[e].obs_ix = -1000000; P.rec[e].obs_iy = -1000000;   // the observation window must be rebuilt
}

// NumPy pairwise-sum recursion for a contiguous run of n doubles -> leaf blocks + post-order combine program
static void ox_rec(OxProgram *p, int off, int n) {
    if (n <= 128) {
        const int id = p->n_leaves++;
        p->leaf_off[id] = off; p->leaf_len[id] = n;
        p->ops[p->n_ops++] = id;
        return;
    }
    int n2 = n / 2;
    n2 -= n2 % 8;
    ox_rec(p, off, n2);
    ox_rec(p, off + n2, n - n2);
    p->ops[p->n_ops++] = -1;
}
static void build_ox_program(OxProgram *p, int n) {
    memset(p, 0, sizeof(*p));
    ox_rec(p, 0, n);
    // the post-order program as a tree with level-sorted internal nodes (see OxProgram)
    int st[64], lvl[2 * D2D_OX_MAX_LEAVES] = {0}, L[D2D_OX_MAX_LEAVES], R[D2D_OX_MAX_LEAVES], ID[D2D_OX_MAX_LEAVES];
    int sp = 0, next = p->n_leaves, ni = 0, maxlev = 0;
    for (int o = 0; o < p->n_ops; o++) {
        const int op = p->ops[o];
        if (op >= 0) { st[sp++] = op; continue; }
        const int r = st[--sp], l = st[--sp];
        L[ni] = l; R[ni] = r; ID[ni] = next;
        lvl[next] = 1 + (lvl[l] > lvl[r] ? lvl[l] : lvl[r]);
        if (lvl[next] > maxlev) maxlev = lvl[next];
        st[sp++] = next++;
        ni++;
    }
    p->root = st[0];
    p->n_levels = maxlev;
    int w = 0;
    for (int lev = 1; lev <= maxlev; lev++) {
        p->lev_off[lev - 1] = w;
        for (int j = 0; j < ni; j++)
            if (lvl[ID[j]] == lev) { p->node_id[w] = ID[j]; p->node_l[w] = L[j]; p->node_r[w] = R[j]; w++; }
    }
    p->lev_off[maxlev] = w;
}

// ------------------------------------------------------------------------------------------ per-env state layout
// Bump when the packed state format changes in a way the config does not show (it is part of the fingerprint).
#define D2D_STATE_LAYOUT_VERSION 1

static uint64_t fnv1a(uint64_t x, const void *p, size_t n) {
    const unsigned char *c = (const unsigned char *)p;
    for (size_t i = 0; i < n; i++) { x ^= c[i]; x *= 1099511628211ull; }
    return x;
}

// The field table of d2d_clone_kernel from the EnvRows tags (one field per plane; packed rows 16-B aligned, the whole
// packed state a multiple of 128 B) and the fingerprint of the layout: the config without num_envs / device /
// envs_per_block (which change neither the rows nor their meaning), the layout version, and every field's name and shape.
static bool build_state_layout(d2d_handle *h) {
    CloneTable &T = h->state_tab;
    memset(&T, 0, sizeof(T));
    d2d_config c = h->cfg;
    c.num_envs = 0; c.device = 0; c.envs_per_block = 0;
    const uint32_t version = D2D_STATE_LAYOUT_VERSION;
    uint64_t fp = fnv1a(14695981039346656037ull, &version, sizeof(version));
    fp = fnv1a(fp, &c, sizeof(c));
    uint64_t pack = 0;
    for (const BufDesc &b : h->bufs)
        for (int p = 0; p < b.rows.planes; p++) {
            if (T.n == D2D_CLONE_MAX_FIELDS) return false;
            CloneField &f = T.f[T.n++];
            f.off = b.offset + (uint64_t)p * b.rows.plane_stride;
            f.stride = (uint64_t)b.rows.row_stride;
            f.bytes = (unsigned int)b.rows.row_bytes;
            f.pack = (unsigned int)pack;
            pack = (pack + f.bytes + 15) / 16 * 16;
            fp = fnv1a(fp, b.name.c_str(), b.name.size() + 1);
            fp = fnv1a(fp, &p, sizeof(p));
            fp = fnv1a(fp, &f.bytes, sizeof(f.bytes));
            fp = fnv1a(fp, &f.pack, sizeof(f.pack));
        }
    T.pack_bytes = (unsigned int)((pack + 127) / 128 * 128);
    h->state_fingerprint = fnv1a(fp, &T.pack_bytes, sizeof(T.pack_bytes));
    return true;
}

// ------------------------------------------------------------------------------------------ create / destroy
extern "C" int d2d_create(const d2d_config *cfg, d2d_handle **out) {
    if (!cfg || !out) { g_create_err = "null argument"; return D2D_ERR_INVALID; }
    if (cfg->struct_size != (int32_t)sizeof(d2d_config)) { g_create_err = "d2d_config size mismatch (ABI)"; return D2D_ERR_INVALID; }
    if (cfg->num_envs <= 0 || cfg->num_agents < 0 || cfg->num_agents > 4000) { g_create_err = "bad num_envs / num_agents"; return D2D_ERR_INVALID; }
    if (cfg->motion_profile != D2D_MOTION_CVM && cfg->motion_profile != D2D_MOTION_RVO) { g_create_err = "bad motion_profile"; return D2D_ERR_INVALID; }
    if (cfg->planner < D2D_PLANNER_NOMOVE || cfg->planner > D2D_PLANNER_JERK) { g_create_err = "bad planner"; return D2D_ERR_INVALID; }
    if (cfg->planner == D2D_PLANNER_JERK && cfg->envs_per_block > 0) {
        g_create_err = "the Jerk_Primitive planner is only implemented on the default warp-per-env kernel (envs_per_block = 0)";
        return D2D_ERR_INVALID;
    }
    if (cfg->motion_profile == D2D_MOTION_RVO && d2d_rvo_smem_bytes(cfg->num_agents) > 200 * 1024) {
        g_create_err = "RVO motion profile: too many agents for one block's shared memory"; return D2D_ERR_INVALID;
    }
    if ((int)(cfg->map_w / cfg->map_scale) != D2D_GRID || (int)(cfg->map_h / cfg->map_scale) != D2D_GRID) {
        g_create_err = "only 50x50-cell maps are supported (map_size // map_scale == 50)"; return D2D_ERR_INVALID;
    }
    if (4 * (int)(cfg->drone_view_depth / cfg->map_scale) + 1 != D2D_LOCAL) {
        g_create_err = "only drone_view_depth // map_scale == 8 (33x33 local map) is supported"; return D2D_ERR_INVALID;
    }
    if (cfg->n_rays <= 0 || cfg->n_rays > 1024 || cfg->n_targets < 1 || cfg->n_targets > D2D_MAX_TARGETS ||
        cfg->n_u > D2D_MAX_U || cfg->n_samp > D2D_MAX_SAMP || cfg->n_way > D2D_MAX_WAY || cfg->n_yaw > D2D_MAX_YAW ||
        cfg->n_owl_u < 0 || cfg->n_owl_u > D2D_MAX_OWL_U || cfg->owl_repeat < 0) {
        g_create_err = "table size out of range"; return D2D_ERR_INVALID;
    }
    if ((cfg->oxford & D2D_POLICY_OXFORD) && cfg->n_yaw > D2D_OX_MAX_YAW) {
        g_create_err = "Oxford policy: at most 8 candidate yaw rates (the reference has 6, yaw_planner.py:65)"; return D2D_ERR_INVALID;
    }
    if (cfg->var_cam != 0.0 && cfg->envs_per_block > 0) {
        g_create_err = "var_cam != 0 (noisy measurements) is only implemented on the default warp-per-env kernels (envs_per_block = 0)";
        return D2D_ERR_INVALID;
    }
    d2d_handle *h = new d2d_handle();
    h->cfg = *cfg;
    cudaError_t ce = cudaSetDevice(cfg->device);
    if (ce != cudaSuccess) { g_create_err = std::string("cudaSetDevice: ") + cudaGetErrorString(ce); delete h; return D2D_ERR_CUDA; }
    const int B = cfg->num_envs, N = cfg->num_agents;
    const int Bpad = (B + 15) / 16 * 16;
    const int NP = (N > 0 ? N : 1);
    h->B = B; h->Bpad = Bpad; h->N = N; h->NP = NP; h->HW = (NP + 31) / 32;
    // envs per block / threads: E*n_rays ray items per block, one per thread when it fits
    int E = cfg->envs_per_block;
    if (E != 4 && E != 8 && E != 16) E = 8;
    while (E > 4 && (size_t)E * cfg->n_rays > 1024) E /= 2;   // keep >= 1 thread per ray when possible
    h->E = E;
    int T = (E * cfg->n_rays + 31) / 32 * 32;
    const int maxT = (E * 50 + 31) / 32 * 32;   // launch bound of the instantiation (see d2d_step_fused_kernel)
    if (T > maxT) T = maxT;
    if (T < 64) T = 64;
    h->T = T;

    size_t cur = 0;
    DevP &P = h->P;
    memset(&P, 0, sizeof(P));
    const int64_t sB = Bpad;
#define SHP(...) {__VA_ARGS__}
    size_t o_apos = add_buf(h, cur, "agent_pos", D2D_F64, 3, SHP(B, N, 2), SHP(NP * 2, 2, 1), (size_t)sB * NP * 2,
                            env_rows(NP * 16));
    size_t o_apref = add_buf(h, cur, "agent_pref", D2D_F64, 3, SHP(B, N, 2), SHP(NP * 2, 2, 1), (size_t)sB * NP * 2,
                            env_rows(NP * 16));
    size_t o_apos0 = add_buf(h, cur, "agent_pos0", D2D_F64, 3, SHP(B, N, 2), SHP(NP * 2, 2, 1), (size_t)sB * NP * 2,
                            env_rows(NP * 16));
    size_t o_apref0 = add_buf(h, cur, "agent_pref0", D2D_F64, 3, SHP(B, N, 2), SHP(NP * 2, 2, 1), (size_t)sB * NP * 2,
                            env_rows(NP * 16));
    const bool rvo = cfg->motion_profile == D2D_MOTION_RVO;
    const size_t vel_elems = rvo ? (size_t)sB * NP * 2 : 2;
    size_t o_avel = add_buf(h, cur, "agent_vel", D2D_F64, 3, SHP(B, N, 2), SHP(NP * 2, 2, 1), vel_elems,
                            rvo ? env_rows(NP * 16) : NOT_ENV_STATE);
    size_t o_avel0 = add_buf(h, cur, "agent_vel0", D2D_F64, 3, SHP(B, N, 2), SHP(NP * 2, 2, 1), vel_elems,
                            rvo ? env_rows(NP * 16) : NOT_ENV_STATE);
    size_t o_aveln = add_buf(h, cur, "agent_vel_next", D2D_F64, 3, SHP(B, N, 2), SHP(NP * 2, 2, 1), vel_elems, NOT_ENV_STATE);
    size_t o_robs = add_buf(h, cur, "rvo_obstacles", D2D_F64, 3, SHP(B, D2D_RVO_MAX_OBS, 3), SHP(D2D_RVO_MAX_OBS * 3, 3, 1),
                            rvo ? (size_t)sB * D2D_RVO_MAX_OBS * 3 : 4,
                            rvo ? env_rows(D2D_RVO_MAX_OBS * 3 * 8) : NOT_ENV_STATE);
    size_t o_rnobs = add_buf(h, cur, "rvo_num_obstacles", D2D_I32, 1, SHP(B), SHP(1), sB,
                            rvo ? env_rows(4) : NOT_ENV_STATE);
    size_t o_arad = add_buf(h, cur, "agent_radius", D2D_F64, 2, SHP(B, N), SHP(NP, 1), (size_t)sB * NP,
                            env_rows(NP * 8));
    size_t o_trad0 = add_buf(h, cur, "tracker_radius0", D2D_F64, 2, SHP(B, N), SHP(NP, 1), (size_t)sB * NP,
                            env_rows(NP * 8));
    size_t o_gt = add_buf(h, cur, "gt_rows", D2D_I64, 2, SHP(B, D2D_GRID), SHP(D2D_GRID, 1), (size_t)sB * D2D_GRID,
                            env_rows(D2D_GT_ROW_BYTES));
    size_t o_bel = add_buf(h, cur, "belief", D2D_U8, 3, SHP(B, D2D_GRID, D2D_GRID), SHP(D2D_BELIEF_STRIDE, D2D_GRID, 1),
                           (size_t)sB * D2D_BELIEF_STRIDE, env_rows(D2D_BELIEF_STRIDE));
    // per-env scalar state: one 128-byte EnvRec per env; its fields are exposed as strided [B] views
    size_t o_rec = add_buf(h, cur, "env_records", D2D_U8, 2, SHP(B, (int64_t)sizeof(EnvRec)), SHP((int64_t)sizeof(EnvRec), 1),
                           (size_t)sB * sizeof(EnvRec), env_rows(sizeof(EnvRec)));
    {
        const size_t rb = (size_t)sB * sizeof(EnvRec);
        const int64_t s8 = sizeof(EnvRec) / 8, s4 = sizeof(EnvRec) / 4, s1 = sizeof(EnvRec);
#define RECF(name, field, dt, st) add_view(h, name, dt, 1, SHP(B), SHP(st), o_rec + offsetof(EnvRec, field), rb - offsetof(EnvRec, field))
        RECF("drone_x", px, D2D_F64, s8); RECF("drone_y", py, D2D_F64, s8); RECF("drone_yaw", yaw, D2D_F64, s8);
        RECF("drone_vx", vx, D2D_F64, s8); RECF("drone_vy", vy, D2D_F64, s8);
        RECF("target_x", tgx, D2D_F64, s8); RECF("target_y", tgy, D2D_F64, s8);
        RECF("steps", steps, D2D_I32, s4); RECF("state_machine", sm, D2D_I32, s4); RECF("fail_count", fail, D2D_I32, s4);
        RECF("target_cursor", tcur, D2D_I32, s4);
        RECF("tracker_buffer_count", bufc, D2D_I32, s4); RECF("tracker_buffer_ts", bufts, D2D_I32, s4);
        RECF("tracked_agent", tracked, D2D_I32, s4);
        RECF("traj_nseg", nseg, D2D_I32, s4); RECF("traj_cursor", cursor, D2D_I32, s4);
        RECF("obs_ix", obs_ix, D2D_I32, s4); RECF("obs_iy", obs_iy, D2D_I32, s4);
        RECF("pending_reset", pending_reset, D2D_U8, s1); RECF("oxford_fresh", ox_fresh, D2D_U8, s1);
        RECF("owl_fresh", owl_fresh, D2D_U8, s1);
#undef RECF
        add_view(h, "drone_pose0", D2D_F64, 2, SHP(3, B), SHP(1, s8), o_rec + offsetof(EnvRec, p0x), rb - offsetof(EnvRec, p0x));
    }
    size_t o_col = add_buf(h, cur, "collision_flag", D2D_U8, 1, SHP(B), SHP(1), sB, env_rows(1));
    size_t o_dead = add_buf(h, cur, "dead_lock_flag", D2D_U8, 1, SHP(B), SHP(1), sB, env_rows(1));
    size_t o_frz = add_buf(h, cur, "freezing_flag", D2D_U8, 1, SHP(B), SHP(1), sB, env_rows(1));
    size_t o_done = add_buf(h, cur, "done", D2D_U8, 1, SHP(B), SHP(1), sB, env_rows(1));
    size_t o_lm = add_buf(h, cur, "local_map", D2D_U8, 4, SHP(B, 1, D2D_LOCAL, D2D_LOCAL),
                          SHP(D2D_LOCAL_CELLS, D2D_LOCAL_CELLS, D2D_LOCAL, 1), (size_t)sB * D2D_LOCAL_CELLS, env_rows(D2D_LOCAL_CELLS));
    size_t o_yawo = add_buf(h, cur, "yaw_angle", D2D_F32, 2, SHP(B, 1), SHP(1, 1), sB, env_rows(4));
    size_t o_rew = add_buf(h, cur, "reward", D2D_F32, 1, SHP(B), SHP(1), sB, NOT_ENV_STATE);
    size_t o_hit = add_buf(h, cur, "hit", D2D_I8, 2, SHP(B, N), SHP(NP, 1), (size_t)sB * NP, env_rows(NP));
    size_t o_tact = add_buf(h, cur, "tracker_active", D2D_U8, 2, SHP(B, N), SHP(NP, 1), (size_t)sB * NP, env_rows(NP));
    size_t o_tmu = add_buf(h, cur, "tracker_mu", D2D_F64, 3, SHP(B, N, 4), SHP(NP * 4, 4, 1), (size_t)sB * NP * 4,
                            env_rows(NP * 32));
    size_t o_tsg = add_buf(h, cur, "tracker_sigma", D2D_F64, 4, SHP(B, N, 4, 4), SHP(NP * 16, 16, 4, 1), (size_t)sB * NP * 16,
                            env_rows(NP * 128));
    size_t o_trad = add_buf(h, cur, "tracker_radius", D2D_F64, 2, SHP(B, N), SHP(NP, 1), (size_t)sB * NP,
                            env_rows(NP * 8));
    size_t o_tts = add_buf(h, cur, "tracker_ts", D2D_I32, 2, SHP(B, N), SHP(NP, 1), (size_t)sB * NP,
                            env_rows(NP * 4));
    size_t o_coef = add_buf(h, cur, "traj_coeff", D2D_F64, 3, SHP(B, D2D_MAX_SEGMENTS, 6), SHP(D2D_MAX_SEGMENTS * 6, 6, 1),
                            cfg->planner == D2D_PLANNER_PRIMITIVE ? (size_t)sB * D2D_MAX_SEGMENTS * 6 : 16,
                            cfg->planner == D2D_PLANNER_PRIMITIVE ? env_rows(D2D_MAX_SEGMENTS * 6 * 8) : NOT_ENV_STATE);
    size_t o_need = add_buf(h, cur, "need_plan", D2D_U8, 1, SHP(B), SHP(1), sB, env_rows(1));
    size_t o_pok = add_buf(h, cur, "plan_ok", D2D_U8, 1, SHP(B), SHP(1), sB, env_rows(1));
    size_t o_rep = add_buf(h, cur, "replan", D2D_U8, 1, SHP(B), SHP(1), sB, env_rows(1));
    size_t o_tac = add_buf(h, cur, "tmp_active_count", D2D_I32, 1, SHP(B), SHP(1), sB, NOT_ENV_STATE);
    size_t o_tat = add_buf(h, cur, "tmp_active_ts", D2D_I32, 1, SHP(B), SHP(1), sB, NOT_ENV_STATE);
    const bool noisy = cfg->var_cam != 0.0;
    size_t o_rk = add_buf(h, cur, "rng_key", D2D_I32, 2, SHP(B, 624), SHP(624, 1), noisy ? (size_t)sB * 624 : 16,
                            noisy ? env_rows(624 * 4) : NOT_ENV_STATE);
    size_t o_rk0 = add_buf(h, cur, "rng_key0", D2D_I32, 2, SHP(B, 624), SHP(624, 1), noisy ? (size_t)sB * 624 : 16,
                            noisy ? env_rows(624 * 4) : NOT_ENV_STATE);
    size_t o_rp = add_buf(h, cur, "rng_pos", D2D_I32, 2, SHP(4, B), SHP(B, 1), (size_t)4 * sB,      // pos, pos0, has, has0
                          env_rows(4, 4, sB * 4));
    size_t o_rg = add_buf(h, cur, "rng_gauss", D2D_F64, 2, SHP(2, B), SHP(B, 1), (size_t)2 * sB,     // gauss, gauss0
                          env_rows(8, 2, sB * 8));
    size_t o_oxp = add_buf(h, cur, "oxford_program", D2D_U8, 1, SHP((int64_t)sizeof(OxProgram)), SHP(1), sizeof(OxProgram),
                            NOT_ENV_STATE);
    size_t o_oxs = add_buf(h, cur, "oxford_seen_call", D2D_I32, 1, SHP(1), SHP(1),
                           (cfg->oxford & D2D_POLICY_OXFORD) ? (size_t)sB * D2D_OX_SEEN_STRIDE / 2 : 4,   // uint16 [B][2560]
                           (cfg->oxford & D2D_POLICY_OXFORD) ? env_rows(D2D_OX_SEEN_STRIDE * 2) : NOT_ENV_STATE);
    size_t o_oxc = add_buf(h, cur, "oxford_calls", D2D_I32, 1, SHP(B), SHP(1), sB, env_rows(4));
    size_t o_oxt = add_buf(h, cur, "oxford_tables", D2D_F64, 2, SHP(2, D2D_OX_TAB), SHP(D2D_OX_TAB, 1), 2 * D2D_OX_TAB,
                            NOT_ENV_STATE);
    const bool owl = (cfg->oxford & D2D_POLICY_OWL) != 0;
    size_t o_owlU = add_buf(h, cur, "owl_U", D2D_F64, 2, SHP(B, D2D_OWL_BINS), SHP(D2D_OWL_BINS, 1), owl ? (size_t)sB * D2D_OWL_BINS : 2,
                            owl ? env_rows(D2D_OWL_BINS * 8) : NOT_ENV_STATE);
    size_t o_owlq = add_buf(h, cur, "owl_queue_len", D2D_I32, 1, SHP(B), SHP(1), sB, env_rows(4));
    size_t o_owlu = add_buf(h, cur, "owl_queue_value", D2D_F64, 1, SHP(B), SHP(1), sB, env_rows(8));
    size_t o_dacc = add_buf(h, cur, "drone_acc", D2D_F64, 2, SHP(B, 2), SHP(2, 1), (size_t)sB * 2, env_rows(16));
    size_t o_jerk = add_buf(h, cur, "jerk_tables", D2D_U8, 1, SHP((int64_t)sizeof(d2d_jerk_tables)), SHP(1),
                            cfg->planner == D2D_PLANNER_JERK ? sizeof(d2d_jerk_tables) : 16, NOT_ENV_STATE);
    size_t o_stats = add_buf(h, cur, "stats", D2D_I64, 1, SHP(D2D_NUM_STATS), SHP(1), D2D_NUM_STATS, NOT_ENV_STATE);
    size_t o_tab = add_buf(h, cur, "tables", D2D_U8, 1, SHP((int64_t)sizeof(DevTables)), SHP(1), sizeof(DevTables),
                            NOT_ENV_STATE);
    // caller data (+ the stamp slot of the resident gated kernel): not env state
    size_t o_stage = add_buf(h, cur, "actions_staging", D2D_F64, 1, SHP(B), SHP(1), sB + 8, NOT_ENV_STATE);
    size_t o_plan_ws = 0;
    size_t plan_ws_bytes = 0;
    if (cfg->planner == D2D_PLANNER_PRIMITIVE) {
        plan_ws_bytes = d2d_plan_workspace_bytes(cfg->n_u) * (size_t)D2D_PLAN_SLOTS;
        o_plan_ws = add_buf(h, cur, "plan_workspace", D2D_U8, 1, SHP((int64_t)plan_ws_bytes), SHP(1), plan_ws_bytes,
                            NOT_ENV_STATE);
    }
    size_t o_plan_list = add_buf(h, cur, "plan_list", D2D_I32, 1, SHP(B + 8), SHP(1), sB + 8, NOT_ENV_STATE);
    size_t o_plan_over = add_buf(h, cur, "plan_overflow", D2D_I32, 1, SHP(B + 8), SHP(1), sB + 8, NOT_ENV_STATE);
#undef SHP
    if (!build_state_layout(h)) {
        g_create_err = "per-env state: more than " + std::to_string(D2D_CLONE_MAX_FIELDS) + " rows"; delete h; return D2D_ERR_INVALID;
    }
    h->arena_bytes = (cur + 255) / 256 * 256;
    ce = cudaMalloc((void **)&h->arena, h->arena_bytes);
    if (ce != cudaSuccess) {
        g_create_err = std::string("cudaMalloc arena (") + std::to_string(h->arena_bytes) + " B): " + cudaGetErrorString(ce);
        delete h; return D2D_ERR_NOMEM;
    }
    ce = cudaMemset(h->arena, 0, h->arena_bytes);
    if (ce != cudaSuccess) { g_create_err = std::string("cudaMemset: ") + cudaGetErrorString(ce); cudaFree(h->arena); delete h; return D2D_ERR_CUDA; }

    unsigned char *A = h->arena;
    P.B = B; P.N = N; P.NP = NP; P.HW = h->HW;
    P.n_rays = cfg->n_rays; P.planner = cfg->planner; P.trackers = cfg->trackers; P.auto_reset = cfg->auto_reset;
    P.n_targets = cfg->n_targets; P.n_u = cfg->n_u; P.n_samp = cfg->n_samp; P.n_way = cfg->n_way; P.n_yaw = cfg->n_yaw;
    P.dt = cfg->dt; P.scale = cfg->map_scale; P.inv_scale = 1.0 / cfg->map_scale; P.map_w = cfg->map_w; P.map_h = cfg->map_h;
    P.agent_radius = cfg->agent_radius; P.max_acc = cfg->drone_max_acceleration; P.drone_r = cfg->drone_radius;
    P.max_yaw_speed = cfg->drone_max_yaw_speed; P.depth2 = cfg->drone_view_depth * cfg->drone_view_depth;
    P.fov = cfg->drone_view_range * D2D_DEG2RAD;                 // radians(drone.yaw_range), utils.py:575
    P.max_steps = cfg->max_flight_time / cfg->dt;                // drone_v2.py:89
    P.var_cam = cfg->var_cam; P.max_speed = cfg->drone_max_speed;
    P.view_depth = cfg->drone_view_depth; P.view_range_deg = cfg->drone_view_range;
    // a sample is evaluated only if the previous one was closer than depth: reach = depth + step*sqrt(2) (+ slack)
    P.cull_reach = cfg->drone_view_depth + (cfg->map_scale - 1.0) * 1.4142135623730951 + 1e-3;
    P.ray_a0 = -P.fov / 2; P.ray_da = P.fov / (double)cfg->n_rays;
    P.ox_cos_thresh = cfg->ox_cos_thresh;
    {   // sample m is at most m*(scale-1)*sqrt(2) from the drone; skip the depth test while that is < 0.99*depth
        const double lmax = (cfg->map_scale - 1.0) * 1.4142135623730951;
        int m = 0;
        while ((double)(m + 1) * lmax < 0.99 * cfg->drone_view_depth) m++;
        P.m_far = m + 1;                     // samples 0..m are provably inside the view depth
    }
    memcpy(P.targets, cfg->targets, sizeof(P.targets));
    P.apos = (double2 *)(A + o_apos); P.apref = (double2 *)(A + o_apref);
    P.apos0 = (double2 *)(A + o_apos0); P.apref0 = (double2 *)(A + o_apref0);
    P.arad = (double *)(A + o_arad); P.trk_radius0 = (double *)(A + o_trad0);
    P.motion_rvo = rvo ? 1 : 0;
    P.avel = (double2 *)(A + o_avel); P.avel0 = (double2 *)(A + o_avel0); P.avel_next = (double2 *)(A + o_aveln);
    P.rvo_obs = (double *)(A + o_robs); P.rvo_nobs = (int *)(A + o_rnobs);
    P.gt_rows = (uint64_t *)(A + o_gt); P.belief = A + o_bel;
    P.rec = (EnvRec *)(A + o_rec);
    P.collision = A + o_col; P.dead_lock = A + o_dead; P.freezing = A + o_frz; P.done = A + o_done;
    P.local_map = A + o_lm; P.yaw_obs = (float *)(A + o_yawo); P.reward = (float *)(A + o_rew); P.hit = (int8_t *)(A + o_hit);
    P.trk_active = A + o_tact; P.trk_mu = (double *)(A + o_tmu); P.trk_sigma = (double *)(A + o_tsg);
    P.trk_radius = (double *)(A + o_trad); P.trk_ts = (int *)(A + o_tts);
    P.traj_coeff = (double *)(A + o_coef);
    P.need_plan = A + o_need; P.plan_ok = A + o_pok; P.replan = A + o_rep;
    P.ox_seen = (cfg->oxford & D2D_POLICY_OXFORD) ? (uint16_t *)(A + o_oxs) : nullptr;
    P.owl_U = owl ? (double *)(A + o_owlU) : nullptr; P.owl_q = (int *)(A + o_owlq); P.owl_u = (double *)(A + o_owlu);
    P.n_owl_u = cfg->n_owl_u; P.owl_repeat = cfg->owl_repeat;
    P.drone_acc = (double2 *)(A + o_dacc);
    P.jerk = cfg->planner == D2D_PLANNER_JERK ? (const d2d_jerk_tables *)(A + o_jerk) : nullptr;
    P.ox_calls = (int *)(A + o_oxc); P.ox_tab = (const double *)(A + o_oxt); P.ox_last = nullptr;
    P.lm_mirror = nullptr; P.yaw_mirror = nullptr; P.done_mirror = nullptr;
#if defined(D2D_WARP_PROF) || defined(D2D_PLAN_PROF)
    cudaMalloc((void **)&P.prof, (size_t)B * 96); cudaMemset(P.prof, 0, (size_t)B * 96);
#endif
    P.tmp_act_cnt = (int *)(A + o_tac); P.tmp_act_ts = (int *)(A + o_tat);
    P.rng_key = noisy ? (uint32_t *)(A + o_rk) : nullptr; P.rng_key0 = noisy ? (uint32_t *)(A + o_rk0) : nullptr;
    P.rng_pos = (int *)(A + o_rp); P.rng_pos0 = P.rng_pos + sB; P.rng_has = P.rng_pos + 2 * sB; P.rng_has0 = P.rng_pos + 3 * sB;
    P.rng_gauss = (double *)(A + o_rg); P.rng_gauss0 = P.rng_gauss + sB;
    h->ox_prog = (OxProgram *)(A + o_oxp);
    P.stats = (unsigned long long *)(A + o_stats);
    P.tab = (const DevTables *)(A + o_tab);
    P.plan_ws = cfg->planner == D2D_PLANNER_PRIMITIVE ? (A + o_plan_ws) : nullptr;
    P.plan_list = (int *)(A + o_plan_list);
    P.plan_over = (int *)(A + o_plan_over);
    h->stage_actions = (double *)(A + o_stage);

    DevTables tab;
    memset(&tab, 0, sizeof(tab));
    memcpy(tab.u_space, cfg->u_space, sizeof(tab.u_space));
    memcpy(tab.t_samp, cfg->t_samp, sizeof(tab.t_samp)); memcpy(tab.t_samp2, cfg->t_samp2, sizeof(tab.t_samp2));
    memcpy(tab.t_way, cfg->t_way, sizeof(tab.t_way)); memcpy(tab.t_way2, cfg->t_way2, sizeof(tab.t_way2));
    memcpy(tab.t_way_x2, cfg->t_way_x2, sizeof(tab.t_way_x2));
    memcpy(tab.v_yaw_space, cfg->v_yaw_space, sizeof(tab.v_yaw_space));
    // RVO candidate directions np.arange(0, 2*3.14, 0.2) (utils.py:365): element i is 0 + i*0.2; math.cos / math.sin are
    // this host's libm, the same functions the reference calls
    for (int i = 0; i < D2D_RVO_THETAS; i++) { const double th = 0.0 + (double)i * 0.2; tab.rvo_cos[i] = cos(th); tab.rvo_sin[i] = sin(th); }
    // Owl.update_U (yaw_planner.py:181-182): cos / sin of math.radians(d_i), d_i = 0, 10, ..., 350 (this host's libm, as above)
    memcpy(tab.owl_u_space, cfg->owl_u_space, sizeof(tab.owl_u_space));
    for (int i = 0; i < D2D_OWL_BINS; i++) { const double r = (10.0 * i) * (D2D_PI / 180.0); tab.owl_cos[i] = cos(r); tab.owl_sin[i] = sin(r); }
    ce = cudaMemcpy(A + o_tab, &tab, sizeof(tab), cudaMemcpyHostToDevice);
    if (ce != cudaSuccess) { g_create_err = std::string("cudaMemcpy tables: ") + cudaGetErrorString(ce); cudaFree(h->arena); delete h; return D2D_ERR_CUDA; }

    {   // exact value of last_time_observed after k consecutive `+= dt` from 0.0 (cell seen) and from 5.0 (never seen)
        std::vector<double> t(2 * D2D_OX_TAB);
        double v0 = 0.0, v5 = 5.0;
        for (int k = 0; k < D2D_OX_TAB; k++) { t[k] = v0; t[D2D_OX_TAB + k] = v5; v0 = v0 + 1.0 * cfg->dt; v5 = v5 + 1.0 * cfg->dt; }
        ce = cudaMemcpy(A + o_oxt, t.data(), t.size() * 8, cudaMemcpyHostToDevice);
        if (ce != cudaSuccess) { g_create_err = std::string("cudaMemcpy oxford tables: ") + cudaGetErrorString(ce); cudaFree(h->arena); delete h; return D2D_ERR_CUDA; }
    }
    {
        OxProgram prog;
        build_ox_program(&prog, D2D_CELLS);
        ce = cudaMemcpy(A + o_oxp, &prog, sizeof(prog), cudaMemcpyHostToDevice);
        if (ce != cudaSuccess) { g_create_err = std::string("cudaMemcpy oxford program: ") + cudaGetErrorString(ce); cudaFree(h->arena); delete h; return D2D_ERR_CUDA; }
    }
    h->smem_pre = d2d_pre_smem_bytes(E, NP, h->HW);
    h->smem_plan = d2d_plan_smem_bytes(NP, cfg->n_u, cfg->n_samp);
    if (cfg->planner == D2D_PLANNER_PRIMITIVE && h->smem_pre > 227 * 1024) {
        g_create_err = "shared memory per block exceeds 227 KB (Primitive path; lower envs_per_block)";
        cudaFree(h->arena); delete h; return D2D_ERR_INVALID;
    }
    h->smem_step = d2d_step_smem_bytes(E, NP, h->HW);
    if (h->smem_step > 227 * 1024) {
        g_create_err = "shared memory per block exceeds 227 KB (too many agents per env for this envs_per_block)";
        cudaFree(h->arena); delete h; return D2D_ERR_INVALID;
    }
    *out = h;
    return D2D_OK;
}

// A kernel is waiting at its gate for actions that will not come (destroy / re-bind): complete that step with action 0.
static void pipe_release(d2d_handle *h) {
    if (h->pipe_mode == 2 && h->pipe_courier) {      // resident kernel with a courier: stamp "last step, actions = 0"
        const unsigned long long stamp = ((unsigned long long)(h->pipe_seq + 1) << 1) | (1ull << 62);
        __atomic_store_n((unsigned long long *)(h->gate_host + 8), stamp, __ATOMIC_RELEASE);
    } else if (h->pipe_mode == 2 && h->pipe_pub) {   // resident kernel fed by the copy engine: a proper stamp that says "last step"
        memset(h->pipe_pub, 0, (size_t)h->B * 8);
        const unsigned long long stamp = ((unsigned long long)(h->pipe_seq + 1) << 1);
        memcpy(h->pipe_pub + h->B, &stamp, 8);
        cudaMemcpyAsync(h->stage_actions, h->pipe_pub, (size_t)(h->B + 1) * 8, cudaMemcpyHostToDevice, h->copy_stream);
    } else {
        cudaMemsetAsync(h->stage_actions, 0, (size_t)h->B * 8, h->copy_stream);
    }
    cudaStreamSynchronize(h->io_stream);
    h->pipe_inflight = false;
    h->pipe_mode = 0;
    h->pipe_seq += 1;
}

extern "C" int d2d_destroy(d2d_handle *h) {
    if (!h) return D2D_OK;
    cudaSetDevice(h->cfg.device);
    if (h->pipe_inflight) pipe_release(h);   // release the kernel that waits for its actions (the state is going away anyway)
    if (h->pipe_pub) cudaFreeHost(h->pipe_pub);
    if (h->pipe_count) cudaFree(h->pipe_count);
    if (h->dbg_n && getenv("D2D_PIPE_DEBUG"))
        fprintf(stderr, "[d2d pipelined] calls %ld: publish+launch %.2f us, wait %.2f us (%.1f event polls), total %.2f us per call\n",
                h->dbg_n, h->dbg_launch_ns / h->dbg_n * 1e-3, h->dbg_wait_ns / h->dbg_n * 1e-3, (double)h->dbg_polls / h->dbg_n,
                h->dbg_total_ns / h->dbg_n * 1e-3);
    if (h->gate_host) cudaFreeHost((void *)h->gate_host);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->side_stream) cudaStreamDestroy(h->side_stream);
    for (int i = 0; i < 2; i++) if (h->side_ev[i]) cudaEventDestroy(h->side_ev[i]);
    for (int i = 0; i < 3; i++) if (h->pipe_ev[i]) cudaEventDestroy(h->pipe_ev[i]);
    if (h->arena) cudaFree(h->arena);
    if (h->ox_export) cudaFree(h->ox_export);
    if (h->clone_idx) cudaFree(h->clone_idx);
    if (h->clone_ev) cudaEventDestroy(h->clone_ev);
    if (h->wg_tab) cudaFree(h->wg_tab);
    if (h->wg_idx) cudaFree(h->wg_idx);
    if (h->wg_ev) cudaEventDestroy(h->wg_ev);
    if (h->wg_fault) cudaFreeHost((void *)h->wg_fault);
    if (h->wg_claim) cudaFree(h->wg_claim);
    if (h->ep_mem) cudaFree(h->ep_mem);
    if (h->ep_queue) cudaFree(h->ep_queue);
    delete h;
    return D2D_OK;
}

extern "C" int d2d_get_buffer(d2d_handle *h, const char *name, d2d_buffer_info *out) {
    if (!h || !name || !out) return D2D_ERR_INVALID;
    if (std::string(name) == "oxford_last_time_observed") {
        // Oxford.last_time_observed_map (yaw_planner.py:49,95-97) as float64 [B,50,50]: expanded from the compact state by a
        // kernel on the legacy default stream, then synchronised (debug / test accessor, not part of the hot path)
        if (!(h->cfg.oxford & D2D_POLICY_OXFORD)) { h->err = "oxford_last_time_observed: handle was created without the Oxford state"; return D2D_ERR_STATE; }
        CUDA_TRY(h, cudaSetDevice(h->cfg.device));
        if (!h->ox_export) CUDA_TRY(h, cudaMalloc((void **)&h->ox_export, (size_t)h->B * D2D_CELLS * 8));
        CUDA_TRY(h, cudaDeviceSynchronize());
        d2d_oxford_export_kernel<<<h->B, 256>>>(h->P, h->ox_export);
        h->launches++;
        CUDA_TRY(h, cudaDeviceSynchronize());
        out->dev_ptr = h->ox_export; out->nbytes = (int64_t)h->B * D2D_CELLS * 8; out->dtype = D2D_F64; out->ndim = 3;
        out->shape[0] = h->B; out->shape[1] = D2D_GRID; out->shape[2] = D2D_GRID; out->shape[3] = 1;
        out->strides[0] = D2D_CELLS; out->strides[1] = D2D_GRID; out->strides[2] = 1; out->strides[3] = 1;
        return D2D_OK;
    }
    {   // the episode log's buffers live outside the arena (allocated by d2d_enable_episode_log)
        const std::string n(name);
        if (n == "episode_log" || n == "episode_log_head" || n == "world_seed") {
            if (!h->ep_mem) { h->err = "d2d_get_buffer(" + n + "): the episode log is not enabled"; return D2D_ERR_STATE; }
            const bool recs = n == "episode_log", hd = n == "episode_log_head";
            out->dev_ptr = recs ? (void *)h->ep.rec : hd ? (void *)h->ep.head : (void *)h->ep.world_seed;
            out->dtype = recs ? D2D_U8 : D2D_I64;
            out->ndim = recs ? 2 : 1;
            out->shape[0] = recs ? h->ep.capacity : hd ? 4 : h->B;
            out->shape[1] = recs ? (int64_t)sizeof(d2d_episode_record) : 1; out->shape[2] = 1; out->shape[3] = 1;
            out->strides[0] = recs ? (int64_t)sizeof(d2d_episode_record) : 1;
            out->strides[1] = 1; out->strides[2] = 1; out->strides[3] = 1;
            out->nbytes = recs ? h->ep.capacity * (int64_t)sizeof(d2d_episode_record) : out->shape[0] * 8;
            return D2D_OK;
        }
    }
#if defined(D2D_WARP_PROF) || defined(D2D_PLAN_PROF)
    if (std::string(name) == "warp_prof") {
        out->dev_ptr = h->P.prof; out->nbytes = (int64_t)h->B * 96; out->dtype = D2D_I64; out->ndim = 2;
        out->shape[0] = h->B; out->shape[1] = 12; out->shape[2] = 1; out->shape[3] = 1;
        out->strides[0] = 12; out->strides[1] = 1; out->strides[2] = 1; out->strides[3] = 1;
        return D2D_OK;
    }
#endif
    for (const BufDesc &b : h->bufs) {
        if (b.name == name) {
            out->dev_ptr = h->arena + b.offset; out->nbytes = (int64_t)b.nbytes; out->dtype = b.dtype; out->ndim = b.ndim;
            for (int i = 0; i < 4; i++) { out->shape[i] = b.shape[i]; out->strides[i] = b.strides[i]; }
            return D2D_OK;
        }
    }
    h->err = std::string("unknown buffer: ") + name;
    return D2D_ERR_INVALID;
}

// ------------------------------------------------------------------------------------------ world upload
extern "C" int d2d_set_world(d2d_handle *h, int32_t first_env, int32_t count, const double *agent_pos,
                             const double *agent_pref, const double *agent_radius, const double *tracker_radius,
                             const uint8_t *gt_grid, const double *drone_pose) {
    if (!h) return D2D_ERR_INVALID;
    if (first_env < 0 || count <= 0 || first_env + count > h->B || !gt_grid || !drone_pose ||
        (h->N > 0 && (!agent_pos || !agent_pref || !agent_radius || !tracker_radius))) {
        h->err = "d2d_set_world: bad range or null array"; return D2D_ERR_INVALID;
    }
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const DevP &P = h->P;
    const int N = h->N, NP = h->NP;
    const size_t e0 = (size_t)first_env;
    if (N > 0) {   // NP == N, rows are dense
        CUDA_TRY(h, cudaMemcpy(P.apos0 + e0 * NP, agent_pos, (size_t)count * N * 16, cudaMemcpyHostToDevice));
        CUDA_TRY(h, cudaMemcpy(P.apref0 + e0 * NP, agent_pref, (size_t)count * N * 16, cudaMemcpyHostToDevice));
        CUDA_TRY(h, cudaMemcpy(P.arad + e0 * NP, agent_radius, (size_t)count * N * 8, cudaMemcpyHostToDevice));
        CUDA_TRY(h, cudaMemcpy(P.trk_radius0 + e0 * NP, tracker_radius, (size_t)count * N * 8, cudaMemcpyHostToDevice));
    }
    std::vector<uint64_t> rows((size_t)count * D2D_GRID);
    for (int c = 0; c < count; c++)
        for (int i = 0; i < D2D_GRID; i++) {
            uint64_t bits = 0;
            for (int j = 0; j < D2D_GRID; j++)
                if (gt_grid[((size_t)c * D2D_GRID + i) * D2D_GRID + j] == 1) bits |= (1ull << j);
            rows[(size_t)c * D2D_GRID + i] = bits;
        }
    CUDA_TRY(h, cudaMemcpy(P.gt_rows + e0 * D2D_GRID, rows.data(), rows.size() * 8, cudaMemcpyHostToDevice));
    // reset pose -> the p0x, p0y, p0yaw fields of the env records (24 contiguous bytes per 128-byte record)
    CUDA_TRY(h, cudaMemcpy2D(&P.rec[e0].p0x, sizeof(EnvRec), drone_pose, 24, 24, (size_t)count, cudaMemcpyHostToDevice));
    // reset exactly those envs
    std::vector<uint8_t> mask((size_t)h->B, 0);
    for (int c = 0; c < count; c++) mask[e0 + c] = 1;
    uint8_t *dmask = nullptr;
    CUDA_TRY(h, cudaMalloc((void **)&dmask, (size_t)h->B));
    cudaError_t ce = cudaMemcpy(dmask, mask.data(), (size_t)h->B, cudaMemcpyHostToDevice);
    if (ce == cudaSuccess) {
        d2d_reset_kernel<<<h->B, 128>>>(P, dmask);
        h->launches++;
        ce = cudaDeviceSynchronize();
    }
    cudaFree(dmask);
    if (ce != cudaSuccess) { h->err = std::string("d2d_set_world reset: ") + cudaGetErrorString(ce); return D2D_ERR_CUDA; }
    h->world_set = true;
    h->mir_stale = true;
    return D2D_OK;
}

extern "C" int d2d_set_rng(d2d_handle *h, int32_t first_env, int32_t count, const uint32_t *key, const int32_t *pos,
                           const int32_t *has_gauss, const double *gauss) {
    if (!h || !key || !pos || !has_gauss || !gauss || first_env < 0 || count <= 0 || first_env + count > h->B) {
        if (h) h->err = "d2d_set_rng: bad argument";
        return D2D_ERR_INVALID;
    }
    if (h->cfg.var_cam == 0.0) return D2D_OK;     // the stream has no observable effect without measurement noise
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const DevP &P = h->P;
    const size_t e0 = (size_t)first_env, n = (size_t)count;
    CUDA_TRY(h, cudaMemcpy(P.rng_key0 + e0 * 624, key, n * 624 * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(P.rng_key + e0 * 624, key, n * 624 * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(P.rng_pos0 + e0, pos, n * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(P.rng_pos + e0, pos, n * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(P.rng_has0 + e0, has_gauss, n * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(P.rng_has + e0, has_gauss, n * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(P.rng_gauss0 + e0, gauss, n * 8, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(P.rng_gauss + e0, gauss, n * 8, cudaMemcpyHostToDevice));
    h->rng_set = true;
    return D2D_OK;
}

extern "C" int d2d_set_rvo(d2d_handle *h, int32_t first_env, int32_t count, const double *agent_vel, const double *obstacles,
                           const int32_t *num_obstacles, int32_t max_obstacles) {
    if (!h || first_env < 0 || count <= 0 || first_env + count > h->B || !num_obstacles || max_obstacles < 0 ||
        max_obstacles > D2D_RVO_MAX_OBS || (h->N > 0 && !agent_vel) || (max_obstacles > 0 && !obstacles)) {
        if (h) h->err = "d2d_set_rvo: bad argument (at most 16 obstacles per env)";
        return D2D_ERR_INVALID;
    }
    if (!h->P.motion_rvo) { h->err = "d2d_set_rvo: handle was created with motion_profile = CVM"; return D2D_ERR_STATE; }
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const DevP &P = h->P;
    const size_t e0 = (size_t)first_env;
    if (h->N > 0) {
        CUDA_TRY(h, cudaMemcpy(P.avel0 + e0 * h->NP, agent_vel, (size_t)count * h->N * 16, cudaMemcpyHostToDevice));
        CUDA_TRY(h, cudaMemcpy(P.avel + e0 * h->NP, agent_vel, (size_t)count * h->N * 16, cudaMemcpyHostToDevice));
    }
    std::vector<double> ob((size_t)count * D2D_RVO_MAX_OBS * 3, 0.0);
    std::vector<int> nob((size_t)count);
    for (int c = 0; c < count; c++) {
        const int m = num_obstacles[c];
        if (m < 0 || m > max_obstacles) { h->err = "d2d_set_rvo: num_obstacles out of range"; return D2D_ERR_INVALID; }
        nob[c] = m;
        for (int q = 0; q < m * 3; q++) ob[(size_t)c * D2D_RVO_MAX_OBS * 3 + q] = obstacles[((size_t)c * max_obstacles) * 3 + q];
    }
    CUDA_TRY(h, cudaMemcpy(P.rvo_obs + e0 * D2D_RVO_MAX_OBS * 3, ob.data(), ob.size() * 8, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(P.rvo_nobs + e0, nob.data(), nob.size() * 4, cudaMemcpyHostToDevice));
    h->rvo_set = true;
    return D2D_OK;
}

extern "C" int d2d_set_jerk_tables(d2d_handle *h, const d2d_jerk_tables *tables) {
    if (!h || !tables) return D2D_ERR_INVALID;
    if (h->cfg.planner != D2D_PLANNER_JERK) { h->err = "d2d_set_jerk_tables: handle was not created with planner = D2D_PLANNER_JERK"; return D2D_ERR_STATE; }
    for (int i = 0; i < D2D_JERK_H; i++) {
        if (tables->times[i] <= 0 || tables->times[i] > D2D_JERK_MAXT) { h->err = "d2d_set_jerk_tables: times out of range"; return D2D_ERR_INVALID; }
        for (int m = 0; m < 144; m++) if (tables->tie_order[m][i] >= D2D_JERK_H) { h->err = "d2d_set_jerk_tables: bad tie order"; return D2D_ERR_INVALID; }
    }
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    CUDA_TRY(h, cudaMemcpy((void *)h->P.jerk, tables, sizeof(d2d_jerk_tables), cudaMemcpyHostToDevice));
    h->jerk_set = true;
    return D2D_OK;
}

extern "C" int d2d_reset(d2d_handle *h, const uint8_t *mask_dev, void *stream) {
    if (!h) return D2D_ERR_INVALID;
    D2D_NO_PIPE(h);
    if (!h->world_set) { h->err = "d2d_reset before d2d_set_world"; return D2D_ERR_STATE; }
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    d2d_reset_kernel<<<h->B, 128, 0, (cudaStream_t)stream>>>(h->P, mask_dev);
    h->launches++;
    CUDA_TRY(h, cudaGetLastError());
    h->mir_stale = true;          // the eager reset rewrites the device observation only
    return D2D_OK;
}

__global__ void d2d_request_reset_kernel(const DevP P, const uint8_t *__restrict__ mask) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < P.B && (!mask || mask[e])) P.rec[e].pending_reset = 1;
}

extern "C" int d2d_request_reset(d2d_handle *h, const uint8_t *mask_dev, void *stream) {
    if (!h) return D2D_ERR_INVALID;
    D2D_NO_PIPE(h);
    if (!h->world_set) { h->err = "d2d_request_reset before d2d_set_world"; return D2D_ERR_STATE; }
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    d2d_request_reset_kernel<<<(h->B + 255) / 256, 256, 0, (cudaStream_t)stream>>>(h->P, mask_dev);
    h->launches++;
    CUDA_TRY(h, cudaGetLastError());
    return D2D_OK;
}

// pinned (page-locked, mapped) host pointer -> the address kernels can store through; null on failure
static void *mirror_dev_ptr(d2d_handle *h, void *host, const char *what) {
    cudaPointerAttributes at;
    cudaError_t ce = cudaPointerGetAttributes(&at, host);
    if (ce != cudaSuccess || at.type != cudaMemoryTypeHost || !at.devicePointer) {
        cudaGetLastError();
        h->err = std::string("d2d_bind_host_mirror: ") + what + " is not pinned host memory (cudaHostAlloc / cudaHostRegister)";
        return nullptr;
    }
    return at.devicePointer;
}

extern "C" int d2d_bind_host_mirror(d2d_handle *h, uint8_t *local_map_host, float *yaw_host, uint8_t *done_host) {
    if (!h) return D2D_ERR_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    CUDA_TRY(h, cudaDeviceSynchronize());             // no kernel may still be storing through the old mirror
    void *dl = nullptr, *dy = nullptr, *dd = nullptr;
    if (local_map_host) {
        if (((uintptr_t)local_map_host & 3) != 0) { h->err = "d2d_bind_host_mirror: local_map_host must be 4-byte aligned"; return D2D_ERR_INVALID; }
        if (!(dl = mirror_dev_ptr(h, local_map_host, "local_map_host"))) return D2D_ERR_INVALID;
    }
    if (yaw_host && !(dy = mirror_dev_ptr(h, yaw_host, "yaw_host"))) return D2D_ERR_INVALID;
    if (done_host && !(dd = mirror_dev_ptr(h, done_host, "done_host"))) return D2D_ERR_INVALID;
    h->P.lm_mirror = (uint8_t *)dl; h->P.yaw_mirror = (float *)dy; h->P.done_mirror = (uint8_t *)dd;
    h->mir_lm = local_map_host; h->mir_yaw = yaw_host; h->mir_done = done_host;
    h->mir_stale = true;
    return D2D_OK;
}

extern "C" int d2d_set_drone_pose(d2d_handle *h, const double *pose_host, void *stream) {
    if (!h || !pose_host) return D2D_ERR_INVALID;
    D2D_NO_PIPE(h);
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    double *tmp = nullptr;
    CUDA_TRY(h, cudaMalloc((void **)&tmp, (size_t)h->B * 24));
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t ce = cudaMemcpyAsync(tmp, pose_host, (size_t)h->B * 24, cudaMemcpyHostToDevice, st);
    if (ce == cudaSuccess) {
        d2d_set_pose_kernel<<<(h->B + 255) / 256, 256, 0, st>>>(h->P, tmp);
        h->launches++;
        ce = cudaStreamSynchronize(st);
    }
    cudaFree(tmp);
    if (ce != cudaSuccess) { h->err = std::string("d2d_set_drone_pose: ") + cudaGetErrorString(ce); return D2D_ERR_CUDA; }
    return D2D_OK;
}

// ------------------------------------------------------------------------------------------ step
template <int E>
static int launch_fused(d2d_handle *h, const double *actions, cudaStream_t st) {
    const int rc = ensure_smem_attr(h, (const void *)d2d_step_fused_kernel<E>, "fused");
    if (rc != D2D_OK) return rc;
    const int grid = (h->B + E - 1) / E;
    d2d_step_fused_kernel<E><<<grid, h->T, h->smem_step, st>>>(h->P, actions);
    h->launches++;
    return D2D_OK;
}

template <int WPB, int MINB, bool ILP2, bool GATED>
static int launch_fused_warp_io(d2d_handle *h, const double *actions, cudaStream_t st) {
    const size_t smem = (size_t)WPB * d2d_warp_slice_bytes(h->NP, h->HW, GATED ? D2D_FUSED_WARP_EXTRA : 0);
    if (smem > 227 * 1024) { h->err = "warp-per-env kernel: shared memory per block exceeds 227 KB"; return D2D_ERR_INVALID; }
    const int rc = ensure_smem_attr(h, (const void *)d2d_step_fused_warp_kernel<WPB, MINB, ILP2, GATED>, "fused warp");
    if (rc != D2D_OK) return rc;
    d2d_step_fused_warp_kernel<WPB, MINB, ILP2, GATED><<<(h->B + WPB - 1) / WPB, WPB * 32, smem, st>>>(h->P, actions);
    h->launches++;
    return D2D_OK;
}
__global__ void d2d_fill_sentinel_kernel(unsigned long long *p, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = D2D_ACTION_SENTINEL;
}

// d2d_step_pipelined sets P.gate -> the GATED instantiation; everything else runs the plain one
template <int WPB, int MINB, bool ILP2>
static int launch_fused_warp(d2d_handle *h, const double *actions, cudaStream_t st) {
    if (h->P.gate) return launch_fused_warp_io<WPB, MINB, ILP2, true>(h, actions, st);
    return launch_fused_warp_io<WPB, MINB, ILP2, false>(h, actions, st);
}

static int step_primitive(d2d_handle *h, const double *actions, cudaStream_t st);

template <int WPB>
static int launch_jerk_warp(d2d_handle *h, const double *actions, cudaStream_t st) {
    const size_t smem = (size_t)WPB * d2d_warp_slice_bytes(h->NP, h->HW, d2d_jerk_warp_extra(h->NP));
    if (smem > 227 * 1024) { h->err = "Jerk_Primitive step kernel: shared memory per block exceeds 227 KB"; return D2D_ERR_INVALID; }
    const int rc = ensure_smem_attr(h, (const void *)d2d_step_jerk_warp_kernel<WPB>, "jerk warp");
    if (rc != D2D_OK) return rc;
    d2d_step_jerk_warp_kernel<WPB><<<(h->B + WPB - 1) / WPB, WPB * 32, smem, st>>>(h->P, actions);
    h->launches++;
    return D2D_OK;
}

// The episode log behind a step (and, with a seed queue, the generation of the worlds it handed out).  Nothing while the
// log is disabled.
static int log_step(d2d_handle *h, cudaStream_t st) {
    if (!h->ep_mem) return D2D_OK;
    d2d_episode_log_kernel<<<h->ep_blocks, D2D_EP_THREADS, 0, st>>>(h->P, h->ep);
    h->launches++;
    if (h->ep_qlen > 0) {
        const int blocks = (h->B + D2D_WG_WARPS - 1) / D2D_WG_WARPS;
        d2d_worldgen_list_kernel<<<blocks < 4 * 148 ? blocks : 4 * 148, D2D_WG_WARPS * 32, 0, st>>>(
            h->P, h->wg_tab, h->ep.gen_env, h->ep.gen_key, h->ep.gen_count, h->wg_fault_dev, h->wg_claim);
        h->launches++;
    }
    CUDA_TRY(h, cudaGetLastError());
    return D2D_OK;
}

static int step_impl(d2d_handle *h, const double *actions_dev, void *stream);

extern "C" int d2d_step(d2d_handle *h, const double *actions_dev, void *stream) {
    const int rc = step_impl(h, actions_dev, stream);
    return rc != D2D_OK ? rc : log_step(h, (cudaStream_t)stream);
}

static int step_impl(d2d_handle *h, const double *actions_dev, void *stream) {
    if (!h || !actions_dev) return D2D_ERR_INVALID;
    D2D_NO_PIPE(h);
    if (!h->world_set) { h->err = "d2d_step before d2d_set_world"; return D2D_ERR_STATE; }
    if (h->cfg.var_cam != 0.0 && !h->rng_set) { h->err = "var_cam != 0: d2d_set_rng must provide the np.random stream state"; return D2D_ERR_STATE; }
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    if (h->P.motion_rvo) {      // RVO.RVO_update (drone_v2.py:169-171) for every env, before Agent.step
        if (!h->rvo_set) { h->err = "motion_profile = RVO: d2d_set_rvo must provide velocities and obstacles"; return D2D_ERR_STATE; }
        const size_t sm = d2d_rvo_smem_bytes(h->N);
        const int rca = ensure_smem_attr(h, (const void *)d2d_rvo_kernel, "rvo");
        if (rca != D2D_OK) return rca;
        d2d_rvo_kernel<<<h->B, d2d_rvo_warps(h->N) * 32, sm, st>>>(h->P);
        h->launches++;
    }
    const int epb = h->cfg.envs_per_block;
    if (h->cfg.planner == D2D_PLANNER_NOMOVE && epb <= 0) {
        // default: one warp per env, single copy of the ray body (smallest code: the kernel is instruction-cache
        // sensitive once several waves de-phase the warps; measured equal to the 2-rays-per-lane variant at one wave)
        rc = launch_fused_warp<4, 7, false>(h, actions_dev, st);
    } else if (h->cfg.planner == D2D_PLANNER_NOMOVE && epb == 1) {
        rc = launch_fused_warp<4, 7, true>(h, actions_dev, st);
    } else if (h->cfg.planner == D2D_PLANNER_NOMOVE && epb == 2) {
        rc = launch_fused_warp<4, 7, false>(h, actions_dev, st);
    } else if (h->cfg.planner == D2D_PLANNER_NOMOVE && epb == 3) {
        rc = launch_fused_warp<7, 4, true>(h, actions_dev, st);
    } else if (h->cfg.planner == D2D_PLANNER_NOMOVE) {
        switch (h->E) {
            case 4: rc = launch_fused<4>(h, actions_dev, st); break;
            case 16: rc = launch_fused<16>(h, actions_dev, st); break;
            default: rc = launch_fused<8>(h, actions_dev, st); break;
        }
    } else if (h->cfg.planner == D2D_PLANNER_JERK) {
        if (!h->jerk_set) { h->err = "planner = Jerk_Primitive: d2d_set_jerk_tables must provide the heading tables"; return D2D_ERR_STATE; }
        rc = launch_jerk_warp<4>(h, actions_dev, st);
    } else {
        rc = step_primitive(h, actions_dev, st);
    }
    if (rc != D2D_OK) return rc;
    CUDA_TRY(h, cudaGetLastError());
    return D2D_OK;
}

static int launch_prim_warp_entry(d2d_handle *h, const double *actions, cudaStream_t st, double *ox_next);

extern "C" int d2d_step_plan_oxford(d2d_handle *h, const double *actions_dev, double *next_actions_dev, void *stream) {
    if (!h || !actions_dev || !next_actions_dev) return D2D_ERR_INVALID;
    D2D_NO_PIPE(h);
    if (!h->world_set) { h->err = "d2d_step_plan_oxford before d2d_set_world"; return D2D_ERR_STATE; }
    if (!(h->cfg.oxford & D2D_POLICY_OXFORD)) { h->err = "d2d_step_plan_oxford: handle was created without the Oxford state (cfg.oxford & 1)"; return D2D_ERR_STATE; }
    if (h->cfg.var_cam != 0.0 && !h->rng_set) { h->err = "var_cam != 0: d2d_set_rng must provide the np.random stream state"; return D2D_ERR_STATE; }
    if (h->cfg.planner != D2D_PLANNER_PRIMITIVE || h->cfg.envs_per_block > 0 || h->P.motion_rvo) {
        // nothing to overlap (or a path made of other kernels): the two calls this entry point stands for
        int rc = step_impl(h, actions_dev, stream);
        if (rc == D2D_OK) rc = d2d_plan_oxford(h, next_actions_dev, stream);
        return rc != D2D_OK ? rc : log_step(h, (cudaStream_t)stream);
    }
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const int rc = launch_prim_warp_entry(h, actions_dev, (cudaStream_t)stream, next_actions_dev);
    if (rc != D2D_OK) return rc;
    CUDA_TRY(h, cudaGetLastError());
    return log_step(h, (cudaStream_t)stream);
}

#define D2D_RESIDENT_WPB 28          // resident gated kernel: one 28-warp block per SM (28 x 148 = 4144 envs in flight)

template <int WPB, int MINB, bool SYNC, bool GATED, bool SMALL = false>
static int launch_rollout(d2d_handle *h, const double *actions, int K, long long stride, cudaStream_t st, unsigned int t_first = 0,
                          int extra_blocks = 0) {
    const size_t smem = (size_t)WPB * d2d_warp_slice_bytes(SMALL ? D2D_SMALL_N : h->NP, SMALL ? 1 : h->HW,
                                                           GATED ? D2D_FUSED_WARP_EXTRA : 0) + (GATED ? 256 : 0);
    if (smem > 227 * 1024) { h->err = "rollout kernel: shared memory per block exceeds 227 KB"; return D2D_ERR_INVALID; }
    const int rc = ensure_smem_attr(h, (const void *)d2d_rollout_warp_kernel<WPB, MINB, SYNC, GATED, SMALL>, "rollout warp");
    if (rc != D2D_OK) return rc;
    static const int sync_every = getenv("D2D_ROLLOUT_SYNC") ? atoi(getenv("D2D_ROLLOUT_SYNC")) : 1;
    d2d_rollout_warp_kernel<WPB, MINB, SYNC, GATED, SMALL><<<(h->B + WPB - 1) / WPB + extra_blocks, WPB * 32, smem, st>>>(
        h->P, actions, K, stride, sync_every > 0 ? sync_every : 1, t_first);
    return D2D_OK;
}

// envs the resident gated kernel can hold at once: every env's warp must be on an SM for the whole run (a warp that waits
// for a later wave's slot would wait forever: the first wave only leaves when the host ends the run)
static int resident_capacity(d2d_handle *h) {
    if (h->resident_capacity >= 0) return h->resident_capacity;
    constexpr int WPB = D2D_RESIDENT_WPB;
    const size_t smem = (size_t)WPB * d2d_warp_slice_bytes(h->NP, h->HW, D2D_FUSED_WARP_EXTRA) + 256;
    int cap = 0, nb = 0, sms = 0;
    if (smem <= 227 * 1024 && ensure_smem_attr(h, (const void *)d2d_rollout_warp_kernel<WPB, 1, false, true>, "rollout warp") == D2D_OK &&
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, d2d_rollout_warp_kernel<WPB, 1, false, true>, WPB * 32, smem) == cudaSuccess &&
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->cfg.device) == cudaSuccess)
        { cap = nb * sms * WPB; h->resident_blocks = nb * sms; }
    else
        cudaGetLastError();
    if (getenv("D2D_PIPE_DEBUG")) fprintf(stderr, "[d2d pipelined] resident kernel: %d blocks/SM x %d SMs, smem %zu B -> capacity %d envs (%s)\n", nb, sms, smem, cap, cudaGetErrorString(cudaPeekAtLastError()));
    h->resident_capacity = cap;
    return cap;
}

extern "C" int d2d_rollout(d2d_handle *h, const double *actions_dev, int32_t num_steps, int64_t action_stride, void *stream) {
    if (!h || !actions_dev || num_steps < 1) return D2D_ERR_INVALID;
    D2D_NO_PIPE(h);
    if (!h->world_set) { h->err = "d2d_rollout before d2d_set_world"; return D2D_ERR_STATE; }
    if (h->cfg.var_cam != 0.0 && !h->rng_set) { h->err = "var_cam != 0: d2d_set_rng must provide the np.random stream state"; return D2D_ERR_STATE; }
    if (h->cfg.planner != D2D_PLANNER_NOMOVE || h->P.motion_rvo || h->cfg.envs_per_block > 0) {
        h->err = "d2d_rollout: NoMove planner, CVM motion profile and the default warp kernels only (use d2d_step)";
        return D2D_ERR_INVALID;
    }
    if (action_stride != 0 && action_stride < h->B) { h->err = "d2d_rollout: action_stride must be 0 or >= num_envs"; return D2D_ERR_INVALID; }
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    // experiment knob (tools/rollout_bench.py): block shape / per-step block barrier of the rollout kernel
    static const int variant = getenv("D2D_ROLLOUT_VARIANT") ? atoi(getenv("D2D_ROLLOUT_VARIANT")) : 0;
    int rc;
    // The resident kernel pays off while the batch is a wave or two of 28-warp blocks (4096 envs: 16.7 vs 21.4 us per step).
    // Large batches keep the SMs busier with the 4-warp blocks of the per-step kernel, which the hardware back-fills one by
    // one (131072 envs, N = 96: 0.75 ms per step against 0.81 ms), so they run the K steps as K per-step launches -- same
    // results either way (tests/test_gpu_rollout.py).
    // ... and so does a handle with an episode log: every step's done bytes must be seen by the log kernel
    if ((variant == 0 && h->B > 2 * 28 * 148) || h->ep_mem) {
        for (int t = 0; t < num_steps; t++) {
            rc = launch_fused_warp<4, 7, false>(h, actions_dev + (size_t)t * (size_t)action_stride, st);
            if (rc == D2D_OK) rc = log_step(h, st);
            if (rc != D2D_OK) return rc;
        }
        CUDA_TRY(h, cudaGetLastError());
        return D2D_OK;
    }
    switch (variant) {
        case 1: rc = launch_rollout<4, 7, false, false>(h, actions_dev, num_steps, action_stride, st); break;
        case 2: rc = launch_rollout<4, 7, true, false>(h, actions_dev, num_steps, action_stride, st); break;
        case 3: rc = launch_rollout<7, 4, true, false>(h, actions_dev, num_steps, action_stride, st); break;
        case 4: rc = launch_rollout<14, 2, true, false>(h, actions_dev, num_steps, action_stride, st); break;
        // the small-crowd form (N <= 32, see d2d_rollout_warp_kernel); larger crowds take the general one
        default: rc = h->N <= D2D_SMALL_N ? launch_rollout<28, 1, true, false, true>(h, actions_dev, num_steps, action_stride, st)
                                          : launch_rollout<28, 1, true, false>(h, actions_dev, num_steps, action_stride, st);
                 break;
    }
    if (rc != D2D_OK) return rc;
    h->launches++;
    CUDA_TRY(h, cudaGetLastError());
    return D2D_OK;
}

extern "C" int d2d_step_host(d2d_handle *h, const double *actions_host, uint8_t *local_map_host, float *yaw_host,
                             uint8_t *done_host, void *stream) {
    if (!h) return D2D_ERR_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    // actions_host == NULL: the actions are already on the device, in the buffer "actions_staging" (written there by
    // d2d_plan_oxford / d2d_plan_gaze when the policy runs on the GPU).
    // Pinned (page-locked, device-mapped) actions are read by the step kernels straight from host memory: every warp
    // requests its env's action at kernel entry and uses it at the end of the step, so the PCIe latency is hidden and no
    // copy has to be enqueued.  Pageable memory goes through the device staging buffer.
    const double *act = actions_host ? nullptr : h->stage_actions;
    if (actions_host) {
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, actions_host) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer)
            act = (const double *)at.devicePointer;
        else
            cudaGetLastError();
    }
    if (!act) {
        CUDA_TRY(h, cudaMemcpyAsync(h->stage_actions, actions_host, (size_t)h->B * 8, cudaMemcpyHostToDevice, st));
        act = h->stage_actions;
    }
    int rc = d2d_step(h, act, stream);
    if (rc != D2D_OK) return rc;
    // a buffer bound as the zero-copy mirror was already written by the step kernels (only the bytes that changed);
    // anything else -- or a mirror that missed an eager reset -- is copied back in full
    const bool fresh = !h->mir_stale;
    if (local_map_host && !(fresh && local_map_host == h->mir_lm))
        CUDA_TRY(h, cudaMemcpyAsync(local_map_host, h->P.local_map, (size_t)h->B * D2D_LOCAL_CELLS, cudaMemcpyDeviceToHost, st));
    if (yaw_host && !(fresh && yaw_host == h->mir_yaw))
        CUDA_TRY(h, cudaMemcpyAsync(yaw_host, h->P.yaw_obs, (size_t)h->B * 4, cudaMemcpyDeviceToHost, st));
    if (done_host && !(fresh && done_host == h->mir_done))
        CUDA_TRY(h, cudaMemcpyAsync(done_host, h->P.done, (size_t)h->B, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(h, cudaStreamSynchronize(st));
    // the full copies above also refreshed whichever mirrors were passed; a bound mirror that was NOT passed stays stale
    if (h->mir_stale && (!h->mir_lm || local_map_host == h->mir_lm) && (!h->mir_yaw || yaw_host == h->mir_yaw) &&
        (!h->mir_done || done_host == h->mir_done))
        h->mir_stale = false;
    return D2D_OK;
}

extern "C" int d2d_bind_host_io(d2d_handle *h, const double *actions_host, uint8_t *local_map_host, float *yaw_host,
                                uint8_t *done_host, void *stream) {
    if (!h) return D2D_ERR_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    if (h->pipe_inflight) pipe_release(h);   // re-binding abandons the pre-launched step: it completes with action 0, then re-sync
    int rc = d2d_bind_host_mirror(h, local_map_host, yaw_host, done_host);     // synchronises the device first
    if (rc != D2D_OK) return rc;
    h->io_bound = false;
    if (!actions_host && !local_map_host && !yaw_host && !done_host) return D2D_OK;
    if (actions_host) {
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, actions_host) != cudaSuccess || at.type != cudaMemoryTypeHost || !at.devicePointer) {
            cudaGetLastError();
            h->err = "d2d_bind_host_io: actions_host is not pinned host memory (cudaHostAlloc / cudaHostRegister)";
            return D2D_ERR_INVALID;
        }
        h->io_actions_dev = (const double *)at.devicePointer;
        h->io_actions_host = actions_host;
    } else {
        h->io_actions_dev = h->stage_actions;
        h->io_actions_host = nullptr;
    }
    if (!h->gate_host) {
        void *p = nullptr;
        CUDA_TRY(h, cudaHostAlloc(&p, 128, cudaHostAllocMapped));
        memset(p, 0, 128);
        h->gate_host = (volatile unsigned int *)p;
        void *dp = nullptr;
        CUDA_TRY(h, cudaHostGetDevicePointer(&dp, p, 0));
        h->gate_dev = (unsigned int *)dp;
        for (int i = 0; i < 3; i++) CUDA_TRY(h, cudaEventCreateWithFlags(&h->pipe_ev[i], cudaEventDisableTiming));
        CUDA_TRY(h, cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));

    }
    h->io_lm = local_map_host; h->io_yaw = yaw_host; h->io_done = done_host;
    h->io_stream = (cudaStream_t)stream;
    h->io_bound = true;
    return D2D_OK;
}

// one synchronous step through the bound buffers (also refreshes a stale mirror with full copies)
static int step_bound_sync(d2d_handle *h, bool plan_oxford = false) {
    const int rc = plan_oxford ? d2d_step_plan_oxford(h, h->io_actions_dev, h->stage_actions, (void *)h->io_stream)
                               : d2d_step(h, h->io_actions_dev, (void *)h->io_stream);
    if (rc != D2D_OK) return rc;
    cudaStream_t st = h->io_stream;
    if (h->mir_stale) {
        if (h->io_lm) CUDA_TRY(h, cudaMemcpyAsync(h->io_lm, h->P.local_map, (size_t)h->B * D2D_LOCAL_CELLS, cudaMemcpyDeviceToHost, st));
        if (h->io_yaw) CUDA_TRY(h, cudaMemcpyAsync(h->io_yaw, h->P.yaw_obs, (size_t)h->B * 4, cudaMemcpyDeviceToHost, st));
        if (h->io_done) CUDA_TRY(h, cudaMemcpyAsync(h->io_done, h->P.done, (size_t)h->B, cudaMemcpyDeviceToHost, st));
    }
    CUDA_TRY(h, cudaStreamSynchronize(st));
    h->mir_stale = false;
    return D2D_OK;
}

extern "C" int d2d_step_bound(d2d_handle *h) {
    if (!h) return D2D_ERR_INVALID;
    if (!h->io_bound) { h->err = "d2d_step_bound before d2d_bind_host_io"; return D2D_ERR_STATE; }
    D2D_NO_PIPE(h);
    return step_bound_sync(h);
}

extern "C" int d2d_step_bound_plan_oxford(d2d_handle *h) {
    if (!h) return D2D_ERR_INVALID;
    if (!h->io_bound) { h->err = "d2d_step_bound_plan_oxford before d2d_bind_host_io"; return D2D_ERR_STATE; }
    if (h->io_actions_dev != h->stage_actions) {
        h->err = "d2d_step_bound_plan_oxford: the actions must come from \"actions_staging\" (bind with actions_host = NULL)";
        return D2D_ERR_STATE;
    }
    D2D_NO_PIPE(h);
    return step_bound_sync(h, true);
}

static int step_pipelined_prelaunch(d2d_handle *h, int32_t prelaunch_next) {
    cudaStream_t st = h->io_stream;
    const double t_in = now_ns();
    const unsigned int seq = h->pipe_seq + 1;            // the step whose actions the caller has just written
    h->P.gate = (unsigned long long *)h->stage_actions; h->P.gate_fault = h->gate_dev + 16;
    int rc = D2D_OK;
    const bool first = !h->pipe_inflight;                 // first step of a pipelined run: nothing was pre-launched
    if (first) {
        // sentinels first; the copy stream must not deliver the actions before they are in place
        d2d_fill_sentinel_kernel<<<(h->B + 255) / 256, 256, 0, st>>>((unsigned long long *)h->stage_actions, h->B);
        h->launches++;
        if (cudaEventRecord(h->pipe_ev[2], st) != cudaSuccess || cudaStreamWaitEvent(h->copy_stream, h->pipe_ev[2], 0) != cudaSuccess)
            rc = D2D_ERR_CUDA;
    }
    // publish: ONE async copy moves the caller's actions over the sentinels in the device staging buffer.  The previous
    // step's kernel has completed (its event was waited for) and has put the sentinels back.  Issued before this step's own
    // kernel in the first-step case, so that blocking launches (CUDA_LAUNCH_BLOCKING, sanitizers) cannot starve it.
    if (rc == D2D_OK && cudaMemcpyAsync(h->stage_actions, h->io_actions_host, (size_t)h->B * 8, cudaMemcpyHostToDevice, h->copy_stream) != cudaSuccess) rc = D2D_ERR_CUDA;
    if (first) {
        if (rc == D2D_OK) rc = launch_fused_warp<4, 7, false>(h, h->stage_actions, st);
        if (rc == D2D_OK && cudaEventRecord(h->pipe_ev[seq & 1], st) != cudaSuccess) rc = D2D_ERR_CUDA;
    }
    h->pipe_seq = seq;
    h->pipe_inflight = false;
    h->pipe_mode = 0;
    if (rc == D2D_OK && prelaunch_next) {                 // the next step starts behind this one and runs up to its gate
        rc = launch_fused_warp<4, 7, false>(h, h->stage_actions, st);
        if (rc == D2D_OK && cudaEventRecord(h->pipe_ev[(seq + 1) & 1], st) != cudaSuccess) rc = D2D_ERR_CUDA;
        if (rc == D2D_OK) { h->pipe_inflight = true; h->pipe_mode = 1; }
    }
    h->P.gate = nullptr; h->P.gate_fault = nullptr;
    if (rc != D2D_OK && h->err.empty()) h->err = std::string("d2d_step_pipelined: ") + cudaGetErrorString(cudaGetLastError());
    if (rc != D2D_OK) { if (h->err.empty()) h->err = "d2d_step_pipelined: launch failed"; return rc; }
    // wait for THIS step only (the pre-launched one keeps running): poll its event, no blocking driver call
    const double t_l = now_ns();
    for (;;) {
        const cudaError_t q = cudaEventQuery(h->pipe_ev[seq & 1]);
        h->dbg_polls++;
        if (q == cudaSuccess) break;
        if (q != cudaErrorNotReady) { h->err = std::string("d2d_step_pipelined: ") + cudaGetErrorString(q); return D2D_ERR_CUDA; }
#if defined(__x86_64__) || defined(__i386__)
        __builtin_ia32_pause();
#endif
    }
    const double t_out = now_ns();
    h->dbg_launch_ns += t_l - t_in; h->dbg_wait_ns += t_out - t_l; h->dbg_total_ns += t_out - t_in; h->dbg_n++;
    if (h->gate_host[16]) { h->err = "d2d_step_pipelined: a step kernel gave up waiting for its actions"; return D2D_ERR_STATE; }
    return D2D_OK;
}

// Resident form: ONE kernel (d2d_rollout_warp_kernel<GATED>) serves the whole run.  Per step the host copies the caller's
// actions plus a stamp word ((sequence number << 1) | another step follows) into the device staging slots with one async
// copy and polls a pinned word the kernel writes when every env has finished the step.  No launch and no stream completion
// on the per-step path; the envs' working sets never leave the SMs between steps.
static int step_pipelined_resident(d2d_handle *h, int32_t more) {
    cudaStream_t st = h->io_stream;
    const double t_in = now_ns();
    const unsigned int seq = h->pipe_seq + 1;
    const bool first = !h->pipe_inflight;
    volatile unsigned long long *stamp_host = (volatile unsigned long long *)(h->gate_host + 8);   // byte 32 of the pinned block
    if (first) {
        // An SM that holds no env block runs the courier block: the kernel then pulls the actions out of the caller's pinned
        // buffer by itself.  Otherwise (the batch fills every SM) the copy engine delivers them, one async copy per step.
        const bool no_courier = getenv("D2D_NO_COURIER") != nullptr;    // test / measurement knob
        h->pipe_courier = !no_courier && (h->B + D2D_RESIDENT_WPB - 1) / D2D_RESIDENT_WPB + 1 <= h->resident_blocks;
        if (!h->pipe_count) CUDA_TRY(h, cudaMalloc((void **)&h->pipe_count, 64));
        if (!h->pipe_courier && !h->pipe_pub) {
            void *p = nullptr;
            CUDA_TRY(h, cudaHostAlloc(&p, (size_t)(h->B + 1) * 8, cudaHostAllocDefault));
            h->pipe_pub = (double *)p;
        }
    }
    const unsigned long long stamp = ((unsigned long long)seq << 1) | (more ? 1ull : 0ull);
    if (!h->pipe_courier) {
        memcpy(h->pipe_pub, h->io_actions_host, (size_t)h->B * 8);
        memcpy(h->pipe_pub + h->B, &stamp, 8);
    }
    int rc = D2D_OK;
    if (first) {
        // sentinels (and a stamp that matches no step) first; nothing may deliver actions before they are in place
        d2d_fill_sentinel_kernel<<<(h->B + 1 + 255) / 256, 256, 0, st>>>((unsigned long long *)h->stage_actions, h->B + 1);
        h->launches++;
        if (cudaMemsetAsync(h->pipe_count, 0, 8, st) != cudaSuccess || cudaEventRecord(h->pipe_ev[2], st) != cudaSuccess ||
            cudaStreamWaitEvent(h->copy_stream, h->pipe_ev[2], 0) != cudaSuccess)
            rc = D2D_ERR_CUDA;
    }
    // publish (before the launch in the first-step case: blocking launches -- sanitizers -- must not starve the kernel)
    if (h->pipe_courier) {
        __atomic_store_n((unsigned long long *)stamp_host, stamp, __ATOMIC_RELEASE);    // the caller's action stores come first
    } else if (rc == D2D_OK && cudaMemcpyAsync(h->stage_actions, h->pipe_pub, (size_t)(h->B + 1) * 8, cudaMemcpyHostToDevice,
                                               h->copy_stream) != cudaSuccess) {
        rc = D2D_ERR_CUDA;
    }
    if (first && rc == D2D_OK) {
        h->P.gate = (unsigned long long *)h->stage_actions; h->P.gate_fault = h->gate_dev + 16;
        h->P.gate_count = h->pipe_count; h->P.gate_done = h->gate_dev;
        h->P.gate_src = h->pipe_courier ? (const unsigned long long *)h->io_actions_dev : nullptr;
        h->P.gate_stamp_host = (const unsigned long long *)(h->gate_dev + 8);
        rc = launch_rollout<D2D_RESIDENT_WPB, 1, false, true>(h, h->stage_actions, 0x7fffffff, 0, st, seq, h->pipe_courier ? 1 : 0);
        h->P.gate = nullptr; h->P.gate_fault = nullptr; h->P.gate_count = nullptr; h->P.gate_done = nullptr;
        h->P.gate_src = nullptr; h->P.gate_stamp_host = nullptr;
        if (rc == D2D_OK) h->launches++;
    }
    if (rc != D2D_OK) {
        if (h->err.empty()) h->err = std::string("d2d_step_pipelined: ") + cudaGetErrorString(cudaGetLastError());
        return rc;
    }
    h->pipe_seq = seq;
    h->pipe_inflight = more != 0;
    h->pipe_mode = more ? 2 : 0;
    const double t_l = now_ns();
    // wait for THIS step: the kernel writes its sequence number once every env's stores are visible
    long polls = 0;
    while (h->gate_host[0] != seq) {
        if (h->gate_host[16]) break;
        if ((++polls & 0xfff) == 0) {
            const cudaError_t q = cudaStreamQuery(st);
            if (q != cudaErrorNotReady && q != cudaSuccess) {
                h->pipe_inflight = false; h->pipe_mode = 0;
                h->err = std::string("d2d_step_pipelined: ") + cudaGetErrorString(q); return D2D_ERR_CUDA;
            }
            if (now_ns() - t_l > 20e9) {
                h->pipe_inflight = false; h->pipe_mode = 0;
                h->err = "d2d_step_pipelined: the resident step kernel did not complete the step within 20 s"; return D2D_ERR_STATE;
            }
        }
#if defined(__x86_64__) || defined(__i386__)
        __builtin_ia32_pause();
#endif
    }
    h->dbg_polls += polls;
    if (!more || h->gate_host[16]) {                     // the run ends: the kernel writes the env records back and leaves
        h->pipe_inflight = false; h->pipe_mode = 0;
        CUDA_TRY(h, cudaStreamSynchronize(st));
    }
    const double t_out = now_ns();
    h->dbg_launch_ns += t_l - t_in; h->dbg_wait_ns += t_out - t_l; h->dbg_total_ns += t_out - t_in; h->dbg_n++;
    if (h->gate_host[16]) { h->gate_host[16] = 0; h->err = "d2d_step_pipelined: the step kernel gave up waiting for its actions"; return D2D_ERR_STATE; }
    return D2D_OK;
}

extern "C" int d2d_step_pipelined(d2d_handle *h, int32_t prelaunch_next) {
    if (!h) return D2D_ERR_INVALID;
    if (!h->io_bound) { h->err = "d2d_step_pipelined before d2d_bind_host_io"; return D2D_ERR_STATE; }
    // The gate lives in the NoMove warp kernels; everything else, and a step that must refresh a stale mirror, runs
    // synchronously (same results, nothing pre-launched).
    // ... and so do batches whose step lasts much longer than the launch + wake-up latency being hidden (~10 us): beyond
    // ~16k envs the gated instantiation's bookkeeping costs more than the overlap returns (measured at 131072 envs: -6 %).
    // An enabled episode log must see every step's done bytes: synchronous path as well.
    const bool can_pipe = h->cfg.planner == D2D_PLANNER_NOMOVE && h->cfg.envs_per_block <= 0 && !h->P.motion_rvo &&
                          h->io_actions_dev != h->stage_actions && (long long)h->B * h->cfg.n_rays <= 16384ll * 50 &&
                          !h->ep_mem;
    if (!can_pipe || (h->mir_stale && !h->pipe_inflight)) {
        D2D_NO_PIPE(h);
        return step_bound_sync(h);
    }
    if (!h->world_set) { h->err = "d2d_step before d2d_set_world"; return D2D_ERR_STATE; }
    if (h->cfg.var_cam != 0.0 && !h->rng_set) { h->err = "var_cam != 0: d2d_set_rng must provide the np.random stream state"; return D2D_ERR_STATE; }
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    // a batch that fits the GPU in one wave is served by the resident kernel; a larger one by one pre-launched kernel per step
    const bool no_resident = getenv("D2D_NO_RESIDENT") != nullptr;      // test / measurement knob
    const int mode = h->pipe_inflight ? h->pipe_mode : ((!no_resident && h->B <= resident_capacity(h)) ? 2 : 1);
    return mode == 2 ? step_pipelined_resident(h, prelaunch_next) : step_pipelined_prelaunch(h, prelaunch_next);
}

extern "C" int d2d_stats(d2d_handle *h, int64_t *out_host, int32_t reset, void *stream) {
    if (!h || !out_host) return D2D_ERR_INVALID;
    D2D_NO_PIPE(h);
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(h, cudaMemcpyAsync(out_host, h->P.stats, D2D_NUM_STATS * 8, cudaMemcpyDeviceToHost, st));
    if (reset) CUDA_TRY(h, cudaMemsetAsync(h->P.stats, 0, D2D_NUM_STATS * 8, st));
    CUDA_TRY(h, cudaStreamSynchronize(st));
    return D2D_OK;
}

// ------------------------------------------------------------------------------------------ per-env state: clone / save / load
extern "C" int d2d_state_layout(const d2d_handle *h, int64_t *bytes_per_env, uint64_t *fingerprint) {
    if (!h) return D2D_ERR_INVALID;
    if (bytes_per_env) *bytes_per_env = h->state_tab.pack_bytes;
    if (fingerprint) *fingerprint = h->state_fingerprint;
    return D2D_OK;
}

// Host index arrays: every entry in [0, num_envs); `written` (dst of a clone, envs of a load) without repeats, and no env
// both read and written.  Checked before anything is enqueued.
static int check_env_indices(d2d_handle *h, const char *what, const int32_t *read, const int32_t *written, int32_t count) {
    std::vector<uint8_t> w(written ? (size_t)h->B : 0, 0);
    for (int32_t i = 0; written && i < count; i++) {
        const int32_t e = written[i];
        if (e < 0 || e >= h->B) { h->err = std::string(what) + ": env index " + std::to_string(e) + " out of range"; return D2D_ERR_INVALID; }
        if (w[e]) { h->err = std::string(what) + ": env " + std::to_string(e) + " is written twice"; return D2D_ERR_INVALID; }
        w[e] = 1;
    }
    for (int32_t i = 0; read && i < count; i++) {
        const int32_t e = read[i];
        if (e < 0 || e >= h->B) { h->err = std::string(what) + ": env index " + std::to_string(e) + " out of range"; return D2D_ERR_INVALID; }
        if (written && w[e]) { h->err = std::string(what) + ": env " + std::to_string(e) + " is both a source and a destination"; return D2D_ERR_INVALID; }
    }
    return D2D_OK;
}

// A packed state buffer must be device memory of the handle's device, 16-B aligned.
static int check_state_ptr(d2d_handle *h, const char *what, const void *p) {
    if (!p) { h->err = std::string(what) + ": null state buffer"; return D2D_ERR_INVALID; }
    if (((uintptr_t)p & 15) != 0) { h->err = std::string(what) + ": the state buffer must be 16-byte aligned"; return D2D_ERR_INVALID; }
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess || at.type != cudaMemoryTypeDevice || at.device != h->cfg.device) {
        cudaGetLastError();
        h->err = std::string(what) + ": the state buffer is not device memory of device " + std::to_string(h->cfg.device);
        return D2D_ERR_INVALID;
    }
    return D2D_OK;
}

// One launch of d2d_clone_kernel over `count` copies.  The index arrays go to a per-handle device buffer with one copy on
// `stream`; an event recorded behind each kernel that reads the buffer makes the next call's stream wait before it
// overwrites the buffer, so consecutive calls on different streams never race on it.
static int launch_clone(d2d_handle *h, int mode, const int32_t *src_host, const int32_t *dst_host, int32_t count,
                        unsigned char *packed, cudaStream_t st) {
    const int nidx = (src_host ? 1 : 0) + (dst_host ? 1 : 0);
    const size_t need = (size_t)nidx * count * 4;
    if (!h->clone_ev) CUDA_TRY(h, cudaEventCreateWithFlags(&h->clone_ev, cudaEventDisableTiming));
    if (need > h->clone_idx_bytes) {
        CUDA_TRY(h, cudaEventSynchronize(h->clone_ev));          // the old buffer may still be read by an earlier kernel
        if (h->clone_idx) CUDA_TRY(h, cudaFree(h->clone_idx));
        h->clone_idx = nullptr; h->clone_idx_bytes = 0;
        CUDA_TRY(h, cudaMalloc((void **)&h->clone_idx, need));
        h->clone_idx_bytes = need;
    }
    int *idx = h->clone_idx;
    if (need) {
        h->clone_stage.resize((size_t)nidx * count);
        if (src_host) memcpy(h->clone_stage.data(), src_host, (size_t)count * 4);
        if (dst_host) memcpy(h->clone_stage.data() + (src_host ? (size_t)count : 0), dst_host, (size_t)count * 4);
        CUDA_TRY(h, cudaStreamWaitEvent(st, h->clone_ev, 0));
        CUDA_TRY(h, cudaMemcpyAsync(idx, h->clone_stage.data(), need, cudaMemcpyHostToDevice, st));
    }
    const int *src = src_host ? idx : nullptr, *dst = dst_host ? idx + (src_host ? count : 0) : nullptr;
    d2d_clone_kernel<<<count, D2D_CLONE_THREADS, 0, st>>>(h->state_tab, mode, h->arena, packed, src, dst);
    h->launches++;
    CUDA_TRY(h, cudaGetLastError());
    CUDA_TRY(h, cudaEventRecord(h->clone_ev, st));
    return D2D_OK;
}

extern "C" int d2d_clone_envs(d2d_handle *h, const int32_t *src_host, const int32_t *dst_host, int32_t count, void *stream) {
    if (!h) return D2D_ERR_INVALID;
    D2D_NO_PIPE(h);
    if (!h->world_set) { h->err = "d2d_clone_envs before d2d_set_world"; return D2D_ERR_STATE; }
    if (count < 0 || (count > 0 && (!src_host || !dst_host))) { h->err = "d2d_clone_envs: bad count or null index array"; return D2D_ERR_INVALID; }
    int rc = check_env_indices(h, "d2d_clone_envs", src_host, dst_host, count);
    if (rc != D2D_OK || count == 0) return rc;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    rc = launch_clone(h, D2D_CLONE_ARENA, src_host, dst_host, count, nullptr, (cudaStream_t)stream);
    if (rc != D2D_OK) return rc;
    h->mir_stale = true;          // the clone rewrites the device observation only
    return D2D_OK;
}

extern "C" int d2d_save_state(d2d_handle *h, const int32_t *envs_host, int32_t count, void *state_dev, void *stream) {
    if (!h) return D2D_ERR_INVALID;
    D2D_NO_PIPE(h);
    if (!h->world_set) { h->err = "d2d_save_state before d2d_set_world"; return D2D_ERR_STATE; }
    if (count < 0 || (!envs_host && count > h->B)) { h->err = "d2d_save_state: bad count"; return D2D_ERR_INVALID; }
    int rc = check_env_indices(h, "d2d_save_state", envs_host, nullptr, count);
    if (rc != D2D_OK || count == 0) return rc;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    if ((rc = check_state_ptr(h, "d2d_save_state", state_dev)) != D2D_OK) return rc;
    return launch_clone(h, D2D_CLONE_SAVE, envs_host, nullptr, count, (unsigned char *)state_dev, (cudaStream_t)stream);
}

extern "C" int d2d_load_state(d2d_handle *h, const int32_t *envs_host, int32_t count, const void *state_dev,
                              uint64_t fingerprint, void *stream) {
    if (!h) return D2D_ERR_INVALID;
    D2D_NO_PIPE(h);
    if (!h->world_set) { h->err = "d2d_load_state before d2d_set_world"; return D2D_ERR_STATE; }
    if (count < 0 || (!envs_host && count > h->B)) { h->err = "d2d_load_state: bad count"; return D2D_ERR_INVALID; }
    if (fingerprint != h->state_fingerprint) {
        h->err = "d2d_load_state: the state was saved from a handle with another layout (fingerprint mismatch)";
        return D2D_ERR_INVALID;
    }
    int rc = check_env_indices(h, "d2d_load_state", nullptr, envs_host, count);
    if (rc != D2D_OK || count == 0) return rc;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    if ((rc = check_state_ptr(h, "d2d_load_state", state_dev)) != D2D_OK) return rc;
    std::vector<int32_t> all;
    if (!envs_host) { all.resize(count); for (int32_t i = 0; i < count; i++) all[i] = i; envs_host = all.data(); }
    rc = launch_clone(h, D2D_CLONE_LOAD, nullptr, envs_host, count, (unsigned char *)state_dev, (cudaStream_t)stream);
    if (rc != D2D_OK) return rc;
    h->mir_stale = true;
    return D2D_OK;
}

// ------------------------------------------------------------------------------------------ world generation
extern "C" int d2d_set_world_sources(d2d_handle *h, const d2d_world_source *srcs, int32_t count) {
    if (!h) return D2D_ERR_INVALID;
    if (!srcs || count < 1 || count > D2D_WORLD_MAX_SOURCES) {
        h->err = "d2d_set_world_sources: " + std::to_string(count) + " sources (1.." + std::to_string(D2D_WORLD_MAX_SOURCES) +
                 ", non-null array)";
        return D2D_ERR_INVALID;
    }
    D2D_NO_PIPE(h);
    std::vector<unsigned char> tmp((size_t)count * sizeof(WgTables));
    WgTables *T = (WgTables *)tmp.data();
    for (int32_t i = 0; i < count; i++) {           // all checked before anything changes
        const d2d_world_source *src = srcs + i;
        const char *bad = wg_build_tables(T + i, src, h->cfg.targets, h->cfg.n_targets, h->cfg.map_scale, h->N,
                                          h->P.motion_rvo, h->cfg.var_cam != 0.0 ? 1 : 0);
        if (!bad && (src->map_w != h->cfg.map_w || src->map_h != h->cfg.map_h || src->drone_radius != h->cfg.drone_radius ||
                     src->agent_radius != h->cfg.agent_radius))
            bad = "map size, drone_radius or agent_radius differ from the config";
        if (bad) { h->err = "d2d_set_world_sources: source " + std::to_string(i) + ": " + bad; return D2D_ERR_INVALID; }
    }
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    if (!h->wg_fault) {
        CUDA_TRY(h, cudaHostAlloc((void **)&h->wg_fault, 2 * sizeof(unsigned long long), cudaHostAllocMapped));
        h->wg_fault[0] = 0ull; h->wg_fault[1] = 0ull;
        CUDA_TRY(h, cudaHostGetDevicePointer((void **)&h->wg_fault_dev, (void *)h->wg_fault, 0));
    }
    if (!h->wg_claim) {
        CUDA_TRY(h, cudaMalloc((void **)&h->wg_claim, sizeof(unsigned int)));
        CUDA_TRY(h, cudaMemset(h->wg_claim, 0, sizeof(unsigned int)));
    }
    if (count > h->wg_cap) {                        // grows only: a captured graph keeps a valid table address until then
        CUDA_TRY(h, cudaDeviceSynchronize());        // no generation kernel may still read the old table
        WgTables *t = nullptr;
        if (cudaMalloc((void **)&t, (size_t)count * sizeof(WgTables)) != cudaSuccess) {
            cudaGetLastError();
            h->err = "d2d_set_world_sources: cudaMalloc failed"; return D2D_ERR_NOMEM;
        }
        if (h->wg_tab) cudaFree(h->wg_tab);
        h->wg_tab = t; h->wg_cap = count;
    } else {
        CUDA_TRY(h, cudaDeviceSynchronize());        // no generation kernel (nor one behind a queue step) may still read it
    }
    CUDA_TRY(h, cudaMemcpy(h->wg_tab, T, (size_t)count * sizeof(WgTables), cudaMemcpyHostToDevice));
    h->wg_count = count;
    return D2D_OK;
}

extern "C" int d2d_set_world_source(d2d_handle *h, const d2d_world_source *src) { return d2d_set_world_sources(h, src, 1); }

// A world the generation kernels gave up on: reported (and cleared, with the claim in stream order) by the next
// d2d_generate_worlds / d2d_read_episode_log.
static bool take_wg_fault(d2d_handle *h, const char *what, cudaStream_t st) {
    const unsigned long long fault = h->wg_fault ? h->wg_fault[0] : 0ull;
    if (!fault) return false;
    const unsigned long long env = h->wg_fault[1];
    h->wg_fault[0] = 0ull; h->wg_fault[1] = 0ull;
    cudaMemsetAsync(h->wg_claim, 0, sizeof(unsigned int), st);
    h->err = std::string(what) + ": the world of seed " + std::to_string((unsigned)(fault & 0xffffffffull)) + " from source " +
             std::to_string((unsigned)((fault >> 32) & 0x7fffffffull)) + " (env " + std::to_string(env) +
             ") could not be built: more than " + std::to_string(D2D_WORLD_MAX_REJECTS) +
             " rejected draws in a row; that env's world is undefined";
    return true;
}

// Seeds (source 0, [0, 2^32)) or world keys whose source is in the table; false (error set) on the first bad one.
static bool check_world_keys(d2d_handle *h, const char *what, const int64_t *keys, int64_t count, bool seeds_only) {
    for (int64_t i = 0; i < count; i++) {
        const long long k = (long long)keys[i];
        if (seeds_only && (k < 0 || k > 0xffffffffll)) {
            h->err = std::string(what) + ": seed " + std::to_string(k) + " outside [0, 2**32)";
            return false;
        }
        if (k < 0 || (k >> 32) >= h->wg_count) {
            h->err = std::string(what) + ": key " + std::to_string(k) + (k < 0 ? " is negative" : ": source " +
                     std::to_string(k >> 32) + " outside the table of " + std::to_string(h->wg_count) + " world sources");
            return false;
        }
    }
    return true;
}

static int generate_worlds(d2d_handle *h, const int32_t *envs_host, const int64_t *keys_host, int32_t count, int32_t flags,
                           void *stream, bool seeds_only);

extern "C" int d2d_generate_worlds(d2d_handle *h, const int32_t *envs_host, const int64_t *seeds_host, int32_t count,
                                   int32_t flags, void *stream) {
    return generate_worlds(h, envs_host, seeds_host, count, flags, stream, true);
}

extern "C" int d2d_generate_worlds_keyed(d2d_handle *h, const int32_t *envs_host, const int64_t *keys_host, int32_t count,
                                         int32_t flags, void *stream) {
    return generate_worlds(h, envs_host, keys_host, count, flags, stream, false);
}

// seeds_only: d2d_generate_worlds (every key a seed of source 0, checked as such)
static int generate_worlds(d2d_handle *h, const int32_t *envs_host, const int64_t *keys_host, int32_t count, int32_t flags,
                           void *stream, bool seeds_only) {
    if (!h) return D2D_ERR_INVALID;
    D2D_NO_PIPE(h);
    if (!h->wg_tab) { h->err = "d2d_generate_worlds before d2d_set_world_sources"; return D2D_ERR_STATE; }
    if (take_wg_fault(h, "d2d_generate_worlds", (cudaStream_t)stream)) return D2D_ERR_STATE;
    if (flags != D2D_WORLD_EAGER && flags != D2D_WORLD_LAZY) {
        h->err = "d2d_generate_worlds: flags must be D2D_WORLD_EAGER or D2D_WORLD_LAZY"; return D2D_ERR_INVALID;
    }
    if (count < 0 || (count > 0 && (!envs_host || !keys_host))) { h->err = "d2d_generate_worlds: bad count or null array"; return D2D_ERR_INVALID; }
    int rc = check_env_indices(h, "d2d_generate_worlds", nullptr, envs_host, count);
    if (rc != D2D_OK) return rc;
    if (!check_world_keys(h, "d2d_generate_worlds", keys_host, count, seeds_only)) return D2D_ERR_INVALID;
    if (count == 0) return D2D_OK;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    const bool eager = flags == D2D_WORLD_EAGER;
    // envs, keys (8-byte aligned) and (eager) the reset mask in one staged copy; the event keeps the next call from
    // overwriting the device buffer while a kernel still reads it (as launch_clone does)
    const size_t ko = (size_t)count + (count & 1), mo = ko + 2 * (size_t)count;
    const size_t words = mo + (eager ? ((size_t)h->B + 3) / 4 : 0);
    if (!h->wg_ev) CUDA_TRY(h, cudaEventCreateWithFlags(&h->wg_ev, cudaEventDisableTiming));
    if (words * 4 > h->wg_idx_bytes) {
        CUDA_TRY(h, cudaEventSynchronize(h->wg_ev));
        if (h->wg_idx) CUDA_TRY(h, cudaFree(h->wg_idx));
        h->wg_idx = nullptr; h->wg_idx_bytes = 0;
        CUDA_TRY(h, cudaMalloc((void **)&h->wg_idx, words * 4));
        h->wg_idx_bytes = words * 4;
    }
    h->wg_stage.assign(words, 0);
    memcpy(h->wg_stage.data(), envs_host, (size_t)count * 4);
    memcpy(h->wg_stage.data() + ko, keys_host, (size_t)count * 8);
    uint8_t *mask = (uint8_t *)(h->wg_stage.data() + mo);
    if (eager) for (int32_t i = 0; i < count; i++) mask[envs_host[i]] = 1;
    CUDA_TRY(h, cudaStreamWaitEvent(st, h->wg_ev, 0));
    CUDA_TRY(h, cudaMemcpyAsync(h->wg_idx, h->wg_stage.data(), words * 4, cudaMemcpyHostToDevice, st));
    d2d_worldgen_kernel<<<(count + D2D_WG_WARPS - 1) / D2D_WG_WARPS, D2D_WG_WARPS * 32, 0, st>>>(
        h->P, h->wg_tab, h->wg_idx, (const long long *)(h->wg_idx + ko), count, eager ? 0 : 1, h->wg_fault_dev,
        h->wg_claim);
    h->launches++;
    CUDA_TRY(h, cudaGetLastError());
    if (eager) {
        d2d_reset_kernel<<<h->B, 128, 0, st>>>(h->P, (const uint8_t *)(h->wg_idx + mo));
        h->launches++;
        CUDA_TRY(h, cudaGetLastError());
        h->mir_stale = true;      // the eager reset rewrites the device observation only
    }
    CUDA_TRY(h, cudaEventRecord(h->wg_ev, st));
    h->world_set = true;
    if (h->cfg.var_cam != 0.0) h->rng_set = true;
    if (h->P.motion_rvo) h->rvo_set = true;
    return D2D_OK;
}

// ------------------------------------------------------------------------------------------ episode log + seed queue
extern "C" int d2d_enable_episode_log(d2d_handle *h, int64_t capacity) {
    if (!h) return D2D_ERR_INVALID;
    if (capacity < 0 || capacity > ((int64_t)1 << 40) / (int64_t)sizeof(d2d_episode_record)) {
        h->err = "d2d_enable_episode_log: capacity out of range"; return D2D_ERR_INVALID;
    }
    D2D_NO_PIPE(h);
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    CUDA_TRY(h, cudaDeviceSynchronize());            // no kernel may still use the old buffers
    if (h->ep_mem) CUDA_TRY(h, cudaFree(h->ep_mem));
    h->ep_mem = nullptr; h->ep = EpLog{}; h->ep_qlen = 0;
    if (capacity == 0) return D2D_OK;
    const size_t B = (size_t)h->B;
    const size_t o_head = (size_t)capacity * sizeof(d2d_episode_record);
    const size_t o_seed = o_head + 64, o_list = o_seed + (B * 8 + 15) / 16 * 16, o_genv = o_list + (B * 4 + 15) / 16 * 16;
    const size_t o_gkey = o_genv + (B * 4 + 15) / 16 * 16, bytes = o_gkey + (B * 8 + 15) / 16 * 16;
    unsigned char *m = nullptr;
    if (cudaMalloc((void **)&m, bytes) != cudaSuccess) {
        cudaGetLastError();
        h->err = "d2d_enable_episode_log: cudaMalloc of " + std::to_string(bytes) + " B failed"; return D2D_ERR_NOMEM;
    }
    if (cudaMemset(m, 0, bytes) != cudaSuccess) { cudaFree(m); h->err = "d2d_enable_episode_log: cudaMemset failed"; return D2D_ERR_CUDA; }
    h->ep_mem = m;
    h->ep.rec = (d2d_episode_record *)m; h->ep.capacity = capacity;
    h->ep.head = (long long *)(m + o_head); h->ep.gen_count = (int *)(m + o_head + 32);
    h->ep.ticket = (unsigned int *)(m + o_head + 36);
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->cfg.device) != cudaSuccess || sms <= 0) sms = 148;
    h->ep_blocks = (h->B + 31) / 32 < sms ? (h->B + 31) / 32 : sms;
    h->ep.world_seed = (long long *)(m + o_seed); h->ep.list = (int *)(m + o_list);
    h->ep.gen_env = (int *)(m + o_genv); h->ep.gen_key = (long long *)(m + o_gkey);
    h->ep.queue = h->ep_queue;
    return D2D_OK;
}

extern "C" int d2d_read_episode_log(d2d_handle *h, d2d_episode_record *out_host, int64_t *count, int64_t *dropped, void *stream) {
    if (!h) return D2D_ERR_INVALID;
    if (!count || !dropped || !out_host) { h->err = "d2d_read_episode_log: null argument"; return D2D_ERR_INVALID; }
    D2D_NO_PIPE(h);
    if (!h->ep_mem) { h->err = "d2d_read_episode_log: the episode log is not enabled"; return D2D_ERR_STATE; }
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(h, cudaStreamSynchronize(st));
    if (take_wg_fault(h, "d2d_read_episode_log", st)) return D2D_ERR_STATE;
    long long written = 0;
    CUDA_TRY(h, cudaMemcpyAsync(&written, h->ep.head, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(h, cudaStreamSynchronize(st));
    const long long n = written < h->ep.capacity ? written : h->ep.capacity;
    if (n > 0)
        CUDA_TRY(h, cudaMemcpyAsync(out_host, h->ep.rec, (size_t)n * sizeof(d2d_episode_record), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(h, cudaMemsetAsync(h->ep.head, 0, 8, st));
    CUDA_TRY(h, cudaStreamSynchronize(st));
    *count = n;
    *dropped = written - n;
    return D2D_OK;
}

static int set_world_queue(d2d_handle *h, const char *what, const int64_t *keys_host, int64_t count, void *stream,
                           bool seeds_only);

extern "C" int d2d_set_seed_queue(d2d_handle *h, const int64_t *seeds_host, int64_t count, void *stream) {
    return set_world_queue(h, "d2d_set_seed_queue", seeds_host, count, stream, true);
}

extern "C" int d2d_set_world_queue(d2d_handle *h, const int64_t *keys_host, int64_t count, void *stream) {
    return set_world_queue(h, "d2d_set_world_queue", keys_host, count, stream, false);
}

// seeds_only: d2d_set_seed_queue (every key a seed of source 0, checked as such)
static int set_world_queue(d2d_handle *h, const char *what, const int64_t *keys_host, int64_t count, void *stream,
                           bool seeds_only) {
    if (!h) return D2D_ERR_INVALID;
    D2D_NO_PIPE(h);
    if (!h->wg_tab) { h->err = std::string(what) + " before d2d_set_world_sources"; return D2D_ERR_STATE; }
    if (!h->cfg.auto_reset) { h->err = std::string(what) + ": the handle was created with auto_reset = 0"; return D2D_ERR_STATE; }
    if (!h->ep_mem) { h->err = std::string(what) + ": the episode log is not enabled"; return D2D_ERR_STATE; }
    if (count < 0 || (count > 0 && !keys_host)) { h->err = std::string(what) + ": bad count or null array"; return D2D_ERR_INVALID; }
    if (!check_world_keys(h, what, keys_host, count, seeds_only)) return D2D_ERR_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    if (count > h->ep_queue_cap) {                   // grows only: a captured graph keeps a valid queue address
        CUDA_TRY(h, cudaDeviceSynchronize());        // no log kernel may still read the old queue
        long long *q = nullptr;
        if (cudaMalloc((void **)&q, (size_t)count * 8) != cudaSuccess) {
            cudaGetLastError();
            h->err = std::string(what) + ": cudaMalloc failed"; return D2D_ERR_NOMEM;
        }
        if (h->ep_queue) cudaFree(h->ep_queue);
        h->ep_queue = q; h->ep_queue_cap = count; h->ep.queue = q;
    } else {
        CUDA_TRY(h, cudaStreamSynchronize(st));      // the last log kernel on this stream has read the old keys
    }
    if (count > 0) CUDA_TRY(h, cudaMemcpyAsync(h->ep_queue, keys_host, (size_t)count * 8, cudaMemcpyHostToDevice, st));
    h->ep_qhead[0] = 0; h->ep_qhead[1] = count;
    CUDA_TRY(h, cudaMemcpyAsync(h->ep.head + 2, h->ep_qhead, 16, cudaMemcpyHostToDevice, st));
    CUDA_TRY(h, cudaStreamSynchronize(st));
    h->ep_qlen = count;
    return D2D_OK;
}

// ------------------------------------------------------------------------------------------ rendering
extern "C" int d2d_render(d2d_handle *h, const int32_t *envs_host, int32_t first_env, int32_t count, int32_t pixels_per_cell,
                          int32_t layers, uint8_t *frames_dev, void *stream) {
    if (!h) return D2D_ERR_INVALID;
    D2D_NO_PIPE(h);
    if (!h->world_set) { h->err = "d2d_render before d2d_set_world"; return D2D_ERR_STATE; }
    if (count < 0) { h->err = "d2d_render: negative count"; return D2D_ERR_INVALID; }
    if (pixels_per_cell < 1 || pixels_per_cell > D2D_RENDER_MAX_PPC) {
        h->err = "d2d_render: pixels_per_cell " + std::to_string(pixels_per_cell) + " outside 1.." + std::to_string(D2D_RENDER_MAX_PPC);
        return D2D_ERR_INVALID;
    }
    if (layers & ~D2D_RENDER_ALL) { h->err = "d2d_render: unknown layer bits " + std::to_string(layers & ~D2D_RENDER_ALL); return D2D_ERR_INVALID; }
    RenderList list;
    if (envs_host) {
        if (count > D2D_RENDER_MAX_LIST) {
            h->err = "d2d_render: a list of " + std::to_string(count) + " envs (at most " + std::to_string(D2D_RENDER_MAX_LIST) +
                     "; render a larger selection as a contiguous range)";
            return D2D_ERR_INVALID;
        }
        int rc = check_env_indices(h, "d2d_render", envs_host, nullptr, count);
        if (rc != D2D_OK) return rc;
        memcpy(list.e, envs_host, (size_t)count * 4);
    } else if (first_env < 0 || first_env > h->B || count > h->B - first_env) {
        h->err = "d2d_render: envs [" + std::to_string(first_env) + ", " + std::to_string((long long)first_env + count) +
                 ") outside [0, " + std::to_string(h->B) + ")";
        return D2D_ERR_INVALID;
    }
    if (count == 0) return D2D_OK;
    if (!frames_dev) { h->err = "d2d_render: null frame buffer"; return D2D_ERR_INVALID; }
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, frames_dev) != cudaSuccess || at.type != cudaMemoryTypeDevice || at.device != h->cfg.device) {
        cudaGetLastError();
        h->err = "d2d_render: the frame buffer is not device memory of device " + std::to_string(h->cfg.device);
        return D2D_ERR_INVALID;
    }
    RenderArgs a;
    a.frames = frames_dev; a.first_env = first_env; a.count = count; a.use_list = envs_host ? 1 : 0;
    a.ppc = pixels_per_cell; a.layers = layers; a.W = D2D_GRID * pixels_per_cell;
    a.band_rows = D2D_RENDER_BAND_PIX / a.W < D2D_GRID * pixels_per_cell ? D2D_RENDER_BAND_PIX / a.W : D2D_GRID * pixels_per_cell;
    a.nbands = (D2D_GRID * pixels_per_cell + a.band_rows - 1) / a.band_rows;
    a.s = h->cfg.map_scale / (double)pixels_per_cell;
    a.span = h->P.ray_da * (double)(h->cfg.n_rays - 1);
    const long long blocks = (long long)count * a.nbands;
    d2d_render_kernel<<<(unsigned)blocks, D2D_RENDER_THREADS, 0, (cudaStream_t)stream>>>(h->P, a, list);
    h->launches++;
    CUDA_TRY(h, cudaGetLastError());
    return D2D_OK;
}

// ------------------------------------------------------------------------------------------ difficulty metrics
static int check_dev_out(d2d_handle *h, const char *what, const void *p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess || at.type != cudaMemoryTypeDevice || at.device != h->cfg.device) {
        cudaGetLastError();
        h->err = std::string("d2d_difficulty: ") + what + " is not device memory of device " + std::to_string(h->cfg.device);
        return D2D_ERR_INVALID;
    }
    return D2D_OK;
}

extern "C" int d2d_difficulty(d2d_handle *h, const d2d_difficulty_spec *spec, int32_t first_env, int32_t count,
                              int16_t *first_hit, uint8_t *static_hit, uint8_t *collision_state, void *stream) {
    if (!h) return D2D_ERR_INVALID;
    D2D_NO_PIPE(h);
    if (!h->world_set) { h->err = "d2d_difficulty before d2d_set_world"; return D2D_ERR_STATE; }
    if (h->P.motion_rvo) {
        h->err = "d2d_difficulty: motion_profile = RVO: the agents' motion needs d2d_rvo_kernel, so the metrics must step the "
                 "envs (metrics.global_survivability / metrics.survivability)";
        return D2D_ERR_STATE;
    }
    if (!spec) { h->err = "d2d_difficulty: null spec"; return D2D_ERR_INVALID; }
    const d2d_difficulty_spec &S = *spec;
    if (S.struct_size != (int32_t)sizeof(d2d_difficulty_spec)) { h->err = "d2d_difficulty: d2d_difficulty_spec size mismatch (ABI)"; return D2D_ERR_INVALID; }
    if (S.nx < 1 || S.ny < 1 || (int64_t)S.nx * S.ny > D2D_DIFF_MAX_POS) {
        h->err = "d2d_difficulty: a " + std::to_string(S.nx) + " x " + std::to_string(S.ny) + " grid (1 to " +
                 std::to_string(D2D_DIFF_MAX_POS) + " positions)";
        return D2D_ERR_INVALID;
    }
    if (!std::isfinite(S.x0) || !std::isfinite(S.y0) || !std::isfinite(S.step) || !(S.step > 0.0)) {
        h->err = "d2d_difficulty: x0, y0 and step must be finite and step > 0"; return D2D_ERR_INVALID;
    }
    if (S.steps < 1 || S.steps > D2D_DIFF_MAX_STEPS) {
        h->err = "d2d_difficulty: steps " + std::to_string(S.steps) + " outside 1.." + std::to_string(D2D_DIFF_MAX_STEPS);
        return D2D_ERR_INVALID;
    }
    if (S.n_slots < 0 || S.n_slots > D2D_DIFF_MAX_STEPS) {
        h->err = "d2d_difficulty: n_slots " + std::to_string(S.n_slots) + " outside 0.." + std::to_string(D2D_DIFF_MAX_STEPS);
        return D2D_ERR_INVALID;
    }
    if ((collision_state == nullptr) != (S.n_slots == 0)) {
        h->err = "d2d_difficulty: collision_state must be given exactly when n_slots > 0"; return D2D_ERR_INVALID;
    }
    if (S.n_slots > 0)
        for (int k = 0; k < S.steps; k++) {
            const int s = S.slot[k];
            if ((s >= S.n_slots && s != D2D_DIFF_NO_SLOT) || (k > 0 && s < S.slot[k - 1])) {
                h->err = "d2d_difficulty: slot[" + std::to_string(k) + "] = " + std::to_string(s) +
                         ": the slot table must be non-decreasing with entries < n_slots or D2D_DIFF_NO_SLOT";
                return D2D_ERR_INVALID;
            }
        }
    if (count < 0 || first_env < 0 || first_env > h->B || count > h->B - first_env) {
        h->err = "d2d_difficulty: envs [" + std::to_string(first_env) + ", " + std::to_string((long long)first_env + count) +
                 ") outside [0, " + std::to_string(h->B) + ")";
        return D2D_ERR_INVALID;
    }
    if (count == 0) return D2D_OK;
    if (!first_hit || !static_hit) { h->err = "d2d_difficulty: null output"; return D2D_ERR_INVALID; }
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    int rc;
    if ((rc = check_dev_out(h, "first_hit", first_hit)) != D2D_OK) return rc;
    if ((rc = check_dev_out(h, "static_hit", static_hit)) != D2D_OK) return rc;
    if (collision_state && (rc = check_dev_out(h, "collision_state", collision_state)) != D2D_OK) return rc;
    DiffOut o;
    o.first_hit = first_hit; o.static_hit = static_hit; o.cs = collision_state;
    o.first_env = first_env; o.count = count;
    o.nchunks = (S.nx * S.ny + 63) / 64;
    o.nwords = (S.n_slots + 31) / 32;
    const long long tasks = (long long)count * o.nchunks;
    const size_t smem = (size_t)D2D_DIFF_WARPS * 64 * o.nwords * 4;
    d2d_difficulty_kernel<<<(unsigned)((tasks + D2D_DIFF_WARPS - 1) / D2D_DIFF_WARPS), D2D_DIFF_WARPS * 32, smem,
                            (cudaStream_t)stream>>>(h->P, o, S);
    h->launches++;
    CUDA_TRY(h, cudaGetLastError());
    return D2D_OK;
}

// ------------------------------------------------------------------------------------------ Primitive planner path + Oxford
#include "d2d_plan_host.inl"
