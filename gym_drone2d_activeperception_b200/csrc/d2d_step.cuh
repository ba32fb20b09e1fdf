// d2d_step.cuh -- the per-step kernels (sm_100a).
//
// Work decomposition.  One thread block owns E consecutive environments and walks them through the phases of
// Drone2DEnv2.step (envs/drone_v2.py:152-257) in the reference's order, separated by __syncthreads():
//
//   P0  env leaders load the drone/bookkeeping scalars (lazy auto-reset from the snapshot if the env was done);
//       one thread issues TMA bulk copies (cp.async.bulk -> UBLKCP) of each env's belief grid (2560 B) and
//       ground-truth row bitmap (400 B) from HBM into shared memory, completion on an mbarrier.
//   P1  one work item per (env, agent): Agent.step (utils.py:472-493), write back, keep (x, y, r^2) in shared
//       memory, broad-phase cull against the drone's view reach, drone-vs-agent collision test.
//   P2  one work item per (env, ray): Raycast.castRay (utils.py:620-713) with the reference's exact stepping
//       arithmetic against the shared-memory bitmap and the culled discs; newly seen belief cells are written
//       to shared memory AND to HBM (only cells whose value changes: ~3 byte stores per env-step).
//   P3  one work item per (env, agent): hit mask out, Kalman tracker update (utils.py:242-275).
//   P4  env leaders: planner bookkeeping, step_pos / step_yaw, static collision probes, flags, done, statistics.
//   P5  the block writes its E*1089-byte slice of the local-map observation with coalesced 32-bit stores,
//       gathering from the shared-memory belief grids (Drone2D.get_local_map, utils.py:780-784).
//
// Work items are packed across environment boundaries (item -> (env, k) by division), so lanes stay busy for any
// ray / agent count; everything an environment shares between its threads lives in shared memory.
#pragma once
#include "d2d_state.cuh"
#include "d2d_math.cuh"
#include "d2d_agent_math.cuh"

// big, once-per-env-step helpers: inlined by default; -DD2D_COLD_NOINLINE=1 keeps one shared copy of each
#if defined(D2D_COLD_NOINLINE) && D2D_COLD_NOINLINE
#define D2D_COLD __noinline__
#else
#define D2D_COLD __forceinline__
#endif

// ------------------------------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t d2d_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void d2d_mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(d2d_smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void d2d_mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(d2d_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void d2d_bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     d2d_smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(d2d_smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void d2d_mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    const uint32_t addr = d2d_smem_u32(bar);
    do {
        asm volatile(
            "{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
            : "=r"(ok)
            : "r"(addr), "r"(parity)
            : "memory");
    } while (!ok);
}

// ------------------------------------------------------------------------------------------ shared-memory context
// per-env working set in shared memory: the env's persistent record (copied verbatim from / to HBM) + this step's scratch
struct EnvS : EnvRec {
    int valid, reset, ncull, coll_agent;
    int arch_cnt, arch_ts, act_cnt, act_ts, newly;
    int done_now, ix, iy, ox_was_fresh, owl_was_fresh;
    // Jerk_Primitive: the single waypoint plan() appended this step (traj_planner.py:496-499), consumed by step_pos
    int jerk_has;
    double jerk_px, jerk_py, jerk_vx, jerk_vy, jerk_ax, jerk_ay;
};

struct BlockCtx {
    uint8_t *belief;     // [E][D2D_BELIEF_STRIDE]
    uint64_t *gt;        // [E][50]
    double *sx, *sy, *sr2;  // [E][NP]
    double *mx, *my;        // [E][NP] measurements handed to the trackers (== sx, sy when var_cam == 0)
    uint16_t *cull;      // [E][NP]
    uint32_t *hitw;      // [E][HW]
    EnvS *S;             // [E]
    uint64_t *mbar;
    int *misc;           // [4] block-level scratch
};

__host__ __device__ inline size_t d2d_step_smem_bytes(int E, int NP, int HW) {
    size_t b = (size_t)E * D2D_BELIEF_STRIDE + (size_t)E * D2D_GT_ROW_BYTES;
    b += (size_t)E * NP * 8 * 5;
    b += ((size_t)E * NP * 2 + 15) / 16 * 16;
    b += ((size_t)E * HW * 4 + 15) / 16 * 16;
    b = (b + 15) / 16 * 16;              // EnvS is copied with 16-byte accesses
    b += (size_t)E * sizeof(EnvS);
    b += 16 + 16;
    return b;
}

__device__ __forceinline__ BlockCtx d2d_carve(unsigned char *base, int E, int NP, int HW) {
    BlockCtx c;
    size_t o = 0;
    c.belief = base; o += (size_t)E * D2D_BELIEF_STRIDE;
    c.gt = (uint64_t *)(base + o); o += (size_t)E * D2D_GT_ROW_BYTES;
    c.sx = (double *)(base + o); o += (size_t)E * NP * 8;
    c.sy = (double *)(base + o); o += (size_t)E * NP * 8;
    c.sr2 = (double *)(base + o); o += (size_t)E * NP * 8;
    c.mx = (double *)(base + o); o += (size_t)E * NP * 8;
    c.my = (double *)(base + o); o += (size_t)E * NP * 8;
    c.cull = (uint16_t *)(base + o); o += ((size_t)E * NP * 2 + 15) / 16 * 16;
    c.hitw = (uint32_t *)(base + o); o += ((size_t)E * HW * 4 + 15) / 16 * 16;
    o = (o + 15) / 16 * 16;
    c.S = (EnvS *)(base + o); o += (size_t)E * sizeof(EnvS);
    c.mbar = (uint64_t *)(base + o); o += 16;
    c.misc = (int *)(base + o);
    return c;
}

// ------------------------------------------------------------------------------------------ P0: scalars + bulk loads
// After the record has been copied into the head of `s`: lazy reset (Drone2DEnv2.__init__, drone_v2.py:88-117: drone at the
// init pose, zero velocity, WAIT_FOR_GOAL; Planner.__init__ traj_planner.py:22) and this step's scratch.  One thread.
// CELL = false: ix / iy are left to the caller (the small-crowd rollout keeps them for as long as the pose is unchanged).
template <bool CELL = true>
__device__ __forceinline__ void d2d_env_begin(const DevP &P, EnvS &s, bool was_done) {
    const bool rs = s.pending_reset != 0 || (P.auto_reset && was_done);
    s.ox_was_fresh = s.ox_fresh; s.owl_was_fresh = s.owl_fresh;
    s.pending_reset = 0; s.ox_fresh = 0; s.owl_fresh = 0;   // consumed; written back with the record at the end of the step
    if (rs) {
        s.px = s.p0x; s.py = s.p0y; s.yaw = s.p0yaw; s.vx = 0; s.vy = 0; s.tgx = s.p0x; s.tgy = s.p0y;
        s.steps = 0; s.sm = SM_WAIT_FOR_GOAL; s.fail = 0; s.tcur = 0; s.bufc = 0; s.bufts = 0; s.tracked = 0;
        s.nseg = 0; s.cursor = 0;
        if (P.planner == D2D_PLANNER_JERK) { s.tgx = 0.0; s.tgy = 0.0; }   // Jerk_Primitive.__init__: target = np.zeros(4) (:406)
    }
    if (CELL) { s.ix = d2d_cell(s.px, P.scale, P.inv_scale); s.iy = d2d_cell(s.py, P.scale, P.inv_scale); }
    s.valid = 1; s.reset = rs; s.jerk_has = 0;
    s.ncull = 0; s.coll_agent = 0; s.arch_cnt = 0; s.arch_ts = 0; s.act_cnt = 0; s.act_ts = 0; s.newly = 0; s.done_now = 0;
}

// single-thread load / store of an env's record (block kernels, list kernels): eight 16-byte accesses of one 128-byte line
__device__ D2D_COLD void d2d_load_env_scalars(const DevP &P, EnvS &s, int e) {
    if (e >= P.B) {
        s.valid = 0; s.reset = 0; s.done_now = 0; s.ncull = 0; s.coll_agent = 0;
        return;
    }
    const bool was_done = P.done[e] != 0;
    const uint4 *src = (const uint4 *)(P.rec + e);
    uint4 r[8];
#pragma unroll
    for (int i = 0; i < 8; i++) r[i] = src[i];
#pragma unroll
    for (int i = 0; i < 8; i++) ((uint4 *)&s)[i] = r[i];
    d2d_env_begin(P, s, was_done);
}

__device__ D2D_COLD void d2d_store_env_scalars(const DevP &P, const EnvS &s, int e) {
    uint4 *dst = (uint4 *)(P.rec + e);
#pragma unroll
    for (int i = 0; i < 8; i++) dst[i] = ((const uint4 *)&s)[i];
}

// warp-cooperative variants (one env per warp): a single coalesced 128-byte request each way
__device__ __forceinline__ void d2d_load_env_warp(const DevP &P, EnvS &s, int e, int lane) {
    unsigned long long w = 0ull;
    uint8_t was_done = 0;
    if (lane < 16) w = ((const unsigned long long *)(P.rec + e))[lane];
    if (lane == 0) was_done = P.done[e];
    if (lane < 16) ((unsigned long long *)&s)[lane] = w;
    __syncwarp();
    if (lane == 0) d2d_env_begin(P, s, was_done != 0);
}
__device__ __forceinline__ void d2d_store_env_warp(const DevP &P, const EnvS &s, int e, int lane) {
    if (lane < 16) ((unsigned long long *)(P.rec + e))[lane] = ((const unsigned long long *)&s)[lane];
}

// issue the bulk copies for the block (thread 0) -- belief only for envs that are not being reset
__device__ __forceinline__ void d2d_issue_bulk(const DevP &P, const BlockCtx &c, int env0, int E, bool want_belief) {
    uint32_t bytes = 0;
    for (int i = 0; i < E; i++) {
        if (!c.S[i].valid) continue;
        bytes += D2D_GT_ROW_BYTES;
        if (want_belief && !c.S[i].reset) bytes += D2D_BELIEF_STRIDE;
    }
    d2d_mbar_expect_tx(c.mbar, bytes);
    for (int i = 0; i < E; i++) {
        if (!c.S[i].valid) continue;
        const size_t e = (size_t)(env0 + i);
        d2d_bulk_g2s(c.gt + (size_t)i * D2D_GRID, P.gt_rows + e * D2D_GRID, D2D_GT_ROW_BYTES, c.mbar);
        if (want_belief && !c.S[i].reset)
            d2d_bulk_g2s(c.belief + (size_t)i * D2D_BELIEF_STRIDE, P.belief + e * D2D_BELIEF_STRIDE, D2D_BELIEF_STRIDE, c.mbar);
    }
}

// envs being reset: zero belief in shared memory and HBM; restore the Oxford policy state
__device__ D2D_COLD void d2d_reset_arrays(const DevP &P, const BlockCtx &c, int env0, int E, int tid, int T,
                                          uint64_t *early_bulk = nullptr) {
    if (!c.misc[1]) return;   // block-uniform: no env of this block is being reset (the common case)
    // warp kernels start the bulk copy of the belief grid before they know whether the env is being reset: it must have
    // landed before the shared copy is zeroed
    if (early_bulk) d2d_mbar_wait(early_bulk, 0);
    const int W = D2D_BELIEF_STRIDE / 16;              // 16-byte stores: the grids are 128-byte aligned rows of 2560 bytes
#pragma unroll 1
    for (int w = tid; w < E * W; w += T) {
        const int i = w / W, o = w - i * W;
        if (!c.S[i].valid || !c.S[i].reset) continue;
        ((uint4 *)(c.belief + (size_t)i * D2D_BELIEF_STRIDE))[o] = uint4{0u, 0u, 0u, 0u};
        ((uint4 *)(P.belief + (size_t)(env0 + i) * D2D_BELIEF_STRIDE))[o] = uint4{0u, 0u, 0u, 0u};
    }
    if (P.rng_key) {   // reset() re-seeds np.random with map_id (drone_v2.py:80): restore the post-init stream state
#pragma unroll 1
        for (int w = tid; w < E * 624; w += T) {
            const int i = w / 624, o = w - i * 624;
            if (!c.S[i].valid || !c.S[i].reset) continue;
            const size_t g = (size_t)(env0 + i) * 624 + o;
            P.rng_key[g] = P.rng_key0[g];
            if (o == 0) { const int e2 = env0 + i; P.rng_pos[e2] = P.rng_pos0[e2]; P.rng_has[e2] = P.rng_has0[e2]; P.rng_gauss[e2] = P.rng_gauss0[e2]; }
        }
    }
    if (P.ox_seen) {   // Oxford.__init__ (yaw_planner.py:49): every cell "last observed 5.0 s ago" == never seen, 0 calls
        const int W = D2D_OX_SEEN_STRIDE / 2;
#pragma unroll 1
        for (int w = tid; w < E * W; w += T) {
            const int i = w / W, o = w - i * W;
            if (!c.S[i].valid || !c.S[i].reset || c.S[i].ox_was_fresh) continue;
            ((uint32_t *)(P.ox_seen + (size_t)(env0 + i) * D2D_OX_SEEN_STRIDE))[o] = 0u;
            if (o == 0) P.ox_calls[env0 + i] = 0;
        }
    }
    if (P.owl_U) {    // Owl.__init__ (yaw_planner.py:160-171): U_list zeros, empty queue
#pragma unroll 1
        for (int w = tid; w < E * D2D_OWL_BINS; w += T) {
            const int i = w / D2D_OWL_BINS, o = w - i * D2D_OWL_BINS;
            if (!c.S[i].valid || !c.S[i].reset || c.S[i].owl_was_fresh) continue;
            P.owl_U[(size_t)(env0 + i) * D2D_OWL_BINS + o] = 0.0;
            if (o == 0) P.owl_q[env0 + i] = 0;
        }
    }
}

// an env that is being reset restarts from its snapshot: request it (and the tracker radii the tracker phase will need)
// before the zeroing pass of d2d_reset_arrays so that the DRAM round trip overlaps it (one warp per env)
__device__ __forceinline__ void d2d_reset_prefetch(const DevP &P, const EnvS &s, int e, int lane, double2 &pf_pos,
                                                   double2 &pf_pref) {
    if (s.reset && lane < P.N) {
        const size_t g = (size_t)e * P.NP + lane;
        pf_pos = P.apos0[g]; pf_pref = P.apref0[g];
        asm volatile("prefetch.global.L2 [%0];" ::"l"(P.trk_radius0 + g));
    }
}

// ------------------------------------------------------------------------------------------ P1: Agent.step
// PF: the caller (one warp, E == 1) already holds agent `tid` of the live arrays in registers (pf_*), loaded before the env
// scalars were known so that the two DRAM round trips overlap; an env being reset re-reads its snapshot instead.
template <bool COLLIDE_HERE, bool PF = false>
__device__ __forceinline__ void d2d_phase_agents(const DevP &P, const BlockCtx &c, int env0, int E, int tid, int T,
                                                 double2 pf_pos = double2{0.0, 0.0}, double2 pf_pref = double2{0.0, 0.0},
                                                 double pf_r = 0.0, double2 *keep_pos = nullptr, double2 *keep_pref = nullptr) {
    const double C6 = 0.8660254037844387, S6 = 0.49999999999999994;   // math.cos(pi/6), math.sin(pi/6) (glibc)
    const int N = P.N, NP = P.NP;
#pragma unroll 1
    for (int w = tid; w < E * N; w += T) {
        const int i = w / N, k = w - i * N;
        EnvS &s = c.S[i];
        if (!s.valid) continue;
        const size_t g = (size_t)(env0 + i) * NP + k;
        double2 pos, pref;
        double r;
        if (PF && w == tid) { pos = pf_pos; pref = pf_pref; r = pf_r; }   // live state, or the snapshot if the env is being reset
        else {
            if (s.reset) { pos = P.apos0[g]; pref = P.apref0[g]; }
            else { pos = P.apos[g]; pref = P.apref[g]; }
            r = P.arad[g];
        }
        // CVM (drone_v2.py:178): velocity IS pref_velocity (same ndarray).  RVO (drone_v2.py:169-173): the velocity chosen
        // by d2d_rvo_kernel is an array of its own -- Agent.step rotates / bounces pref_velocity only and moves with the
        // velocity, which is published here as the agent's current one.
        double vx = pref.x, vy = pref.y;
        const bool rvo = P.motion_rvo != 0;
        if (rvo) {
            const double2 v = P.avel_next[g];
            P.avel[g] = v;
            vx = v.x; vy = v.y;
        }
        const double nx = pos.x + vx * P.dt, ny = pos.y + vy * P.dt;
        bool rebound = false;
        if (d2d_norm2_le(vx, vy, 5.0)) {   // utils.py:476-477: rotation by 30 deg rebinds pref_velocity
            const double qx = D2D_FMA(C6, pref.x, -S6 * pref.y);
            const double qy = D2D_FMA(S6, pref.x, C6 * pref.y);
            pref.x = qx; pref.y = qy;
            rebound = true;
        }
        const double edge = P.scale;
        if (nx < edge + r) pref.x = fabs(pref.x);
        else if (nx > P.map_w - edge - r) pref.x = -fabs(pref.x);
        if (ny < edge + r) pref.y = fabs(pref.y);
        else if (ny > P.map_h - edge - r) pref.y = -fabs(pref.y);
        if (!rebound && !rvo) { vx = pref.x; vy = pref.y; }   // CVM aliasing: the bounce is visible through velocity
        pos.x = pos.x + vx * P.dt;
        pos.y = pos.y + vy * P.dt;
        P.apos[g] = pos;
        P.apref[g] = pref;
        if (PF && keep_pos && w == tid) { *keep_pos = pos; *keep_pref = pref; }   // multi-step kernels: next step's input
        const int q = i * NP + k;
        c.sx[q] = pos.x; c.sy[q] = pos.y; c.sr2[q] = r * r;
        // broad phase: a ray sample is never farther than depth + 9*sqrt(2) from the drone
        const double ddx = pos.x - s.px, ddy = pos.y - s.py;
        const double reach = r + P.cull_reach;
        if (ddx * ddx + ddy * ddy <= reach * reach) {
            const int slot = atomicAdd(&s.ncull, 1);
            c.cull[i * NP + slot] = (uint16_t)k;
        }
        if (COLLIDE_HERE) {   // Drone2D.is_collide utils.py:773-776 (drone does not move under NoMove)
            if (d2d_norm2_lt(ddx, ddy, r + P.drone_r)) atomicOr(&s.coll_agent, 1);
        }
    }
}

// ------------------------------------------------------------------------------------------ P2: Raycast.castRay
struct RayOut {
    uint8_t *bel_s;           // belief grid in shared memory
    int e;                    // env index: the HBM addresses (belief row, local_map slice, host mirror) are formed from the
                              // kernel parameters on the rare store path instead of living in registers across the march
    int patch;                // 1: the env's local_map slice is patched in place (window unchanged this step)
    int wi, wj;               // window origin cell (ix-16, iy-16)
    int border_ok;            // 1: every border cell of this env's ground truth is a wall (no ray can leave the grid)
    uint32_t *chg;            // optional shared-memory list of changed cells (cell | value << 16), null if unused
    int *nchg;                // its counter (entries beyond the capacity are counted but not stored)
    int defer_mirror;         // 1: host-mirror stores of patched cells are NOT issued here but replayed from `chg` at the end of
                              // the step (fused warp kernel: keeps PCIe stores out of the march and behind the action gate)
};
#define D2D_CHG_CAP 64
#define D2D_ACTION_SENTINEL 0x7FF8D2D0AC710F05ull      // a NaN payload no caller produces: "action not delivered yet"
#define D2D_FUSED_WARP_EXTRA (D2D_CHG_CAP * 4 + 16)   // changed-cell list + counter behind every warp slice of the fused kernel

// a belief cell changes value (0 -> 1 or 0 -> 2): shared copy, HBM grid, and whatever mirrors the observation
__device__ __forceinline__ void d2d_mark_store(const DevP &P, const RayOut &o, int cell, uint8_t v) {
    o.bel_s[cell] = v;
#if defined(D2D_WARP_PROF) && D2D_WARP_PROF >= 2        // counters perturb the timing: tools/resident_timeline.py --counters
    atomicAdd(&P.prof[(size_t)o.e * 12 + 5], 1ull);     // marks of this env (accumulated over the steps of a launch)
#endif
    P.belief[(size_t)o.e * D2D_BELIEF_STRIDE + cell] = v;
    if (o.patch) {          // the cell is always inside the 33x33 window (view reach < 16 cells)
        const int ci = cell / D2D_GRID, cj = cell - ci * D2D_GRID;
        const int u = ci - o.wi, w = cj - o.wj;
        if ((unsigned)u < (unsigned)D2D_LOCAL && (unsigned)w < (unsigned)D2D_LOCAL) {
            const size_t off = (size_t)o.e * D2D_LOCAL_CELLS + u * D2D_LOCAL + w;
            P.local_map[off] = v;
            if (P.lm_mirror && !o.defer_mirror) {  // one byte over PCIe; counted in the padding word behind the shared belief grid
                P.lm_mirror[off] = v;
                atomicAdd((int *)(o.bel_s + D2D_MIRCNT_OFF), 1);
            }
        }
    }
    if (o.chg) {
        const int slot = atomicAdd(o.nchg, 1);
        if (slot < D2D_CHG_CAP) o.chg[slot] = (uint32_t)cell | ((uint32_t)v << 16);
    }
}
__device__ __forceinline__ void d2d_mark(const DevP &P, const RayOut &o, int ci, int cj, uint8_t v) {
    const int cell = ci * D2D_GRID + cj;
    if (o.bel_s[cell] != v) d2d_mark_store(P, o, cell, v);   // monotone + idempotent: every writer of a cell writes the same value
}

// wrapped ray angle, utils.py:594, 626, 612-618
__device__ __forceinline__ double d2d_ray_angle(const DevP &P, double yaw, int ray) {
    const double ray_angle = P.ray_a0 + P.ray_da * (double)ray;
    const double player_angle = D2D_TWO_PI - yaw * D2D_DEG2RAD;
    double a = player_angle + ray_angle;
    a = copysign(d2d_pymod(fabs(a), D2D_TWO_PI), a);
    if (a < 0) a += D2D_TWO_PI;
    return a;
}

// Hits on the first 32 entries of the culled list are returned as a bit mask over the LIST SLOTS (the caller ORs the
// masks of its rays and publishes them once: no shared-memory atomics inside the march, where a disc seen by ~20 rays
// at the same sample index would serialise them); hits on the unfiltered tail go to `hitw` directly.
// SMALL: the culled list never exceeds 32 entries (at most 32 agents), so there is no tail and `hitw` is not used.
template <bool SAFE = false, bool SMALL = false>
__device__ __forceinline__ uint32_t d2d_cast_ray(const DevP &P, const EnvS &s, double a, double slope, const RayOut &o,
                                                 const uint64_t *gt, const double *sx, const double *sy, const double *sr2,
                                                 const uint16_t *cull, uint32_t *hitw) {
    uint32_t hm = 0u;
    const bool faced_right = (a < 90.0 * D2D_DEG2RAD) || (a > 270.0 * D2D_DEG2RAD);
    const bool faced_up = a > D2D_PI;
    const double step = P.scale - 1.0;
    double xs, ys;
    if (fabs(slope) > 1.0) {
        slope = 1.0 / slope;
        ys = faced_up ? -step : step;
        xs = ys * slope;
    } else {
        xs = faced_right ? step : -step;
        ys = xs * slope;
    }
    const double x0 = s.px, y0 = s.py;
    const int nc = s.ncull;
    // Per-ray prefilter (conservative): a culled disc can only contain a sample of this ray if its centre lies within
    // r (+slack) of the ray's line.  |cross((c - p), d)| <= (r + slack) * |d|, compared squared.  Most rays have no
    // candidate and skip the per-sample disc loop entirely.  For the others the candidates are kept as a bit mask over
    // the culled list (entries >= 32 are not filtered) together with the window of sample indices that can lie inside
    // any candidate disc: sample m sits at p + m*d (+ ~1e-12 of accumulated rounding), so it is inside disc (c, r) only
    // if |m - t| <= r / |d| with t = (c - p).d / |d|^2 -- evaluated in fp32 with a 0.05-sample margin, five orders of
    // magnitude above the fp32 error.  The decision itself stays the reference's sampled point-in-disc test below.
    uint32_t cmask = 0u;
    int mlo = 0x7fff, mhi = -1;
    {
        const double dd2 = xs * xs + ys * ys;
        const float inv_dd2 = 1.0f / (float)dd2;
        const int ncm = (SMALL || nc < 32) ? nc : 32;
#pragma unroll 1
        for (int q = 0; q < ncm; q++) {
            const int k = cull[q];
            const double cx = sx[k] - x0, cy = sy[k] - y0;
            const double cr = cx * ys - cy * xs;
            const double rr = sr2[k] * 1.000001 + 1e-3;          // (r + slack)^2 upper bound
            if (cr * cr <= rr * dd2) {
                cmask |= 1u << q;
                const float t = (float)(cx * xs + cy * ys) * inv_dd2;
                const float hw = sqrtf((float)rr * inv_dd2) + 0.05f;
                mlo = min(mlo, (int)ceilf(t - hw));
                mhi = max(mhi, (int)floorf(t + hw));
            }
        }
        if (!SMALL && nc > 32) { mlo = 0; mhi = 0x7fff; }        // unfiltered tail of a very long culled list
    }
    const unsigned mspan = mhi >= mlo ? (unsigned)(mhi - mlo) : 0u;   // no candidate: mlo = 0x7fff, (m - mlo) wraps to huge
    // The march runs in MIRRORED coordinates: u = x when the ray moves up the axis, -x when it moves down (negation is
    // exact and round-to-nearest is sign-symmetric, so u accumulates bit for bit like x).  In these coordinates every ray
    // moves towards +u, the next cell boundary ub is always ahead and always advances by +scale, and the only direction
    // dependence left is the strictness of the crossing test.
    // int(x // scale) is tracked incrementally: |step| < scale, so a sample moves at most one cell per axis, and
    // x in [scale*ci, scale*(ci+1)) is exactly CPython's floor (multiples of the scale are exact doubles):
    //   moving up  : new cell iff x >= scale*(ci+1)            <=> u >= ub
    //   moving down: new cell iff x <  scale*ci  <=> -x > -scale*ci  <=> u >  ub
    if (SAFE) {
        // Belief-first march for envs whose border ring is all wall (o.border_ok) and whose drone is inside the grid: a ray
        // cannot leave the grid without entering a wall cell first (|step| < cell size), so the loop condition of
        // utils.py:654 can only fail on a border cell, where it is checked exactly.  The belief grid itself tells what the
        // ground truth of a visited cell is (2 = free, 1 = wall; it is only ever written from the ground truth), so the
        // bitmap is consulted for unexplored cells only, and only the linear cell index is tracked.
        const bool xup = xs > 0.0, yup = ys > 0.0;
        int dcx = xup ? D2D_GRID : -D2D_GRID, dcy = yup ? 1 : -1;
        // opaque to the optimiser from here on: otherwise it re-derives both increments from the signs of xs / ys in every
        // iteration instead of keeping two registers
        asm volatile("" : "+r"(dcx), "+r"(dcy));
        const double uxs = fabs(xs), uys = fabs(ys);
        const double ux0 = xup ? x0 : -x0, uy0 = yup ? y0 : -y0;
        double ux = ux0, uy = uy0;
        double uxb = xup ? P.scale * (double)(s.ix + 1) : -(P.scale * (double)s.ix);
        double uyb = yup ? P.scale * (double)(s.iy + 1) : -(P.scale * (double)s.iy);
        const double scale = P.scale;
        // the loop variable is the SHARED-MEMORY ADDRESS of the current belief cell (one LDS per sample, no index arithmetic)
        const uint32_t bel0 = d2d_smem_u32(o.bel_s);
        uint32_t caddr = bel0 + (uint32_t)(s.ix * D2D_GRID + s.iy);
        int m = 0;
        for (;;) {
            if ((unsigned)(m - mlo) <= mspan) {
                const double x = dcx > 0 ? ux : -ux, y = dcy > 0 ? uy : -uy;
                if (!(0.0 < x && 0.0 < y)) break;                      // utils.py:654 comes before the agent test
                bool any = false;
                uint32_t mm = cmask;
                while (mm) {
                    const int q = __ffs(mm) - 1;
                    mm &= mm - 1u;
                    const int k = cull[q];
                    const double ex = sx[k] - x, ey = sy[k] - y;
                    if (ex * ex + ey * ey <= sr2[k]) { hm |= 1u << q; any = true; }
                }
                if (!SMALL) {
#pragma unroll 1
                    for (int q = 32; q < nc; q++) {
                        const int k = cull[q];
                        const double ex = sx[k] - x, ey = sy[k] - y;
                        if (ex * ex + ey * ey <= sr2[k]) { atomicOr(&hitw[k >> 5], 1u << (k & 31)); any = true; }
                    }
                }
                if (any) break;
            }
            uint32_t bel;
            asm volatile("ld.shared.u8 %0, [%1];" : "=r"(bel) : "r"(caddr));
            if (bel != 2u) {
                if (bel == 1u) break;                                  // known wall: nothing to mark
                const int cell = (int)(caddr - bel0);
                const int ci = cell / D2D_GRID, cj = cell - ci * D2D_GRID;
                if ((gt[ci] >> cj) & 1ull) {                           // unexplored wall cell (utils.py:666-670)
                    bool in_map = true;                                // a sample exactly on x == 0 or y == 0 ends the loop first
                    if (ci == 0 || cj == 0) {
                        const double x = dcx > 0 ? ux : -ux, y = dcy > 0 ? uy : -uy;
                        in_map = 0.0 < x && 0.0 < y;
                    }
                    if (in_map) d2d_mark_store(P, o, cell, 1);
                    break;
                }
                if (m >= P.m_far) {
                    const double fx = ux - ux0, fy = uy - uy0;
                    if ((fx * fx + fy * fy) >= P.depth2) break;
                }
                d2d_mark_store(P, o, cell, 2);
            } else if (m >= P.m_far) {                                 // explored free cell: only the view depth can end the ray
                const double fx = ux - ux0, fy = uy - uy0;             // = +-(x - px): same square
                if ((fx * fx + fy * fy) >= P.depth2) break;
            }
            m += 1;
            // advance one sample and track the cell (see the general march below for the derivation): a new cell on an axis
            // iff u >= ub, except that a sample exactly on the boundary stays in its cell when the ray moves DOWN that axis.
            // Written out as predicated PTX: 7 instructions per axis.
            asm("{\n\t"
                ".reg .pred pe, pn;\n\t"
                "add.rn.f64 %0, %0, %3;\n\t"
                "setp.lt.s32 pn, %4, 0;\n\t"
                "setp.eq.and.f64 pe, %0, %1, pn;\n\t"
                "setp.lt.or.f64 pe, %0, %1, pe;\n\t"
                "@!pe add.s32 %2, %2, %4;\n\t"
                "@!pe add.rn.f64 %1, %1, %5;\n\t"
                "}" : "+d"(ux), "+d"(uxb), "+r"(caddr) : "d"(uxs), "r"(dcx), "d"(scale));
            asm("{\n\t"
                ".reg .pred pe, pn;\n\t"
                "add.rn.f64 %0, %0, %3;\n\t"
                "setp.lt.s32 pn, %4, 0;\n\t"
                "setp.eq.and.f64 pe, %0, %1, pn;\n\t"
                "setp.lt.or.f64 pe, %0, %1, pe;\n\t"
                "@!pe add.s32 %2, %2, %4;\n\t"
                "@!pe add.rn.f64 %1, %1, %5;\n\t"
                "}" : "+d"(uy), "+d"(uyb), "+r"(caddr) : "d"(uys), "r"(dcy), "d"(scale));
        }
#if defined(D2D_WARP_PROF) && D2D_WARP_PROF >= 2
        atomicAdd(&P.prof[(size_t)o.e * 12 + 6], (unsigned long long)(m + 1));   // samples marched by this env's rays
        atomicMax(&P.prof[(size_t)o.e * 12 + 7], (unsigned long long)(m + 1));   // longest ray
#endif
        return hm;
    }
    int ci = s.ix, cj = s.iy;
    const bool xup = xs > 0.0, yup = ys > 0.0;
    const int sxi = xup ? 1 : -1, syi = yup ? 1 : -1;
    const double uxs = fabs(xs), uys = fabs(ys);
    double ux = xup ? x0 : -x0, uy = yup ? y0 : -y0;
    double uxb = xup ? P.scale * (double)(ci + 1) : -(P.scale * (double)ci);
    double uyb = yup ? P.scale * (double)(cj + 1) : -(P.scale * (double)cj);
    // sample m lies at most m * step * sqrt(2) from the drone: while that bound is below the view depth the
    // `dist >= depth^2` test (utils.py:668) cannot fire and is skipped (P.m_far, margin >> accumulated rounding).
    int m = 0;
    for (;;) {
        // loop condition utils.py:654: 0 < x < W and 0 < y < H; interior cells satisfy it by construction
        if ((unsigned)(ci - 1) >= (unsigned)(D2D_GRID - 2) || (unsigned)(cj - 1) >= (unsigned)(D2D_GRID - 2)) {
            const double x = xup ? ux : -ux, y = yup ? uy : -uy;
            if (!(0.0 < x && x < P.map_w && 0.0 < y && y < P.map_h)) break;
        }
        if ((unsigned)(m - mlo) <= mspan) {
            const double x = xup ? ux : -ux, y = yup ? uy : -uy;
            bool any = false;
            uint32_t mm = cmask;
            while (mm) {
                const int q = __ffs(mm) - 1;
                mm &= mm - 1u;
                const int k = cull[q];
                const double ex = sx[k] - x, ey = sy[k] - y;
                if (ex * ex + ey * ey <= sr2[k]) {
                    hm |= 1u << q;
                    any = true;
                }
            }
            if (!SMALL) {
#pragma unroll 1
                for (int q = 32; q < nc; q++) {
                    const int k = cull[q];
                    const double ex = sx[k] - x, ey = sy[k] - y;
                    if (ex * ex + ey * ey <= sr2[k]) {
                        atomicOr(&hitw[k >> 5], 1u << (k & 31));
                        any = true;
                    }
                }
            }
            if (any) break;
        }
        const bool wall = (gt[ci] >> cj) & 1ull;
        bool far = false;
        if (m >= P.m_far) {
            const double fx = ux - (xup ? x0 : -x0), fy = uy - (yup ? y0 : -y0);   // = +-(x - px): same square
            far = (fx * fx + fy * fy) >= P.depth2;
        }
        if (wall || far) {
            if (wall) d2d_mark(P, o, ci, cj, 1);
            break;
        }
        d2d_mark(P, o, ci, cj, 2);
        ux = ux + uxs;
        uy = uy + uys;
        m += 1;
        bool cx = ux >= uxb, cy = uy >= uyb;
        if (ux == uxb || uy == uyb) {       // a sample exactly on a cell boundary (rare): moving down it stays in its cell
            if (ux == uxb && !xup) cx = false;
            if (uy == uyb && !yup) cy = false;
        }
        if (cx) { ci += sxi; uxb += P.scale; }
        if (cy) { cj += syi; uyb += P.scale; }
    }
    return hm;
}

// publish a slot mask returned by d2d_cast_ray: bit q -> agent cull[q]
__device__ __forceinline__ void d2d_publish_hits(uint32_t hm, const uint16_t *cull, uint32_t *hitw) {
    while (hm) {
        const int q = __ffs(hm) - 1;
        hm &= hm - 1u;
        const int k = cull[q];
        atomicOr(&hitw[k >> 5], 1u << (k & 31));
    }
}

__device__ __forceinline__ void d2d_phase_rays(const DevP &P, const BlockCtx &c, int env0, int E, int tid, int T) {
    const int R = P.n_rays, NP = P.NP;
    for (int w = tid; w < E * R; w += T) {
        const int i = w / R, ray = w - i * R;
        const EnvS &s = c.S[i];
        if (!s.valid) continue;
        RayOut o;
        o.bel_s = c.belief + (size_t)i * D2D_BELIEF_STRIDE;
        o.e = env0 + i; o.patch = 0; o.wi = 0; o.wj = 0; o.border_ok = 0; o.chg = nullptr; o.nchg = nullptr; o.defer_mirror = 0;
        const double a = d2d_ray_angle(P, s.yaw, ray);
        const uint32_t hm = d2d_cast_ray(P, s, a, d2d_tan(a), o, c.gt + (size_t)i * D2D_GRID, c.sx + i * NP, c.sy + i * NP,
                                         c.sr2 + i * NP, c.cull + i * NP, c.hitw + i * P.HW);
        d2d_publish_hits(hm, c.cull + i * NP, c.hitw + i * P.HW);
    }
}

// all 196 border cells of the env's ground truth are walls (true for every world unless an agent disc erased border
// cells at world generation, utils.py:508-525); evaluated by one warp on the shared-memory row bitmap
__device__ __forceinline__ int d2d_border_intact(const uint64_t *gt, int lane) {
    const uint64_t FULL = (1ull << D2D_GRID) - 1ull, EDGE = 1ull | (1ull << (D2D_GRID - 1));
    bool ok = true;
#pragma unroll
    for (int r = lane; r < D2D_GRID; r += 32) {
        const uint64_t need = (r == 0 || r == D2D_GRID - 1) ? FULL : EDGE;
        ok = ok && ((gt[r] & need) == need);
    }
    return __all_sync(0xffffffffu, ok) ? 1 : 0;
}

// one env per warp: lane handles rays `lane` and `lane + 32` (+64, ...); the two tangent evaluations of a pair are
// independent straight-line code, which gives the scheduler two dependency chains to interleave
// one env per warp.  ILP2: lane handles rays `lane` and `lane + 32` with the two tangent evaluations as independent
// straight-line code (two dependency chains for the scheduler; best when all warps run in phase, i.e. one wave).
// Otherwise a single copy of the ray body (half the code: best when many waves de-phase the warps and the
// instruction cache becomes the limiter).
// SMALL (at most 32 agents, single-copy march only): the env's hit mask over AGENTS is returned in every lane instead of
// being published into the hit words.
template <bool ILP2, bool SMALL = false>
__device__ __forceinline__ uint32_t d2d_phase_rays_warp(const DevP &P, const BlockCtx &c, const RayOut &o, int lane) {
    static_assert(!(ILP2 && SMALL), "the small-crowd form casts one ray per lane per pass");
    const EnvS &s = c.S[0];
    const int R = P.n_rays;
    uint32_t hm = 0u;
    if (ILP2) {
        for (int r0 = lane; r0 < R; r0 += 64) {
            const int r1 = r0 + 32;
            const double a0 = d2d_ray_angle(P, s.yaw, r0), a1 = d2d_ray_angle(P, s.yaw, r1);
            const double t0 = d2d_tan(a0), t1 = d2d_tan(a1);
            hm |= d2d_cast_ray(P, s, a0, t0, o, c.gt, c.sx, c.sy, c.sr2, c.cull, c.hitw);
            if (r1 < R) hm |= d2d_cast_ray(P, s, a1, t1, o, c.gt, c.sx, c.sy, c.sr2, c.cull, c.hitw);
        }
    } else {
        // warp-uniform: border ring intact and drone inside the grid -> the belief-first march
        const bool safe = o.border_ok && (unsigned)s.ix < (unsigned)D2D_GRID && (unsigned)s.iy < (unsigned)D2D_GRID;
#pragma unroll 1
        for (int ray = lane; ray < R; ray += 32) {
            const double a = d2d_ray_angle(P, s.yaw, ray);
            const double tn = d2d_tan(a);
            if (safe) hm |= d2d_cast_ray<true, SMALL>(P, s, a, tn, o, c.gt, c.sx, c.sy, c.sr2, c.cull, c.hitw);
            else hm |= d2d_cast_ray<false, SMALL>(P, s, a, tn, o, c.gt, c.sx, c.sy, c.sr2, c.cull, c.hitw);
        }
    }
    // OR over the warp, then lane q publishes slot q (all rays of the env are cast by this warp)
    hm = __reduce_or_sync(0xffffffffu, hm);
    if (SMALL) return __reduce_or_sync(0xffffffffu, ((hm >> lane) & 1u) ? 1u << c.cull[lane] : 0u);
    if ((hm >> lane) & 1u) {
        const int k = c.cull[lane];
        atomicOr(&c.hitw[k >> 5], 1u << (k & 31));
    }
    return 0u;
}

// ------------------------------------------------------------------------------------------ noisy measurements
// NumPy legacy RandomState (MT19937 + polar gaussian with a cached second value), one stream per env, continued from the
// state left by world generation (drone_v2.py:80, 54).  utils.py:605 draws randn(2) for every in-view agent in index
// order, so lane 0 walks the hit mask sequentially.
struct D2DRng {
    uint32_t *key;      // [624] in HBM
    int pos, has;
    double gauss;
};
__device__ __noinline__ void d2d_mt_regen(uint32_t *mt) {
    const uint32_t UP = 0x80000000u, LO = 0x7fffffffu, MA = 0x9908b0dfu;
    int kk;
    uint32_t y;
#pragma unroll 1
    for (kk = 0; kk < 624 - 397; kk++) { y = (mt[kk] & UP) | (mt[kk + 1] & LO); mt[kk] = mt[kk + 397] ^ (y >> 1) ^ ((y & 1u) ? MA : 0u); }
#pragma unroll 1
    for (; kk < 623; kk++) { y = (mt[kk] & UP) | (mt[kk + 1] & LO); mt[kk] = mt[kk + (397 - 624)] ^ (y >> 1) ^ ((y & 1u) ? MA : 0u); }
    y = (mt[623] & UP) | (mt[0] & LO); mt[623] = mt[396] ^ (y >> 1) ^ ((y & 1u) ? MA : 0u);
}
__device__ __forceinline__ uint32_t d2d_mt_next32(D2DRng &r) {
    if (r.pos == 624) { d2d_mt_regen(r.key); r.pos = 0; }
    uint32_t y = r.key[r.pos++];
    y ^= (y >> 11); y ^= (y << 7) & 0x9d2c5680u; y ^= (y << 15) & 0xefc60000u; y ^= (y >> 18);
    return y;
}
__device__ __forceinline__ double d2d_mt_next_double(D2DRng &r) {
    const int a = (int)(d2d_mt_next32(r) >> 5), b = (int)(d2d_mt_next32(r) >> 6);
    return ((double)a * 67108864.0 + (double)b) / 9007199254740992.0;
}
__device__ __noinline__ double d2d_legacy_gauss(D2DRng &r) {
    if (r.has) { const double t = r.gauss; r.has = 0; r.gauss = 0.0; return t; }
    double f, x1, x2, r2;
    do {
        x1 = 2.0 * d2d_mt_next_double(r) - 1.0;
        x2 = 2.0 * d2d_mt_next_double(r) - 1.0;
        r2 = x1 * x1 + x2 * x2;
    } while (r2 >= 1.0 || r2 == 0.0);
    f = D2D_SQRT(-2.0 * log(r2) / r2);        // device log: <= 1 ulp from glibc's (continuous tolerance 1e-9)
    r.gauss = f * x1; r.has = 1;
    return f * x2;
}
// measurement = position + sigma * randn(2) for every hit agent of ONE env (warp path; called by lane 0)
__device__ __forceinline__ void d2d_measure_env(const DevP &P, const BlockCtx &c, int e) {
    D2DRng r;
    r.key = P.rng_key + (size_t)e * 624; r.pos = P.rng_pos[e]; r.has = P.rng_has[e]; r.gauss = P.rng_gauss[e];
    bool used = false;
#pragma unroll 1
    for (int k = 0; k < P.N; k++) {
        if (!((c.hitw[k >> 5] >> (k & 31)) & 1u)) continue;
        const double g0 = d2d_legacy_gauss(r), g1 = d2d_legacy_gauss(r);
        c.mx[k] = c.sx[k] + P.var_cam * g0;
        c.my[k] = c.sy[k] + P.var_cam * g1;
        used = true;
    }
    if (used) { P.rng_pos[e] = r.pos; P.rng_has[e] = r.has; P.rng_gauss[e] = r.gauss; }
}

// ------------------------------------------------------------------------------------------ P3: hit mask + trackers
__device__ D2D_COLD void d2d_tracker_update(const DevP &P, EnvS &s, size_t g, bool measured, double z0, double z1,
                                            bool was_active) {
    // KalmanFilter.update utils.py:242-275; F = I + 0.1*shift, H = [I 0], Sigma_z = var_cam*I, Sigma_x = q*I
    const double q = (P.var_cam != 0.0) ? 0.1 : 0.001;
    double *mu = P.trk_mu + g * 4, *Sg = P.trk_sigma + g * 16;
    bool active = was_active;                      // already false for an env that is being reset
    int ts = s.reset ? 1 : P.trk_ts[g];
    if (s.reset) {   // fresh KalmanFilter(params) + drone_v2.py:46 radius
        P.trk_radius[g] = P.trk_radius0[g];
        P.trk_active[g] = 0;
        P.trk_ts[g] = 1;
        if (!measured) {   // mu_upds = [zeros], Sigma_upds = [diag(1, 1, 10, 10)] (utils.py:181-197): same state as the eager reset
#pragma unroll
            for (int i = 0; i < 4; i++) mu[i] = 0.0;
#pragma unroll
            for (int i = 0; i < 16; i++) Sg[i] = (i == 0 || i == 5) ? 1.0 : ((i == 10 || i == 15) ? 10.0 : 0.0);
        }
    }
    if (!active && !measured) return;
    double m[4], S[16];
    if (active) {
#pragma unroll
        for (int i = 0; i < 4; i++) m[i] = mu[i];
#pragma unroll
        for (int i = 0; i < 16; i++) S[i] = Sg[i];
        // predict utils.py:225-233, in place: Sigma <- F Sigma F^T + Q with F = I + 0.1*[[0,I],[0,0]]
        m[0] = m[0] + 0.1 * m[2];
        m[1] = m[1] + 0.1 * m[3];
#pragma unroll
        for (int j = 0; j < 4; j++) {   // rows 0,1 += 0.1 * rows 2,3   (F Sigma)
            S[j] = S[j] + 0.1 * S[8 + j];
            S[4 + j] = S[4 + j] + 0.1 * S[12 + j];
        }
#pragma unroll
        for (int i = 0; i < 4; i++) {   // cols 0,1 += 0.1 * cols 2,3   ((F Sigma) F^T)
            S[4 * i + 0] = S[4 * i + 0] + 0.1 * S[4 * i + 2];
            S[4 * i + 1] = S[4 * i + 1] + 0.1 * S[4 * i + 3];
        }
        S[0] += q; S[5] += q; S[10] += q; S[15] += q;
        ts += 1;
        const double lo = 10.0 + P.agent_radius;
        if (S[0] >= 150.0 || !(lo < m[0] && m[0] < P.map_w - 10.0 - P.agent_radius) ||
            !(lo < m[1] && m[1] < P.map_h - 10.0 - P.agent_radius)) {
            // utils.py:235-239: archive a copy, re-initialise (inactive, default radius)
            atomicAdd(&s.arch_cnt, 1);
            atomicAdd(&s.arch_ts, ts);
            active = false;
            P.trk_radius[g] = P.agent_radius;
            m[0] = m[1] = m[2] = m[3] = 0.0;
#pragma unroll
            for (int i = 0; i < 16; i++) S[i] = 0.0;
            S[0] = 1.0; S[5] = 1.0; S[10] = 10.0; S[15] = 10.0;
            ts = 1;
        }
        if (measured) {   // utils.py:249-260
            const double rz = P.var_cam;
            const double s00 = rz + S[0], s01 = S[1], s10 = S[4], s11 = rz + S[5];
            const double det = s00 * s11 - s01 * s10;
            const double idet = 1.0 / det;       // np.linalg.inv of the 2x2 innovation covariance (tolerance 1e-9, not bit-exact)
            const double i00 = s11 * idet, i01 = -s01 * idet, i10 = -s10 * idet, i11 = s00 * idet;
            const double r0 = z0 - m[0], r1 = z1 - m[1];
            // rows 3, 2 first (they need the ORIGINAL rows 0 and 1), then rows 0 and 1 together
#pragma unroll
            for (int i = 3; i >= 2; i--) {
                const double k0 = S[4 * i] * i00 + S[4 * i + 1] * i10, k1 = S[4 * i] * i01 + S[4 * i + 1] * i11;
                m[i] = m[i] + (k0 * r0 + k1 * r1);
#pragma unroll
                for (int j = 0; j < 4; j++) S[4 * i + j] = ((-k0) * S[j] + (-k1) * S[4 + j]) + S[4 * i + j];
            }
            {
                const double k00 = S[0] * i00 + S[1] * i10, k01 = S[0] * i01 + S[1] * i11;
                const double k10 = S[4] * i00 + S[5] * i10, k11 = S[4] * i01 + S[5] * i11;
                m[0] = m[0] + (k00 * r0 + k01 * r1);
                m[1] = m[1] + (k10 * r0 + k11 * r1);
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const double a0 = S[j], a1 = S[4 + j];
                    S[j] = (1.0 - k00) * a0 + (-k01) * a1;
                    S[4 + j] = (-k10) * a0 + (1.0 - k11) * a1;
                }
            }
        }
    } else {   // first sighting utils.py:263-273
        m[0] = z0; m[1] = z1; m[2] = 0.0; m[3] = 0.0;
#pragma unroll
        for (int i = 0; i < 16; i++) S[i] = 0.0;
        S[0] = 1.0; S[5] = 1.0; S[10] = 10.0; S[15] = 10.0;
        ts = 1;
        active = true;
    }
#pragma unroll
    for (int i = 0; i < 4; i++) mu[i] = m[i];
#pragma unroll
    for (int i = 0; i < 16; i++) Sg[i] = S[i];
    P.trk_active[g] = active ? 1 : 0;
    P.trk_ts[g] = ts;
    if (active) {
        atomicAdd(&s.act_cnt, 1);
        atomicAdd(&s.act_ts, ts);
    }
}

// PF: the caller (one warp, E == 1) loaded trk_active of tracker `tid` into pf_act at kernel entry, so the phase does not
// start with a DRAM round trip
template <bool PF = false>
__device__ __forceinline__ void d2d_phase_trackers(const DevP &P, const BlockCtx &c, int env0, int E, int tid, int T,
                                                   uint8_t pf_act = 0) {
    const int N = P.N, NP = P.NP;
#pragma unroll 1
    for (int w = tid; w < E * N; w += T) {
        const int i = w / N, k = w - i * N;
        EnvS &s = c.S[i];
        if (!s.valid) continue;
        const size_t g = (size_t)(env0 + i) * NP + k;
        const bool hit = (c.hitw[i * P.HW + (k >> 5)] >> (k & 31)) & 1u;
        P.hit[g] = hit ? 1 : 0;
        if (P.trackers) {
            const bool was_active = s.reset ? false : ((PF && w == tid) ? (pf_act != 0) : (P.trk_active[g] != 0));
            if (hit && !was_active) atomicAdd(&s.newly, 1);   // utils.py:606-607
            if (was_active || hit || s.reset) {
                const bool noisy = P.var_cam != 0.0;
                d2d_tracker_update(P, s, g, hit, noisy ? c.mx[i * NP + k] : c.sx[i * NP + k],
                                   noisy ? c.my[i * NP + k] : c.sy[i * NP + k], was_active);
            }
        }
    }
}

__device__ __forceinline__ void d2d_prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
// an active tracker's state (ts, mu, Sigma: 4 + 32 + 128 B) is needed long after the ray phase: have it waiting in L2
__device__ __forceinline__ void d2d_prefetch_tracker(const DevP &P, size_t g) {
    d2d_prefetch_l2(P.trk_ts + g);
    d2d_prefetch_l2(P.trk_mu + g * 4);
    d2d_prefetch_l2(P.trk_sigma + g * 16);
}

// ------------------------------------------------------------------------------------------ P4: leaders
__device__ __forceinline__ int d2d_gt_probe(const DevP &P, const uint64_t *gt, double x, double y) {
    if (x >= P.map_w || x < 0 || y >= P.map_h || y < 0) return 1;   // utils.py:546-547
    const int ci = d2d_cell(x, P.scale, P.inv_scale), cj = d2d_cell(y, P.scale, P.inv_scale);
    return (int)((gt[ci] >> cj) & 1ull);
}

// first half of Drone2DEnv2.step (drone_v2.py:153-163): counters, state machine, next target
__device__ __forceinline__ void d2d_leader_begin(const DevP &P, EnvS &s) {
    s.steps += 1;
    if (s.sm == SM_GOAL_REACHED) s.sm = SM_WAIT_FOR_GOAL;
    if (s.sm == SM_WAIT_FOR_GOAL) {
        if (s.tcur < P.n_targets) {
            s.tgx = P.targets[s.tcur][0];
            s.tgy = P.targets[s.tcur][1];
            s.tcur += 1;
        }
        s.sm = SM_PLANNING;
    }
}

// second half (drone_v2.py:196-235) after the planner verdict `success`
__device__ D2D_COLD void d2d_leader_finish(const DevP &P, EnvS &s, const uint64_t *gt, int e, double action,
                                                  bool success, bool with_yaw = true) {
    if (!success) {   // Drone2D.brake utils.py:755-762
        const double nv = d2d_norm2(s.vx, s.vy);
        if (nv <= P.max_acc * P.dt) { s.vx = 0.0; s.vy = 0.0; }
        else {
            s.vx = s.vx - s.vx / nv * P.max_acc * P.dt;
            s.vy = s.vy - s.vy / nv * P.max_acc * P.dt;
            s.px += s.vx * P.dt;
            s.py += s.vy * P.dt;
        }
        s.sm = SM_PLANNING;
        s.fail += 1;
    } else {
        s.sm = SM_EXECUTING;
        s.fail = 0;
    }
    // step_pos utils.py:733-739: pop one waypoint
    const int remaining = s.nseg * P.n_way - s.cursor;
    if (P.planner == D2D_PLANNER_JERK) {
        if (s.jerk_has) {       // acceleration, velocity = the waypoint's; x, y = round(position)
            P.drone_acc[e] = double2{s.jerk_ax, s.jerk_ay};
            s.vx = s.jerk_vx; s.vy = s.jerk_vy;
            s.px = rint(s.jerk_px); s.py = rint(s.jerk_py);
        }
    } else if (remaining > 0) {
        const int seg = s.cursor / P.n_way, ws = s.cursor - seg * P.n_way;
        const int ti = P.n_way - 1 - ws;
        const double *cf = P.traj_coeff + ((size_t)e * D2D_MAX_SEGMENTS + seg) * 6;
        const double t = P.tab->t_way[ti], t2 = P.tab->t_way2[ti], tt = P.tab->t_way_x2[ti];
        // np.array([1,t,t**2]) @ coeff.T on the reference image: fma(t2, h, p + t*v); then np.around, then round()
        s.px = rint(D2D_FMA(t2, cf[2], cf[0] + t * cf[1]));
        s.py = rint(D2D_FMA(t2, cf[5], cf[3] + t * cf[4]));
        s.vx = cf[1] + tt * cf[2];
        s.vy = cf[4] + tt * cf[5];
        s.cursor += 1;
        if (s.cursor == s.nseg * P.n_way) { s.nseg = 0; s.cursor = 0; }
    }
    // step_yaw utils.py:741-743 (the resident gated kernel runs everything above before the action is known, this after)
    if (with_yaw) s.yaw = d2d_pymod(s.yaw + (action * P.max_yaw_speed) * P.dt, 360.0);
}

// the five static probes of Drone2D.is_collide (utils.py:766-771); q = 0..4
__device__ __forceinline__ int d2d_static_probe(const DevP &P, const uint64_t *gt, double px, double py, int q) {
    const double r = P.drone_r;
    const double ox = (q == 0) ? -r : ((q == 2) ? r : 0.0), oy = (q == 3) ? -r : ((q == 4) ? r : 0.0);
    return d2d_gt_probe(P, gt, px + ox, py + oy);
}

__device__ D2D_COLD void d2d_leader_flags(const DevP &P, EnvS &s, const uint64_t *gt, int e, int static_hit = -1,
                                         bool mirror_scalars = true) {
    // is_collide utils.py:764-778
    int col = 0;
    if (static_hit < 0) {
        static_hit = 0;
        for (int q = 0; q < 5; q++) static_hit |= d2d_static_probe(P, gt, s.px, s.py, q);
    }
    if (static_hit) col = 1;
    else if (s.coll_agent) col = 2;
    int dead = 0, frz = 0;
    if (col == 0) {   // drone_v2.py:222-225
        if (d2d_norm2_le(s.px - s.tgx, s.py - s.tgy, 10.0)) s.sm = SM_GOAL_REACHED;
        dead = (s.fail >= 10 && D2D_FMA(s.vy, s.vy, s.vx * s.vx) == 0.0) ? 1 : 0;   // sqrt(t) == 0 <=> t == 0
        frz = ((double)s.steps >= P.max_steps && !dead) ? 1 : 0;
    }
    const int done = (col != 0 || dead || frz || (s.sm == SM_GOAL_REACHED && s.tcur >= P.n_targets)) ? 1 : 0;
    // tracker bookkeeping: archived this step (utils.py:238, drone_v2.py:187) + still-active ones at done (:232-235)
    s.bufc += s.arch_cnt; s.bufts += s.arch_ts; s.tracked += s.newly;
    if (done) { s.bufc += s.act_cnt; s.bufts += s.act_ts; }
    s.done_now = done;
    s.ix = d2d_cell(s.px, P.scale, P.inv_scale); s.iy = d2d_cell(s.py, P.scale, P.inv_scale);
    P.collision[e] = (uint8_t)col; P.dead_lock[e] = (uint8_t)dead; P.freezing[e] = (uint8_t)frz; P.done[e] = (uint8_t)done;
    if (mirror_scalars) P.yaw_obs[e] = (float)s.yaw;
    if (mirror_scalars) {        // the resident gated kernel publishes these per block, coalesced
        if (P.yaw_mirror) P.yaw_mirror[e] = (float)s.yaw;
        if (P.done_mirror) P.done_mirror[e] = (uint8_t)done;
    }
    if (done) {
        atomicAdd(&P.stats[D2D_STAT_EPISODES], 1ull);
        if (s.sm == SM_GOAL_REACHED) atomicAdd(&P.stats[D2D_STAT_SUCCESS], 1ull);
        if (col == 1) atomicAdd(&P.stats[D2D_STAT_STATIC_COLLISION], 1ull);
        if (col == 2) atomicAdd(&P.stats[D2D_STAT_DYNAMIC_COLLISION], 1ull);
        if (frz) atomicAdd(&P.stats[D2D_STAT_FREEZING], 1ull);
        if (dead) atomicAdd(&P.stats[D2D_STAT_DEAD_LOCK], 1ull);
        atomicAdd(&P.stats[D2D_STAT_FLIGHT_STEPS], (unsigned long long)s.steps);
        atomicAdd(&P.stats[D2D_STAT_AGENTS_TRACKED], (unsigned long long)s.bufc);
        atomicAdd(&P.stats[D2D_STAT_TRACKED_STEPS], (unsigned long long)s.bufts);
    }
}

// ------------------------------------------------------------------------------------------ P5: observation
// Drone2D.get_local_map utils.py:780-784: zero-padded 33x33 window centred on the drone's cell.  The block's E envs
// occupy E*1089 contiguous bytes of the observation tensor; E is a multiple of 4, so the slice is 4-byte aligned.
__device__ __forceinline__ void d2d_phase_obs(const DevP &P, const BlockCtx &c, int env0, int E, int tid, int T) {
    uint32_t *out = (uint32_t *)(P.local_map + (size_t)env0 * D2D_LOCAL_CELLS);
    uint32_t *out_m = P.lm_mirror ? (uint32_t *)(P.lm_mirror + (size_t)env0 * D2D_LOCAL_CELLS) : nullptr;
    const int words = E * D2D_LOCAL_CELLS / 4;
    for (int w = tid; w < words; w += T) {
        const int o = w * 4;
        const int i0 = o / D2D_LOCAL_CELLS;
        const int r = o - i0 * D2D_LOCAL_CELLS;
        const int u0 = r / D2D_LOCAL, v0 = r - u0 * D2D_LOCAL;
        uint32_t v = 0;
#pragma unroll
        for (int b = 0; b < 4; b++) {
            // byte b of the word: (env, row, col) derived independently (a word may straddle a row or an env)
            int vb = v0 + b, ub = u0, ib = i0;
            if (vb >= D2D_LOCAL) {
                vb -= D2D_LOCAL;
                ub += 1;
                if (ub >= D2D_LOCAL) { ub = 0; ib += 1; }
            }
            uint32_t cellv = 0;
            if (ib < E) {
                const EnvS &s = c.S[ib];
                const int gi = s.ix - 16 + ub, gj = s.iy - 16 + vb;
                if (s.valid && (unsigned)gi < (unsigned)D2D_GRID && (unsigned)gj < (unsigned)D2D_GRID)
                    cellv = c.belief[(size_t)ib * D2D_BELIEF_STRIDE + gi * D2D_GRID + gj];
            }
            v |= cellv << (8 * b);
        }
        out[w] = v;
        if (out_m) {                                   // the host buffer ends at byte B*1089: no store may cross it
            const size_t g = (size_t)env0 * D2D_LOCAL_CELLS + (size_t)o, end = (size_t)P.B * D2D_LOCAL_CELLS;
            if (g + 4 <= end) out_m[w] = v;
            else for (int b = 0; b < 4; b++) if (g + b < end) ((uint8_t *)out_m)[o + b] = (uint8_t)(v >> (8 * b));
        }
    }
    if (out_m && tid == 0) {
        const int nv = min(E, P.B - env0);
        atomicAdd(&P.stats[D2D_STAT_MIRROR_BYTES], (unsigned long long)(nv > 0 ? nv : 0) * D2D_LOCAL_CELLS);
    }
}

// explored-cell count of envs that finished this step (experiment.py:90 "Grid discovered")
__device__ __forceinline__ void d2d_phase_done_stats(const DevP &P, const BlockCtx &c, int E, int tid, int T) {
    int cnt = 0;
    for (int w = tid; w < E * D2D_CELLS; w += T) {
        const int i = w / D2D_CELLS, o = w - i * D2D_CELLS;
        if (c.S[i].valid && c.S[i].done_now && c.belief[(size_t)i * D2D_BELIEF_STRIDE + o] != 0) cnt++;
    }
    for (int off = 16; off > 0; off >>= 1) cnt += __shfl_down_sync(0xffffffffu, cnt, off);
    if ((tid & 31) == 0 && cnt) atomicAdd(&P.stats[D2D_STAT_GRID_DISCOVERED], (unsigned long long)cnt);
}

// ------------------------------------------------------------------------------------------ fused step (NoMove planner)
// Whole Drone2DEnv2.step in one launch when the planner is NoMove (traj_planner.py:68-76): the drone never moves,
// so the drone-vs-agent test can run with the agent phase and no planner kernel is needed.
template <int E>
__global__ void __launch_bounds__((E * 50 + 31) / 32 * 32, (E == 4 ? 4 : (E == 8 ? 2 : 1))) d2d_step_fused_kernel(const DevP P, const double *__restrict__ actions) {
    extern __shared__ __align__(128) unsigned char smem[];
    const BlockCtx c = d2d_carve(smem, E, P.NP, P.HW);
    const int tid = threadIdx.x, T = blockDim.x;
    const int env0 = blockIdx.x * E;

    if (tid == 0) { d2d_mbar_init(c.mbar, 1); c.misc[0] = 0; c.misc[1] = 0; }
    for (int w = tid; w < E * P.HW; w += T) c.hitw[w] = 0u;
    __syncthreads();
    if (tid < E) {
        d2d_load_env_scalars(P, c.S[tid], env0 + tid);
        if (c.S[tid].reset) c.misc[1] = 1;
    }
    __syncthreads();
    if (tid == 0) d2d_issue_bulk(P, c, env0, E, true);
    d2d_reset_arrays(P, c, env0, E, tid, T);
    d2d_phase_agents<true>(P, c, env0, E, tid, T);
    if (tid < E && c.S[tid].valid) d2d_leader_begin(P, c.S[tid]);
    __syncthreads();
    d2d_mbar_wait(c.mbar, 0);
    d2d_phase_rays(P, c, env0, E, tid, T);
    __syncthreads();
    d2d_phase_trackers(P, c, env0, E, tid, T);
    __syncthreads();
    if (tid < E && c.S[tid].valid) {
        EnvS &s = c.S[tid];
        const int e = env0 + tid;
        // NoMove.plan traj_planner.py:70-73 / NoMove.replan_check :75-76
        s.tgx = -1.0; s.tgy = -1.0;
        P.replan[e] = 0; P.plan_ok[e] = 1; P.need_plan[e] = 0;
        d2d_leader_finish(P, s, c.gt + (size_t)tid * D2D_GRID, e, actions[e], true);
        d2d_leader_flags(P, s, c.gt + (size_t)tid * D2D_GRID, e);
        d2d_store_env_scalars(P, s, e);
        if (s.done_now) c.misc[0] = 1;
    }
    if (tid == 0) {
        int nv = 0;
        for (int i = 0; i < E; i++) nv += c.S[i].valid;
        atomicAdd(&P.stats[D2D_STAT_ENV_STEPS], (unsigned long long)nv);
    }
    __syncthreads();
    d2d_phase_obs(P, c, env0, E, tid, T);
    if (c.misc[0]) d2d_phase_done_stats(P, c, E, tid, T);
}


// =============================================================================================================
// Warp-per-environment variant.  Same phase functions, but every warp owns ONE env (E = 1, T = 32) with a private
// shared-memory slice and its own mbarrier, so the phases are separated by __syncwarp() instead of block barriers:
// warps of a block never wait for each other (the block-wide version spent ~44 % of its stall samples in
// __syncthreads because the agent / tracker / leader phases have few work items).
// =============================================================================================================
__host__ __device__ inline size_t d2d_warp_slice_bytes(int NP, int HW, int extra) {
    size_t b = d2d_step_smem_bytes(1, NP, HW) + (size_t)extra;
    return (b + 127) / 128 * 128;
}

// observation of ONE env written by one warp: bytes [1089*e, 1089*e + 1089) of the tensor; the unaligned head / tail
// (1089 = 1 mod 4) go out as byte stores, the middle as coalesced 32-bit stores.
__device__ __forceinline__ uint32_t d2d_obs_cell(const uint8_t *bel, int ix, int iy, int k) {
    const int u = k / D2D_LOCAL, v = k - u * D2D_LOCAL;
    const int gi = ix - 16 + u, gj = iy - 16 + v;
    if ((unsigned)gi < (unsigned)D2D_GRID && (unsigned)gj < (unsigned)D2D_GRID) return bel[gi * D2D_GRID + gj];
    return 0u;
}

// 4 consecutive window bytes of row u starting at column v (bytes past column 32 are garbage, masked by the caller);
// window byte (u, v) = belief[ix-16+u][iy-16+v], zero outside the 50x50 grid (np.pad, utils.py:783).
__device__ __forceinline__ uint32_t d2d_win4(const uint8_t *bel, int ix, int iy, int u, int v) {
    const int gi = ix - 16 + u;
    if ((unsigned)gi >= (unsigned)D2D_GRID) return 0u;
    const int gj = iy - 16 + v;
    const int a = gi * D2D_GRID + gj;                 // byte address, may leave [0, 2500) by < 20 on masked bytes
    const int al = a & ~3;
    const uint32_t lo = (al >= 0) ? *(const uint32_t *)(bel + al) : 0u;
    const uint32_t hi = (al + 4 >= 0 && al + 4 < D2D_BELIEF_STRIDE) ? *(const uint32_t *)(bel + al + 4) : 0u;
    uint32_t w = __funnelshift_r(lo, hi, (a & 3) * 8);
    if ((unsigned)gj > (unsigned)(D2D_GRID - 4)) {     // some of the 4 columns fall outside [0, 50)
        uint32_t m = 0u;
#pragma unroll
        for (int b = 0; b < 4; b++)
            if ((unsigned)(gj + b) < (unsigned)D2D_GRID) m |= 0xFFu << (8 * b);
        w &= m;
    }
    return w;
}

__device__ __forceinline__ uint32_t d2d_obs_word(const uint8_t *bel, int ix, int iy, int k0) {
    // env-relative bytes k0..k0+3 of the row-major 33x33 window (k0 + 3 < 1089)
    const int u0 = k0 / D2D_LOCAL, v0 = k0 - u0 * D2D_LOCAL;
    uint32_t w = d2d_win4(bel, ix, iy, u0, v0);
    if (v0 > D2D_LOCAL - 4) {                          // the word wraps into the next row
        const int n1 = D2D_LOCAL - v0;                 // bytes taken from row u0 (1..3)
        const uint32_t w2 = d2d_win4(bel, ix, iy, u0 + 1, 0);
        w = (w & ((1u << (8 * n1)) - 1u)) | (w2 << (8 * n1));
    }
    return w;
}

__device__ D2D_COLD void d2d_obs_env_warp(const DevP &P, const uint8_t *bel, int ix, int iy, int e, int lane,
                                         bool to_mirror = true) {
    // bytes [1089*e, 1089*e + 1089) of the observation tensor: unaligned head / tail (1089 = 1 mod 4) as byte stores,
    // the middle as coalesced 32-bit stores assembled with funnel shifts from aligned shared-memory words.
    uint8_t *out = P.local_map + (size_t)e * D2D_LOCAL_CELLS;
    const int head = (4 - (e & 3)) & 3;                 // arena buffers are 256-B aligned
    const int nwords = (D2D_LOCAL_CELLS - head) >> 2;
    const int tail0 = head + 4 * nwords;
    uint8_t *out_m = (to_mirror && P.lm_mirror) ? P.lm_mirror + (size_t)e * D2D_LOCAL_CELLS : nullptr;   // base 4-byte aligned (checked at bind)
    if (lane < head) {
        const uint8_t v = (uint8_t)d2d_obs_cell(bel, ix, iy, lane);
        out[lane] = v;
        if (out_m) out_m[lane] = v;
    }
    if (lane < D2D_LOCAL_CELLS - tail0) {
        const uint8_t v = (uint8_t)d2d_obs_cell(bel, ix, iy, tail0 + lane);
        out[tail0 + lane] = v;
        if (out_m) out_m[tail0 + lane] = v;
    }
    uint32_t *ow = (uint32_t *)(out + head);
    uint32_t *ow_m = out_m ? (uint32_t *)(out_m + head) : nullptr;
#pragma unroll 1
    for (int j = lane; j < nwords; j += 32) {
        const uint32_t v = d2d_obs_word(bel, ix, iy, head + 4 * j);
        ow[j] = v;
        if (ow_m) ow_m[j] = v;
    }
    if (out_m && lane == 0) atomicAdd(&P.stats[D2D_STAT_MIRROR_BYTES], (unsigned long long)D2D_LOCAL_CELLS);
}

// NoMove: an env that is re-initialised keeps its window (same pose, new episode), so the observation of its first step is
// the ZERO window plus the cells that step marks: clear the slice with coalesced stores and let the rays patch it in place,
// instead of gathering 1089 bytes through the funnel-shift path after the step (~1000 warp-instructions on what are already
// the slowest warps of a step: fresh envs march every ray through unexplored cells).
__device__ __forceinline__ void d2d_obs_clear_warp(const DevP &P, int e, int lane, bool to_mirror) {
    uint8_t *out = P.local_map + (size_t)e * D2D_LOCAL_CELLS;
    uint8_t *out_m = (to_mirror && P.lm_mirror) ? P.lm_mirror + (size_t)e * D2D_LOCAL_CELLS : nullptr;
    const int head = (4 - (e & 3)) & 3;
    const int nwords = (D2D_LOCAL_CELLS - head) >> 2;
    const int tail0 = head + 4 * nwords;
    if (lane < head) { out[lane] = 0; if (out_m) out_m[lane] = 0; }
    if (lane < D2D_LOCAL_CELLS - tail0) { out[tail0 + lane] = 0; if (out_m) out_m[tail0 + lane] = 0; }
    uint32_t *ow = (uint32_t *)(out + head);
#pragma unroll 3
    for (int j = lane; j < nwords; j += 32) ow[j] = 0u;
    if (out_m) {
        uint32_t *om = (uint32_t *)(out_m + head);
#pragma unroll 3
        for (int j = lane; j < nwords; j += 32) om[j] = 0u;
        if (lane == 0) atomicAdd(&P.stats[D2D_STAT_MIRROR_BYTES], (unsigned long long)D2D_LOCAL_CELLS);
    }
}

// env e's freshly rewritten observation slice, device tensor -> host mirror (resident gated kernel: the rewrite itself runs
// before the gate, only this copy behind it).  Reads bypass L1: the slice was written by other lanes of this warp.
__device__ __forceinline__ void d2d_obs_mirror_copy_warp(const DevP &P, int e, int lane) {
    const uint8_t *src = P.local_map + (size_t)e * D2D_LOCAL_CELLS;
    uint8_t *dst = P.lm_mirror + (size_t)e * D2D_LOCAL_CELLS;
    const int head = (4 - (e & 3)) & 3;
    const int nwords = (D2D_LOCAL_CELLS - head) >> 2;
    const int tail0 = head + 4 * nwords;
    if (lane < head) dst[lane] = __ldcg(src + lane);
    if (lane < D2D_LOCAL_CELLS - tail0) dst[tail0 + lane] = __ldcg(src + tail0 + lane);
    const uint32_t *sw = (const uint32_t *)(src + head);
    uint32_t *dw = (uint32_t *)(dst + head);
    // all loads of a lane in flight before its first store: this copy sits on the critical path of the step's slowest envs
    uint32_t v[9];                                      // nwords <= 272 = 8.5 x 32
#pragma unroll
    for (int k = 0; k < 9; k++) { const int j = lane + 32 * k; v[k] = j < nwords ? __ldcg(sw + j) : 0u; }
#pragma unroll
    for (int k = 0; k < 9; k++) { const int j = lane + 32 * k; if (j < nwords) dw[j] = v[k]; }
    if (lane == 0) atomicAdd(&P.stats[D2D_STAT_MIRROR_BYTES], (unsigned long long)D2D_LOCAL_CELLS);
}

// explored-cell count of an env that finished this step (experiment.py:90 "Grid discovered"), one warp, four cells per
// word (the 60 padding bytes behind the 2500 cells are zero except the mirror counter word, which is skipped)
__device__ __forceinline__ void d2d_count_explored_warp(const DevP &P, const uint8_t *bel, int lane) {
    int cnt = 0;
#pragma unroll 1
    for (int w = lane; w < D2D_CELLS / 16; w += 32) {            // 156 x 16 bytes = cells 0 .. 2495
        const uint4 v = ((const uint4 *)bel)[w];
        cnt += __popc(__vcmpne4(v.x, 0u) & 0x01010101u) + __popc(__vcmpne4(v.y, 0u) & 0x01010101u) +
               __popc(__vcmpne4(v.z, 0u) & 0x01010101u) + __popc(__vcmpne4(v.w, 0u) & 0x01010101u);
    }
    if (lane == 0) cnt += __popc(__vcmpne4(((const uint32_t *)bel)[D2D_CELLS / 4 - 1], 0u) & 0x01010101u);   // cells 2496 .. 2499
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (lane == 0 && cnt) atomicAdd(&P.stats[D2D_STAT_GRID_DISCOVERED], (unsigned long long)cnt);
}

#ifdef D2D_WARP_PROF
__device__ __forceinline__ void d2d_prof_stamp(const DevP &P, int e, int k, int lane) {
    if (lane == 0) {
        unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); P.prof[(size_t)e * 12 + k] = t;
        if (k == 0) {
            unsigned sm, wi; asm volatile("mov.u32 %0, %%smid;" : "=r"(sm)); asm volatile("mov.u32 %0, %%warpid;" : "=r"(wi));
            P.prof[(size_t)e * 12 + 10] = sm; P.prof[(size_t)e * 12 + 11] = wi;
        }
    }
}
#define D2D_PROF(k) d2d_prof_stamp(P, e, k, lane)
#else
#define D2D_PROF(k)
#endif

// GATED: the instantiation d2d_step_pipelined launches.  The step's action arrives late (the warp waits for it just before
// the yaw update), and every store into the host mirror is held back until then: patched cells are recorded in a
// changed-cell list and replayed behind the gate, so the caller's observation buffers keep the previous step's content until
// it has published the next actions.  The plain instantiation (GATED = false) issues mirror stores as they occur (measured:
// deferring them costs ~15 % at 131072 envs and gains nothing at 4096) and carries none of the gate code.
template <int WPB, int MINB, bool ILP2, bool GATED>
__global__ void __launch_bounds__(WPB * 32, MINB) d2d_step_fused_warp_kernel(const DevP P,
                                                                             const double *__restrict__ actions) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int e = blockIdx.x * WPB + wid;
    if (e >= P.B) return;                                            // warp-uniform
    unsigned char *slice = smem + (size_t)wid * d2d_warp_slice_bytes(P.NP, P.HW, GATED ? D2D_FUSED_WARP_EXTRA : 0);
    const BlockCtx c = d2d_carve(slice, 1, P.NP, P.HW);
    // changed-cell list of this step (host mirror bound: the PCIe stores are replayed from it at the end of the step)
    uint32_t *chg = (uint32_t *)(slice + d2d_step_smem_bytes(1, P.NP, P.HW));
    int *nchg = (int *)(chg + D2D_CHG_CAP);
    EnvS &s = c.S[0];
    D2D_PROF(0);
    // Everything the step needs from HBM is requested up front so that the cold-miss latencies overlap instead of
    // chaining: observation cursor, first 32 agents (speculatively from the live arrays), the bulk copies of the belief
    // grid + ground-truth rows, then the env scalars.
    double2 pf_pos = double2{0.0, 0.0}, pf_pref = double2{0.0, 0.0};
    double pf_r = 0.0;
    uint8_t pf_act = 0;
    if (lane < P.N) {
        const size_t g = (size_t)e * P.NP + lane;
        pf_pos = P.apos[g]; pf_pref = P.apref[g]; pf_r = P.arad[g];
        if (P.trackers) pf_act = P.trk_active[g];
    }
    // same address in every lane: one broadcast request.  Pipelined host path: the action is not chosen yet (see the gate)
    double action = GATED ? 0.0 : actions[e];
    if (lane == 0) {
        if (GATED) *nchg = 0;
        d2d_mbar_init(c.mbar, 1);
        d2d_mbar_expect_tx(c.mbar, D2D_GT_ROW_BYTES + D2D_BELIEF_STRIDE);
        d2d_bulk_g2s(c.gt, P.gt_rows + (size_t)e * D2D_GRID, D2D_GT_ROW_BYTES, c.mbar);
        d2d_bulk_g2s(c.belief, P.belief + (size_t)e * D2D_BELIEF_STRIDE, D2D_BELIEF_STRIDE, c.mbar);
        c.misc[0] = 0;
    }
    d2d_load_env_warp(P, s, e, lane);
    if (lane == 0) c.misc[1] = s.reset;
#pragma unroll 1
    for (int w = lane; w < P.HW; w += 32) c.hitw[w] = 0u;
    __syncwarp();
    D2D_PROF(4);
    d2d_reset_prefetch(P, s, e, lane, pf_pos, pf_pref);
    d2d_reset_arrays(P, c, e, 1, lane, 32, c.mbar);
    d2d_phase_agents<true, true>(P, c, e, 1, lane, 32, pf_pos, pf_pref, pf_r);
    if (pf_act && !s.reset) d2d_prefetch_tracker(P, (size_t)e * P.NP + lane);
    D2D_PROF(5);
    if (lane == 0) d2d_leader_begin(P, s);
    // NoMove: the drone cell cannot change during the step, so if the observation tensor already holds this window it
    // is patched in place by the rays (only cells whose value changes) instead of being rewritten
    __syncwarp();
    const bool patch = !s.reset && s.obs_ix == s.ix && s.obs_iy == s.iy;
    const bool mirror = GATED && P.lm_mirror != nullptr;
    RayOut ro;
    ro.bel_s = c.belief; ro.e = e; ro.patch = patch ? 1 : 0;
    ro.wi = s.ix - 16; ro.wj = s.iy - 16;
    ro.chg = (mirror && patch) ? chg : nullptr; ro.nchg = nchg; ro.defer_mirror = GATED ? 1 : 0;
    D2D_PROF(6);
    d2d_mbar_wait(c.mbar, 0);
    ro.border_ok = d2d_border_intact(c.gt, lane);
    D2D_PROF(1);
    d2d_phase_rays_warp<ILP2>(P, c, ro, lane);
    __syncwarp();
    D2D_PROF(2);
    if (P.var_cam != 0.0) {
        if (lane == 0) d2d_measure_env(P, c, e);
        __syncwarp();
    }
    d2d_phase_trackers<true>(P, c, e, 1, lane, 32, pf_act);
    D2D_PROF(7);
    const int shit = __any_sync(0xffffffffu, lane < 5 ? d2d_static_probe(P, c.gt, s.px, s.py, lane) : 0);
    __syncwarp();
    D2D_PROF(8);
    if (GATED) {
        // Everything above is independent of this step's action (it only turns the yaw at the end of the step,
        // utils.py:741-743).  P.gate is the device staging buffer: it holds a sentinel until the host's copy engine has
        // delivered this step's actions (ONE async copy per step, no separate gate word: an aligned 8-byte word arrives
        // whole).  Each warp waits for its own word, takes it and puts the sentinel back for the next step.  Everything is in
        // DEVICE memory: a kernel polling pinned host memory is served one PCIe read at a time (measured ~17 ns per warp).
        if (lane == 0) {
            volatile unsigned long long *slot = P.gate + e;
            const long long t0 = clock64();
            unsigned long long bits;
            while ((bits = *slot) == D2D_ACTION_SENTINEL) {
                if (clock64() - t0 > 4000000000ll) { *P.gate_fault = 1u; bits = 0ull; break; }   // ~2 s: the host never came back
            }
            action = __longlong_as_double((long long)bits);
            *slot = D2D_ACTION_SENTINEL;
        }
        __syncwarp();
    }
    if (lane == 0) {
        // NoMove.plan traj_planner.py:70-73 / NoMove.replan_check :75-76; the verdict arrays (replan = 0, plan_ok = 1,
        // need_plan = 0) never change under NoMove: d2d_reset_kernel wrote them once
        s.tgx = -1.0; s.tgy = -1.0;
        d2d_leader_finish(P, s, c.gt, e, action, true);
        d2d_leader_flags(P, s, c.gt, e, shit);
        if (e == 0) atomicAdd(&P.stats[D2D_STAT_ENV_STEPS], (unsigned long long)P.B);   // every env steps once per launch
        if (!GATED && patch && P.lm_mirror) {
            const int nb = *(const int *)(c.belief + D2D_MIRCNT_OFF);
            if (nb) atomicAdd(&P.stats[D2D_STAT_MIRROR_BYTES], (unsigned long long)nb);
        }
    }
    __syncwarp();
    D2D_PROF(9);
    // NoMove never moves the drone, but a pose set from outside (d2d_set_drone_pose) invalidates the window; a step that
    // changed more cells than the list holds rewrites the window as well (the mirror must not miss a cell)
    const int n_changed = mirror ? *nchg : 0;
    const bool rewrite = !patch || s.ix != s.obs_ix || s.iy != s.obs_iy || (mirror && n_changed > D2D_CHG_CAP);
    __syncwarp();
    if (rewrite && lane == 0) { s.obs_ix = s.ix; s.obs_iy = s.iy; }
    __syncwarp();
    d2d_store_env_warp(P, s, e, lane);
    if (rewrite) d2d_obs_env_warp(P, c.belief, s.ix, s.iy, e, lane);
    else if (mirror && n_changed > 0) {
        // replay this step's changed cells into the host mirror (one byte each over PCIe)
        for (int q = lane; q < n_changed; q += 32) {
            const int cell = (int)(chg[q] & 0xFFFFu);
            const int ci = cell / D2D_GRID, cj = cell - ci * D2D_GRID;
            P.lm_mirror[(size_t)e * D2D_LOCAL_CELLS + (ci - ro.wi) * D2D_LOCAL + (cj - ro.wj)] = (uint8_t)(chg[q] >> 16);
        }
        if (lane == 0) atomicAdd(&P.stats[D2D_STAT_MIRROR_BYTES], (unsigned long long)n_changed);
    }
    if (s.done_now) d2d_count_explored_warp(P, c.belief, lane);
    D2D_PROF(3);
}

// ------------------------------------------------------------------------------------------ small-crowd rollout phases
// One env per warp and at most 32 agents: lane k owns agent k (global index g), no division, no loop.

// P1: Agent.step under CVM (d2d_rollout serves CVM handles only) from the state the lane holds in registers (live, or the
// snapshot of an env being reset), which is updated in place.  The culled list is built by ballot; returns whether an
// agent collides with the drone (Drone2D.is_collide utils.py:773-776).
__device__ __forceinline__ bool d2d_agents_lane(const DevP &P, const BlockCtx &c, EnvS &s, size_t g, int lane, double2 &pos,
                                                double2 &pref, double r) {
    bool in = false, hit = false;
    if (lane < P.N) {
        d2d_cvm_agent_step(pos.x, pos.y, pref.x, pref.y, r, P.dt, P.scale, P.map_w, P.map_h);
        P.apos[g] = pos;
        P.apref[g] = pref;
        c.sx[lane] = pos.x; c.sy[lane] = pos.y; c.sr2[lane] = r * r;
        const double ddx = pos.x - s.px, ddy = pos.y - s.py;
        const double reach = r + P.cull_reach;
        in = ddx * ddx + ddy * ddy <= reach * reach;
        hit = d2d_norm2_lt(ddx, ddy, r + P.drone_r);
    }
    const uint32_t b = __ballot_sync(0xffffffffu, in);
    if (in) c.cull[__popc(b & ((1u << lane) - 1u))] = (uint16_t)lane;
    if (lane == 0) s.ncull = __popc(b);
    return __any_sync(0xffffffffu, hit);
}

// P3: hit flag and Kalman tracker of agent `lane`; hmask is the env's hit mask over agents
__device__ __forceinline__ void d2d_trackers_lane(const DevP &P, const BlockCtx &c, EnvS &s, size_t g, int lane, uint32_t hmask,
                                                  uint8_t pf_act) {
    if (lane >= P.N) return;
    const bool hit = (hmask >> lane) & 1u;
    P.hit[g] = hit ? 1 : 0;
    if (P.trackers) {
        const bool was_active = !s.reset && pf_act != 0;
        if (hit && !was_active) atomicAdd(&s.newly, 1);   // utils.py:606-607
        if (was_active || hit || s.reset) {
            const bool noisy = P.var_cam != 0.0;
            d2d_tracker_update(P, s, g, hit, noisy ? c.mx[lane] : c.sx[lane], noisy ? c.my[lane] : c.sy[lane], was_active);
        }
    }
}

// P4 under NoMove, one thread: what d2d_leader_finish + d2d_leader_flags do, given the invariants of the drone's pose `inv`
// (bit 0: the static probes hit, bit 1: within reach of NoMove's fixed target (-1, -1)).  NoMove.plan always succeeds, so the
// brake never runs and fail is 0 when the flags are computed: the drone cannot dead-lock.  Only a trajectory written into
// the record from outside (nseg > 0) can move the drone; step_pos then pops its waypoints through the general code and the
// invariants are recomputed for the new pose (the static probes of this step were taken before the move, as in is_collide).
__device__ __forceinline__ void d2d_leader_nomove(const DevP &P, EnvS &s, const uint64_t *gt, int e, double action, bool coll,
                                                  int &inv) {
    const int shit = inv & 1;
    bool goal = (inv & 2) != 0;
    s.tgx = -1.0; s.tgy = -1.0;                                      // NoMove.plan traj_planner.py:70-73
    if (s.nseg * P.n_way - s.cursor > 0) {
        d2d_leader_finish(P, s, gt, e, 0.0, true, false);
        s.ix = d2d_cell(s.px, P.scale, P.inv_scale); s.iy = d2d_cell(s.py, P.scale, P.inv_scale);
        goal = d2d_norm2_le(s.px - s.tgx, s.py - s.tgy, 10.0);
        int sh = 0;
        for (int q = 0; q < 5; q++) sh |= d2d_static_probe(P, gt, s.px, s.py, q);
        inv = sh | (goal ? 2 : 0);
    } else {
        s.sm = SM_EXECUTING; s.fail = 0;
    }
    s.yaw = d2d_pymod(s.yaw + (action * P.max_yaw_speed) * P.dt, 360.0);   // step_yaw utils.py:741-743
    // is_collide utils.py:764-778: the static probes first, then the agents
    const int col = shit ? 1 : (coll ? 2 : 0);
    int frz = 0;
    if (col == 0) {   // drone_v2.py:222-225
        if (goal) s.sm = SM_GOAL_REACHED;
        frz = ((double)s.steps >= P.max_steps) ? 1 : 0;
    }
    const int done = (col != 0 || frz || (s.sm == SM_GOAL_REACHED && s.tcur >= P.n_targets)) ? 1 : 0;
    s.bufc += s.arch_cnt; s.bufts += s.arch_ts; s.tracked += s.newly;
    if (done) { s.bufc += s.act_cnt; s.bufts += s.act_ts; }
    s.done_now = done;
    P.collision[e] = (uint8_t)col; P.dead_lock[e] = 0; P.freezing[e] = (uint8_t)frz; P.done[e] = (uint8_t)done;
    P.yaw_obs[e] = (float)s.yaw;
    if (P.yaw_mirror) P.yaw_mirror[e] = (float)s.yaw;
    if (P.done_mirror) P.done_mirror[e] = (uint8_t)done;
    if (done) {
        atomicAdd(&P.stats[D2D_STAT_EPISODES], 1ull);
        if (s.sm == SM_GOAL_REACHED) atomicAdd(&P.stats[D2D_STAT_SUCCESS], 1ull);
        if (col == 1) atomicAdd(&P.stats[D2D_STAT_STATIC_COLLISION], 1ull);
        if (col == 2) atomicAdd(&P.stats[D2D_STAT_DYNAMIC_COLLISION], 1ull);
        if (frz) atomicAdd(&P.stats[D2D_STAT_FREEZING], 1ull);
        atomicAdd(&P.stats[D2D_STAT_FLIGHT_STEPS], (unsigned long long)s.steps);
        atomicAdd(&P.stats[D2D_STAT_AGENTS_TRACKED], (unsigned long long)s.bufc);
        atomicAdd(&P.stats[D2D_STAT_TRACKED_STEPS], (unsigned long long)s.bufts);
    }
}

// =============================================================================================================
// Multi-step ("rollout") variant of the fused warp kernel: consecutive Drone2DEnv2.step calls of an env in ONE launch.
// Step k+1 of an env depends on step k of the SAME env only, so a warp that owns an env can walk it through many steps
// without ever meeting the other warps: the env's working set (belief grid, ground-truth bitmap, agents, record) is
// fetched from HBM once and stays in shared memory / registers, and every store of a step goes out exactly as the
// single-step kernel issues it (belief cells, patched observation bytes, agents, trackers, verdict arrays).
//
// GATED = false (d2d_rollout): K steps, actions[t * action_stride + e] is the action of env e at step t (stride 0: the
//   same [B] vector every step).  Outputs are bit-identical to K single-step launches (tests/test_gpu_rollout.py); the
//   per-step verdict arrays / observation hold the LAST step's values, the statistics counters the sum over the steps.
// GATED = true (d2d_step_pipelined): a host policy drives the loop.  The kernel stays resident for a whole run of steps;
//   the action of every step arrives through the gate (P.gate: device staging slots holding a sentinel until the host's
//   copy engine has delivered the step's actions), together with a stamped word that says whether another step follows.
//   Everything of step t+1 that does not depend on its action (agents, rays, trackers, probes) runs while the host is
//   still looking at observation t; host-mirror stores are held back behind the gate and replayed; when the last warp
//   has finished step t (all its stores fenced system-wide) it writes t into a pinned host word the host polls.
//
// SYNC: the warps of a block start every step together (one block barrier per step).  Warps that run the same phase at
//   the same time share their instruction fetches; without it the 28 warps of an SM drift apart within a few dozen steps,
//   their combined footprint (the hot path of a step is ~30 KB of SASS) no longer fits the SM's 32 KB L1.5 instruction
//   cache and a third of the warp-state samples become `no_instruction` stalls (profiles/r2_ncu_rollout_cfg2_nosync.txt:
//   20.1 us per step without the barrier, 16.9 us with 28-warp blocks and one barrier per step).  The gate re-aligns the
//   warps by itself, so the GATED form needs no barrier.
//
// SMALL (d2d_rollout when N <= 32; GATED = false only): the small-crowd form.  A latency-bound warp's step is a chain of
//   mostly lane-serial code, so the form strips what N <= 32 and NoMove make constant:
//   - every warp slice is carved for exactly 32 agents and one hit word, so each shared-memory array sits at a fixed offset
//     from the slice base (an immediate) instead of being derived from the runtime N;
//   - lane k owns agent k in the agent and tracker phases; the culled list (at most 32 entries) is built by ballot, the
//     drone-vs-agent test is a warp vote, the march has no tail beyond 32 entries, and the env's hit mask comes out of the
//     ray phase as a warp reduction (stored into the hit word only for the noisy-measurement walk);
//   - under NoMove the drone's pose changes only when the env is reset (or when waypoints were written into the record from
//     outside), so the drone cell, the five static probes and the goal test against NoMove's fixed target are computed
//     once per pose and kept in registers: at kernel entry (after the bulk copy of the ground truth has landed), after
//     every in-kernel reset and after a popped waypoint.  They are never stored in the env record: clone / save / load,
//     d2d_set_drone_pose and in-place reseeding rewrite the record between launches, and every launch recomputes them
//     from whatever the record holds.
//   Results are bit-identical to the general form (tests/test_gpu_rollout.py, tests/test_gpu_rollout_small.py: N = 10, 32, 33).
// =============================================================================================================
#define D2D_GATE_STAMP_SLOT(B) ((size_t)(B))     // staging slot behind the B action slots: (session step << 1) | more
#define D2D_SMALL_N 32                           // agents the small-crowd rollout form carves every warp slice for

template <int WPB, int MINB, bool SYNC, bool GATED, bool SMALL = false>
__global__ void __launch_bounds__(WPB * 32, MINB) d2d_rollout_warp_kernel(const DevP P, const double *__restrict__ actions,
                                                                          int K, long long action_stride, int sync_every,
                                                                          unsigned int t_first) {
    static_assert(!(SMALL && GATED), "the small-crowd form serves d2d_rollout only");
    extern __shared__ __align__(128) unsigned char smem[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int e = blockIdx.x * WPB + wid;
    if (GATED) {                                                     // block arrival counter (see the end of the step)
        if (threadIdx.x == 0) *(int *)(smem + (size_t)WPB * d2d_warp_slice_bytes(P.NP, P.HW, D2D_FUSED_WARP_EXTRA)) = 0;
        __syncthreads();
    }
    if (GATED && P.gate_src && blockIdx.x == gridDim.x - 1) {
        // ---- courier block (owns no env).  Per step: thread 0 polls the stamp word in pinned host memory (one PCIe read in
        // flight at a time: ~1.5 us per poll); when the host has stamped the step, the block pulls the B actions out of the
        // caller's pinned buffer with coalesced reads, drops them over the sentinels in the device staging slots the env warps
        // are polling, and then publishes the stamp on the device.  The host's part of a step is ONE store.
        // (no static __shared__ here: the kernel's dynamic shared-memory limit is raised to the 227 KB maximum)
        unsigned long long &cst = *(unsigned long long *)(smem + (size_t)WPB * d2d_warp_slice_bytes(P.NP, P.HW, D2D_FUSED_WARP_EXTRA) + 128);
        const volatile unsigned long long *hs = (const volatile unsigned long long *)P.gate_stamp_host;
        for (unsigned int t = 0;; t++) {
            if (threadIdx.x == 0) {
                const unsigned long long want = (unsigned long long)(t_first + t);
                const long long t0 = clock64();
                unsigned long long st;
                while ((((st = *hs) >> 1) & 0xffffffffull) != want) {
                    if (clock64() - t0 > 4000000000ll) { *P.gate_fault = 1u; st = (want << 1) | (1ull << 62); break; }   // ~2 s
                }
                cst = st;
            }
            __syncthreads();
            const unsigned long long st = cst;
            const bool zero = (st >> 62) & 1ull;                     // abandoned run (or fault): finish the step with action 0
            // all PCIe reads of a thread in flight before its first store (a load -> store loop would pay one ~2 us round trip
            // per iteration)
#pragma unroll 1
            for (int i0 = threadIdx.x; i0 < P.B; i0 += 8 * (int)blockDim.x) {
                unsigned long long v[8];
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    const int i = i0 + k * (int)blockDim.x;
                    v[k] = (i < P.B && !zero) ? __ldcv(P.gate_src + i) : 0ull;
                }
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    const int i = i0 + k * (int)blockDim.x;
                    if (i < P.B) P.gate[i] = v[k];
                }
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                __threadfence();
                *(volatile unsigned long long *)(P.gate + D2D_GATE_STAMP_SLOT(P.B)) = st & 0x1ffffffffull;
            }
            if (!(st & 1ull)) return;
        }
    }
    if (e >= P.B) {                                                  // warp-uniform; a spare warp only keeps the barriers whole
        if (SYNC) for (int t = 1; t < K; t++) if (t % sync_every == 0) __syncthreads();
        return;
    }
    // slice layout: SMALL carves every slice for D2D_SMALL_N agents and one hit word (compile-time offsets)
    unsigned char *slice = smem + (size_t)wid * d2d_warp_slice_bytes(SMALL ? D2D_SMALL_N : P.NP, SMALL ? 1 : P.HW,
                                                                     GATED ? D2D_FUSED_WARP_EXTRA : 0);
    const BlockCtx c = d2d_carve(slice, 1, SMALL ? D2D_SMALL_N : P.NP, SMALL ? 1 : P.HW);
    // GATED: this step's changed cells
    uint32_t *chg = (uint32_t *)(slice + d2d_step_smem_bytes(1, SMALL ? D2D_SMALL_N : P.NP, SMALL ? 1 : P.HW));
    int *nchg = (int *)(chg + D2D_CHG_CAP);
    // GATED: block-level publication area behind the warp slices: arrival counter, this step's yaw / done of the block's envs
    unsigned char *blk = smem + (size_t)WPB * d2d_warp_slice_bytes(SMALL ? D2D_SMALL_N : P.NP, SMALL ? 1 : P.HW,
                                                                   GATED ? D2D_FUSED_WARP_EXTRA : 0);
    int *blk_cnt = (int *)blk;
    unsigned int *blk_yaw = (unsigned int *)(blk + 16);             // float bits; handed over with shared-memory atomics (below)
    unsigned int *blk_done = (unsigned int *)(blk + 16 + WPB * 4);
    const int blk_envs = min(WPB, P.B - (int)blockIdx.x * WPB);
    EnvS &s = c.S[0];
    const size_t ga = (size_t)e * P.NP + lane;
    double2 pf_pos = double2{0.0, 0.0}, pf_pref = double2{0.0, 0.0};
    double pf_r = 0.0;
    uint8_t pf_act = 0;
    if (lane < P.N) {
        pf_pos = P.apos[ga]; pf_pref = P.apref[ga]; pf_r = P.arad[ga];
        if (P.trackers) pf_act = P.trk_active[ga];
    }
    double action = GATED ? 0.0 : actions[e];
    if (lane == 0) {
        if (GATED) *nchg = 0;
        d2d_mbar_init(c.mbar, 1);
        d2d_mbar_expect_tx(c.mbar, D2D_GT_ROW_BYTES + D2D_BELIEF_STRIDE);
        d2d_bulk_g2s(c.gt, P.gt_rows + (size_t)e * D2D_GRID, D2D_GT_ROW_BYTES, c.mbar);
        d2d_bulk_g2s(c.belief, P.belief + (size_t)e * D2D_BELIEF_STRIDE, D2D_BELIEF_STRIDE, c.mbar);
        c.misc[0] = 0;
    }
    d2d_load_env_warp(P, s, e, lane);
    if (lane == 0) c.misc[1] = s.reset;
    if (!SMALL) {
#pragma unroll 1
        for (int w = lane; w < P.HW; w += 32) c.hitw[w] = 0u;
    }
    __syncwarp();
    int border_ok = 0;
    const bool mirror = GATED && P.lm_mirror != nullptr;
    int inv = 0;   // SMALL, lane 0: the drone-pose invariants of the current pose (bit 0: static probes, bit 1: goal test)
#pragma unroll 1
    for (int t = 0;;) {
        // here: the record is begun (d2d_env_begin), c.misc[1] = s.reset, the hit words are clear, pf_* hold the live agent
        // state of lane's agent (replaced by the snapshot just below when the env is being reset)
        D2D_PROF(0);
        d2d_reset_prefetch(P, s, e, lane, pf_pos, pf_pref);
        d2d_reset_arrays(P, c, e, 1, lane, 32, t == 0 ? c.mbar : nullptr);
        bool coll = false;
        if (SMALL) coll = d2d_agents_lane(P, c, s, ga, lane, pf_pos, pf_pref, pf_r);
        else d2d_phase_agents<true, true>(P, c, e, 1, lane, 32, pf_pos, pf_pref, pf_r, &pf_pos, &pf_pref);
        if (t == 0 && pf_act && !s.reset) d2d_prefetch_tracker(P, ga);
        if (lane == 0) d2d_leader_begin(P, s);
        __syncwarp();
        if (SMALL) {
            if (t == 0) {
                d2d_mbar_wait(c.mbar, 0);
                border_ok = d2d_border_intact(c.gt, lane);           // the ground truth never changes
            }
            if (t == 0 || s.reset) {                                 // warp-uniform: a pose from the record or the reset pose
                const double px = s.px, py = s.py;
                const int sh = __any_sync(0xffffffffu, lane < 5 ? d2d_static_probe(P, c.gt, px, py, lane) : 0);
                if (lane == 0) {
                    inv = sh | (d2d_norm2_le(px - -1.0, py - -1.0, 10.0) ? 2 : 0);   // NoMove's target is (-1, -1)
                    s.ix = d2d_cell(px, P.scale, P.inv_scale); s.iy = d2d_cell(py, P.scale, P.inv_scale);
                }
                __syncwarp();
            }
        }
        // same window as the observation tensor holds: patched in place by the rays; an env that starts a new episode there
        // has its slice cleared first (d2d_obs_clear_warp) -- GATED: on the device only, the host mirror gets the finished slice
        // behind the gate
        // (not with a host mirror that takes its stores as they occur: ~150 single-byte PCIe writes per fresh env cost more
        // than the one coalesced rewrite)
        const bool refill = s.reset && s.obs_ix == s.ix && s.obs_iy == s.iy && (GATED || P.lm_mirror == nullptr);
        const bool patch = (!s.reset || refill) && s.obs_ix == s.ix && s.obs_iy == s.iy;
        if (refill) d2d_obs_clear_warp(P, e, lane, false);
        RayOut ro;
        ro.bel_s = c.belief; ro.e = e; ro.patch = patch ? 1 : 0;
        ro.wi = s.ix - 16; ro.wj = s.iy - 16;
        ro.chg = (mirror && patch && !refill) ? chg : nullptr; ro.nchg = nchg; ro.defer_mirror = GATED ? 1 : 0;
        if (!SMALL && t == 0) {
            d2d_mbar_wait(c.mbar, 0);
            border_ok = d2d_border_intact(c.gt, lane);               // the ground truth never changes
        }
        ro.border_ok = border_ok;
        D2D_PROF(1);
        const uint32_t hmask = d2d_phase_rays_warp<false, SMALL>(P, c, ro, lane);
        __syncwarp();
        D2D_PROF(2);
        if (P.var_cam != 0.0) {
            if (lane == 0) {
                if (SMALL) c.hitw[0] = hmask;
                d2d_measure_env(P, c, e);
            }
            __syncwarp();
        }
        if (SMALL) d2d_trackers_lane(P, c, s, ga, lane, hmask, pf_act);
        else d2d_phase_trackers<true>(P, c, e, 1, lane, 32, pf_act);
        const int shit = SMALL ? 0 : __any_sync(0xffffffffu, lane < 5 ? d2d_static_probe(P, c.gt, s.px, s.py, lane) : 0);
        __syncwarp();
        int more = (t + 1 < K) ? 1 : 0;
        bool rewrite = false;
        int n_changed = 0;
        if (GATED) {
            // Everything of the step except the yaw update is independent of the action (utils.py:741-743 is the only place it
            // is used): planner verdict, step_pos, collision / done flags, statistics and the device-side observation all run
            // BEFORE the gate, while the host is still choosing the action.
            if (lane == 0) {
                s.tgx = -1.0; s.tgy = -1.0;                          // NoMove.plan traj_planner.py:70-73
                d2d_leader_finish(P, s, c.gt, e, 0.0, true, false);
                d2d_leader_flags(P, s, c.gt, e, shit, false);
            }
            __syncwarp();
            n_changed = (mirror && !refill) ? *nchg : 0;
            rewrite = !patch || s.ix != s.obs_ix || s.iy != s.obs_iy || (mirror && n_changed > D2D_CHG_CAP);
            __syncwarp();
            if (rewrite && lane == 0) { s.obs_ix = s.ix; s.obs_iy = s.iy; }
            __syncwarp();
            if (rewrite) d2d_obs_env_warp(P, c.belief, s.ix, s.iy, e, lane, false);      // device tensor only
            if (s.done_now) d2d_count_explored_warp(P, c.belief, lane);
            D2D_PROF(8);
            // Wait for this env's slot to lose the sentinel, take the action, put the sentinel back; then read the stamped word
            // that travels with the actions: (session step << 1) | (another step follows).
            if (lane == 0) {
                volatile unsigned long long *slot = P.gate + e;
                volatile unsigned long long *stamp = P.gate + D2D_GATE_STAMP_SLOT(P.B);
                const unsigned long long want = (unsigned long long)(t_first + (unsigned int)t);
                const long long t0 = clock64();
                unsigned long long bits, st = 0ull;
                bool fault = false;
                while ((bits = *slot) == D2D_ACTION_SENTINEL) {
                    if (clock64() - t0 > 4000000000ll) { fault = true; break; }      // ~2 s: the host never came back
                }
                if (!fault) {
                    while (((st = *stamp) >> 1) != want) {
                        if (clock64() - t0 > 4000000000ll) { fault = true; break; }
                    }
                }
                if (fault) { *P.gate_fault = 1u; bits = 0ull; st = 0ull; }            // finish the step with action 0 and leave
                action = __longlong_as_double((long long)bits);
                *slot = D2D_ACTION_SENTINEL;
                more = (int)(st & 1ull);
                s.yaw = d2d_pymod(s.yaw + (action * P.max_yaw_speed) * P.dt, 360.0);   // step_yaw utils.py:741-743
                P.yaw_obs[e] = (float)s.yaw;
            }
            more = __shfl_sync(0xffffffffu, more, 0);
            D2D_PROF(9);
            // behind the gate: this step's observation bytes go out to the host mirror
            if (mirror) {
                if (rewrite || refill) {
                    __syncwarp();
                    d2d_obs_mirror_copy_warp(P, e, lane);
                } else if (n_changed > 0) {
                    for (int q = lane; q < n_changed; q += 32) {      // one byte each over PCIe
                        const int cell = (int)(chg[q] & 0xFFFFu);
                        const int ci = cell / D2D_GRID, cj = cell - ci * D2D_GRID;
                        P.lm_mirror[(size_t)e * D2D_LOCAL_CELLS + (ci - ro.wi) * D2D_LOCAL + (cj - ro.wj)] = (uint8_t)(chg[q] >> 16);
                    }
                    if (lane == 0) atomicAdd(&P.stats[D2D_STAT_MIRROR_BYTES], (unsigned long long)n_changed);
                }
            }
            __syncwarp();
        } else {
            if (lane == 0) {
                if (SMALL) d2d_leader_nomove(P, s, c.gt, e, action, coll, inv);
                else {
                    s.tgx = -1.0; s.tgy = -1.0;                      // NoMove.plan traj_planner.py:70-73
                    d2d_leader_finish(P, s, c.gt, e, action, true);
                    d2d_leader_flags(P, s, c.gt, e, shit);
                }
                if (patch && P.lm_mirror) {
                    int *cnt = (int *)(c.belief + D2D_MIRCNT_OFF);
                    const int nb = *cnt;
                    if (nb) { atomicAdd(&P.stats[D2D_STAT_MIRROR_BYTES], (unsigned long long)nb); *cnt = 0; }
                }
            }
            __syncwarp();
            rewrite = !patch || s.ix != s.obs_ix || s.iy != s.obs_iy;
            __syncwarp();
            if (rewrite && lane == 0) { s.obs_ix = s.ix; s.obs_iy = s.iy; }
            __syncwarp();
            if (rewrite) d2d_obs_env_warp(P, c.belief, s.ix, s.iy, e, lane);
            if (s.done_now) d2d_count_explored_warp(P, c.belief, lane);
        }
        D2D_PROF(4);
        if (GATED) {
            // Step complete for this env.  The block's LAST warp to get here publishes the block: yaw / done of its envs as two
            // coalesced stores into the host mirror, a device-scope fence and one global arrival count; the last block of the
            // step issues the step's ONE system-scope fence and writes the step's sequence number into the pinned word the
            // host polls.  Every warp's own mirror stores are ordered before that flag through the chain block fence + block
            // counter -> device fence + global counter -> system fence (fences are cumulative).  Measured: a system fence
            // per warp (4096 per step, each waiting for its PCIe writes) 15 us, one per block 10 us, one per step ~1 us.
            int last = 0;
            if (lane == 0) {
                // (atomic accesses on both sides of the hand-over: plain ones are ordered just as well by the fences, but
                // compute-sanitizer's racecheck only models barriers and reports a fence + counter hand-over as a hazard)
                atomicExch(&blk_yaw[wid], __float_as_uint((float)s.yaw)); atomicExch(&blk_done[wid], (unsigned int)s.done_now);
                __threadfence_block();
                last = atomicAdd(blk_cnt, 1) == blk_envs - 1 ? 1 : 0;
            }
            last = __shfl_sync(0xffffffffu, last, 0);
            if (last) {
                __threadfence_block();
                const int e0 = (int)blockIdx.x * WPB;
                if (lane < blk_envs) {
                    if (P.yaw_mirror) P.yaw_mirror[e0 + lane] = __uint_as_float(atomicOr(&blk_yaw[lane], 0u));
                    if (P.done_mirror) P.done_mirror[e0 + lane] = (uint8_t)atomicOr(&blk_done[lane], 0u);
                }
                __syncwarp();
                if (lane == 0) {
                    *blk_cnt = 0;
                    __threadfence();                      // device scope: cheap; the step's ONE system fence is below
                    const unsigned long long n = atomicAdd(P.gate_count, (unsigned long long)blk_envs) + (unsigned long long)blk_envs;
                    if (n == (unsigned long long)P.B * (unsigned long long)(t + 1)) {
                        atomicAdd(&P.stats[D2D_STAT_ENV_STEPS], (unsigned long long)P.B);   // every env stepped once
                        // release at system scope (cumulative: orders every block's mirror stores before the flag); acq_rel is
                        // all a release needs -- __threadfence_system() is the sequentially-consistent fence
                        asm volatile("fence.acq_rel.sys;" ::: "memory");
                        *(volatile unsigned int *)P.gate_done = t_first + (unsigned int)t;
                    }
                }
            }
        }
        D2D_PROF(3);
        t += 1;
        if (!more) break;
        if (SYNC && t % sync_every == 0) __syncthreads();
        // ---- next step of the same env: what d2d_load_env_warp does at kernel entry, from the live record
        if (!GATED) action = actions[(size_t)t * (size_t)action_stride + e];
        if (P.trackers && lane < P.N) pf_act = P.trk_active[ga];     // written by this very lane in the tracker phase
        if (!SMALL) {
#pragma unroll 1
            for (int w = lane; w < P.HW; w += 32) c.hitw[w] = 0u;
        }
        __syncwarp();
        if (lane == 0) {
            const bool was_done = s.done_now != 0;
            d2d_env_begin<!SMALL>(P, s, was_done);
            c.misc[1] = s.reset;
            if (GATED) *nchg = 0;
        }
        __syncwarp();
    }
    d2d_store_env_warp(P, s, e, lane);
    if (!GATED && e == 0 && lane == 0) atomicAdd(&P.stats[D2D_STAT_ENV_STEPS], (unsigned long long)P.B * (unsigned long long)K);
}
