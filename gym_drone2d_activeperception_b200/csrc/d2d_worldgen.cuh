// d2d_worldgen.cuh -- the world of a seed, generated on the device (d2d_generate_worlds): world.generate_world restated for
// one env per warp.  The reference (drone_v2.py:12-66, utils.py:508-525) seeds two streams with map_id:
//   Python `random.Random(seed)`         MT19937 init_by_array([seed]): pillars, then the random agents' positions / radii
//   `np.random.RandomState(seed)`        MT19937 init_genrand(seed): rand(100) group headings, then the measurement noise
// Every decision is taken with the reference's arithmetic in the D2D_HD helpers below; the host-compiled twin
// (wg_generate_host, tests/helpers/worldgen_twin.cpp) runs the same helpers sequentially.  Build with FMA contraction off.
//
// One deliberate deviation: the static-map group velocities use the correctly rounded d2d_sincos where the reference calls
// glibc's np.cos / np.sin (1 ulp apart in ~0.1 % of the directions).  The grid erasure test `(cx-ax)**2 + (cy-ay)**2 <= r**2`
// squares with x*x where Python calls libm pow; the two verdicts can only differ within a few ulp of a disc edge.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>
#include "../../include/drone2d.h"
#include "d2d_math.cuh"

#define D2D_MT_N 624
#define D2D_MT_M 397
#define D2D_WORLD_MAX_REJECTS 65536      // consecutive rejected draws of one pillar / agent before the seed is given up
#define D2D_WG_WARPS 4                   // warps (envs) per block of d2d_worldgen_kernel
#define D2D_WG_GRID 50                   // cells per side (D2D_GRID; this header does not need d2d_state.cuh)
#define D2D_WG_MAX_OBS 16                // RVO obstacle rows per env (D2D_RVO_MAX_OBS)

// Seed-independent tables derived from one d2d_world_source and the config (wg_build_tables); the device holds one per
// source of the handle's table (d2d_set_world_sources), indexed by the key's high word.
struct WgTables {
    d2d_world_source src;
    uint32_t mt_base[D2D_MT_N];          // init_genrand(19650218): the start of every init_by_array
    double targets[D2D_MAX_TARGETS][2];
    double scale;                        // params.map_scale
    int n_targets, N, n_map, rvo, noisy, need_np;
    uint16_t map_cell[2500];             // x * 50 + y of the static-map agents, np.nonzero (row-major) order
    uint8_t map_group[2500];
};

// ------------------------------------------------------------------------------------------------ MT19937
D2D_HD void wg_init_genrand(uint32_t *mt, uint32_t s) {
    mt[0] = s;
    for (int i = 1; i < D2D_MT_N; i++) mt[i] = 1812433253u * (mt[i - 1] ^ (mt[i - 1] >> 30)) + (uint32_t)i;
}

// init_by_array(key = [seed], key_length = 1) (CPython _randommodule.c), starting from mt_base = init_genrand(19650218)
D2D_HD void wg_init_by_array1(uint32_t *mt, const uint32_t *mt_base, uint32_t seed) {
    for (int i = 0; i < D2D_MT_N; i++) mt[i] = mt_base[i];
    int i = 1;
    for (int k = D2D_MT_N; k; k--) {
        mt[i] = (mt[i] ^ ((mt[i - 1] ^ (mt[i - 1] >> 30)) * 1664525u)) + seed;   // + init_key[0] + j, j == 0
        i++;
        if (i >= D2D_MT_N) { mt[0] = mt[D2D_MT_N - 1]; i = 1; }
    }
    for (int k = D2D_MT_N - 1; k; k--) {
        mt[i] = (mt[i] ^ ((mt[i - 1] ^ (mt[i - 1] >> 30)) * 1566083941u)) - (uint32_t)i;
        i++;
        if (i >= D2D_MT_N) { mt[0] = mt[D2D_MT_N - 1]; i = 1; }
    }
    mt[0] = 0x80000000u;
}

// new value of mt[i] in the in-place twist (genrand_uint32 when index >= N); entries < i already hold their new values
D2D_HD uint32_t wg_twist_at(const uint32_t *mt, int i) {
    const uint32_t y = (mt[i] & 0x80000000u) | (mt[i + 1 < D2D_MT_N ? i + 1 : 0] & 0x7fffffffu);
    const int m = i + D2D_MT_M < D2D_MT_N ? i + D2D_MT_M : i + D2D_MT_M - D2D_MT_N;
    return mt[m] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
}

D2D_HD uint32_t wg_temper(uint32_t y) {
    y ^= (y >> 11);
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= (y >> 18);
    return y;
}

// random() / np.random.rand(): ((a >> 5) * 67108864.0 + (b >> 6)) / 2**53 from two consecutive outputs
D2D_HD double wg_random53(uint32_t a, uint32_t b) {
    return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) * (1.0 / 9007199254740992.0);
}

// random.uniform(lo, hi) = lo + (hi - lo) * random()
D2D_HD double wg_uniform(double lo, double hi, double u) { return lo + (hi - lo) * u; }

D2D_HD int wg_bit_length(uint32_t n) {
    int k = 0;
    while (n) { k++; n >>= 1; }
    return k;
}

// ------------------------------------------------------------------------------------------------ placement decisions
// A pillar (x, y, rad) may stay unless it is within drone_radius + 20 + rad of a target or drone_radius + 70 of the drone
// (drone_v2.py:16-24); np.linalg.norm is d2d_norm2
D2D_HD bool wg_pillar_free(const WgTables &T, int ox, int oy, int orad) {
    const d2d_world_source &s = T.src;
    for (int t = 0; t < T.n_targets; t++)
        if (d2d_norm2(T.targets[t][0] - (double)ox, T.targets[t][1] - (double)oy) <= s.drone_radius + 20.0 + (double)orad)
            return false;
    return !(d2d_norm2(s.init_x - (double)ox, s.init_y - (double)oy) <= s.drone_radius + 70.0);
}

// agent candidate (px, py, r) against an accepted agent (qx, qy, qr): norm(q - p) <= qr + r rejects (drone_v2.py:36-38)
D2D_HD bool wg_hits_agent(double px, double py, double r, double qx, double qy, double qr) {
    return d2d_norm2(qx - px, qy - py) <= qr + r;
}

// ... against a pillar: norm([ox, oy] - p) <= orad + r + 10 (drone_v2.py:39-41; the int64 radius plus a float, then + 10)
D2D_HD bool wg_hits_pillar(double px, double py, double r, int ox, int oy, int orad) {
    return d2d_norm2((double)ox - px, (double)oy - py) <= ((double)orad + r) + 10.0;
}

// ... against the drone: norm(p - drone) <= drone_radius + 70 (drone_v2.py:42-43)
D2D_HD bool wg_hits_drone(const WgTables &T, double px, double py) {
    return d2d_norm2(px - T.src.init_x, py - T.src.init_y) <= T.src.drone_radius + 70.0;
}

// the cell range [lo, hi) of a pillar along one axis: max(0, int((c - rad) // scale) - 1) .. min(50, int((c + rad) // scale) + 2)
D2D_HD void wg_pillar_range(const WgTables &T, int c, int rad, int &lo, int &hi) {
    const double inv = 1.0 / T.scale;
    lo = d2d_cell((double)(c - rad), T.scale, inv) - 1;
    hi = d2d_cell((double)(c + rad), T.scale, inv) + 2;
    if (lo < 0) lo = 0;
    if (hi > D2D_WG_GRID) hi = D2D_WG_GRID;
}

// cell (i, j) of a pillar disc: norm([scale (i + .5), scale (j + .5)] - [x, y]) <= rad (utils.py:516-519)
D2D_HD bool wg_pillar_cell(const WgTables &T, int i, int j, int ox, int oy, int orad) {
    return d2d_norm2(T.scale * ((double)i + 0.5) - (double)ox, T.scale * ((double)j + 0.5) - (double)oy) <= (double)orad;
}

// a cell centre inside an agent disc is no longer occupancy (utils.py:521-525): (cx-ax)**2 + (cy-ay)**2 <= r**2 with x*x
D2D_HD bool wg_cell_covered(const WgTables &T, int i, int j, double ax, double ay, double r) {
    const double dx = T.scale * ((double)i + 0.5) - ax, dy = T.scale * ((double)j + 0.5) - ay;
    return dx * dx + dy * dy <= r * r;
}

// cells whose centre can lie in the disc (ax, ay, r): a screen one unit wider than the disc, decided by wg_cell_covered
D2D_HD void wg_cover_range(const WgTables &T, double a, double r, int &lo, int &hi) {
    lo = (int)floor((a - r - 1.0) / T.scale - 0.5);
    hi = (int)ceil((a + r + 1.0) / T.scale - 0.5) + 1;
    if (lo < 0) lo = 0;
    if (hi > D2D_WG_GRID) hi = D2D_WG_GRID;
}

// group heading g: np.random.rand(100)[g] * 2 * np.pi, and its velocity agent_max_speed * [cos, sin] (drone_v2.py:53-62)
D2D_HD void wg_group_velocity(double speed, uint32_t a, uint32_t b, double &vx, double &vy) {
    const double dir = wg_random53(a, b) * 2.0 * D2D_PI;
    double sn, cs;
    d2d_sincos(dir, &sn, &cs);
    vx = speed * cs;
    vy = speed * sn;
}

// ------------------------------------------------------------------------------------------------ tables (host)
// Fails (returns a message) on a source that the config cannot take.  scale: the config's map_scale.
static inline const char *wg_build_tables(WgTables *T, const d2d_world_source *s, const double (*targets)[2], int n_targets,
                                          double scale, int num_agents, int rvo, int noisy) {
    if (s->struct_size != (int32_t)sizeof(d2d_world_source)) return "d2d_world_source size mismatch (ABI)";
    if (s->agent_number < 0 || s->agent_number > D2D_WORLD_MAX_RANDOM) return "agent_number out of range (at most 256)";
    if (s->pillar_number < 0 || s->pillar_number > D2D_WORLD_MAX_PILLARS) return "pillar_number out of range (at most 64)";
    if (rvo && s->pillar_number > 16) return "the RVO motion profile takes at most 16 pillars";
    if (s->map_w != floor(s->map_w) || s->map_h != floor(s->map_h) || s->map_w < 100 || s->map_h < 100 || s->map_w > 1e6 ||
        s->map_h > 1e6)
        return "map size must be integral and at least 100 (randint(50, W - 50))";
    if (!(scale > 0) || (int)(s->map_w / scale) != 50 || (int)(s->map_h / scale) != 50) return "the map must have 50x50 cells";
    if (!(s->agent_radius == -1.0 || s->agent_radius >= 0) || !(s->drone_radius >= 0) || !(fabs(s->agent_max_speed) < 1e6) ||
        !(fabs(s->init_x) < 1e6) || !(fabs(s->init_y) < 1e6))
        return "radius, speed or init position out of range";
    memset(T, 0, sizeof(*T));
    T->src = *s;
    wg_init_genrand(T->mt_base, 19650218u);
    for (int t = 0; t < n_targets; t++) { T->targets[t][0] = targets[t][0]; T->targets[t][1] = targets[t][1]; }
    T->n_targets = n_targets;
    T->scale = scale;
    int n = 0;
    for (int x = 0; x < 50; x++)
        for (int y = 0; y < 50; y++) {
            const int g = s->static_map[x][y];
            if (!g) continue;
            if (g >= D2D_WORLD_GROUPS) return "static map group ids must lie in [0, 100)";
            T->map_cell[n] = (uint16_t)(x * 50 + y);
            T->map_group[n] = (uint8_t)g;
            n++;
        }
    if (s->agent_number + n != num_agents) return "agent_number + the static map's agents must equal the config's num_agents";
    T->n_map = n;
    T->N = num_agents;
    T->rvo = rvo;
    T->noisy = noisy;
    T->need_np = (n > 0 || noisy) ? 1 : 0;
    return nullptr;
}

#if !defined(__CUDACC__)
// ------------------------------------------------------------------------------------------------ host twin
// The same world as d2d_worldgen_kernel, sequentially.  Outputs as d2d_set_world / d2d_set_rng / d2d_set_rvo take them (one
// env): apos, apref [N][2], arad, trad [N], gt_rows [50], pose [3]; rng_key [624] (+ pos 200, no gaussian) when T.noisy;
// avel [N][2], obs [16][3], *nobs when T.rvo.  Returns 0, or -1 when a placement exceeded D2D_WORLD_MAX_REJECTS.
static int wg_generate_host(const WgTables &T, uint32_t seed, double *apos, double *apref, double *arad, double *trad,
                            uint64_t *gt_rows, double *pose, uint32_t *rng_key, double *avel, double *obs, int *nobs) {
    const d2d_world_source &s = T.src;
    static thread_local uint32_t mt[D2D_MT_N];
    int pos = D2D_MT_N;
    auto next = [&]() -> uint32_t {
        if (pos >= D2D_MT_N) { for (int i = 0; i < D2D_MT_N; i++) mt[i] = wg_twist_at(mt, i); pos = 0; }
        return wg_temper(mt[pos++]);
    };
    auto randint = [&](int a, int b) -> int {
        const uint32_t n = (uint32_t)(b - a + 1);
        const int k = wg_bit_length(n);
        uint32_t r;
        do { r = next() >> (32 - k); } while (r >= n);
        return a + (int)r;
    };
    auto random = [&]() -> double { const uint32_t a = next(); return wg_random53(a, next()); };
    wg_init_by_array1(mt, T.mt_base, seed);
    const int W = (int)s.map_w, H = (int)s.map_h;
    int pil[D2D_WORLD_MAX_PILLARS][3];
    for (int np_ = 0, rej = 0; np_ < s.pillar_number;) {
        const int x = randint(50, W - 50), y = randint(50, H - 50), r = randint(15, 20);
        if (wg_pillar_free(T, x, y, r)) { pil[np_][0] = x; pil[np_][1] = y; pil[np_][2] = r; np_++; rej = 0; }
        else if (++rej > D2D_WORLD_MAX_REJECTS) return -1;
    }
    const double rlo = s.agent_radius == -1.0 ? 5.0 : s.agent_radius - 2.0, rhi = s.agent_radius == -1.0 ? 15.0 : s.agent_radius + 2.0;
    for (int k = 0, rej = 0; k < s.agent_number;) {
        const double px = wg_uniform(20.0, (double)(W - 20), random());
        const double py = wg_uniform(20.0, (double)(H - 20), random());
        const double r = wg_uniform(rlo, rhi, random());
        bool free = !wg_hits_drone(T, px, py);
        for (int j = 0; free && j < k; j++) free = !wg_hits_agent(px, py, r, apos[2 * j], apos[2 * j + 1], arad[j]);
        for (int q = 0; free && q < s.pillar_number; q++) free = !wg_hits_pillar(px, py, r, pil[q][0], pil[q][1], pil[q][2]);
        if (free) {
            apos[2 * k] = px; apos[2 * k + 1] = py;
            apref[2 * k] = s.headings[k][0]; apref[2 * k + 1] = s.headings[k][1];
            arad[k] = r; trad[k] = r;
            k++; rej = 0;
        } else if (++rej > D2D_WORLD_MAX_REJECTS) return -1;
    }
    if (T.need_np) {
        wg_init_genrand(mt, seed);
        for (int i = 0; i < D2D_MT_N; i++) mt[i] = wg_twist_at(mt, i);
        for (int m = 0; m < T.n_map; m++) {
            const int k = s.agent_number + m, g = T.map_group[m], c = T.map_cell[m];
            wg_group_velocity(s.agent_max_speed, wg_temper(mt[2 * g]), wg_temper(mt[2 * g + 1]), apref[2 * k], apref[2 * k + 1]);
            apos[2 * k] = (double)(5 + (c / 50) * 10); apos[2 * k + 1] = (double)(5 + (c % 50) * 10);
            arad[k] = 5.0; trad[k] = s.agent_radius;
        }
        if (T.noisy) for (int i = 0; i < D2D_MT_N; i++) rng_key[i] = mt[i];
    }
    for (int i = 0; i < D2D_WG_GRID; i++) {
        uint64_t row = (i == 0 || i == D2D_WG_GRID - 1) ? ((1ull << D2D_WG_GRID) - 1) : (1ull | (1ull << 49));
        for (int q = 0; q < s.pillar_number; q++) {
            int i0, i1, j0, j1;
            wg_pillar_range(T, pil[q][0], pil[q][2], i0, i1);
            wg_pillar_range(T, pil[q][1], pil[q][2], j0, j1);
            if (i < i0 || i >= i1) continue;
            for (int j = j0; j < j1; j++)
                if (wg_pillar_cell(T, i, j, pil[q][0], pil[q][1], pil[q][2])) row |= 1ull << j;
        }
        gt_rows[i] = row;
    }
    for (int k = 0; k < T.N; k++) {
        int i0, i1, j0, j1;
        wg_cover_range(T, apos[2 * k], arad[k], i0, i1);
        wg_cover_range(T, apos[2 * k + 1], arad[k], j0, j1);
        for (int i = i0; i < i1; i++)
            for (int j = j0; j < j1; j++)
                if (wg_cell_covered(T, i, j, apos[2 * k], apos[2 * k + 1], arad[k])) gt_rows[i] &= ~(1ull << j);
    }
    pose[0] = s.init_x; pose[1] = s.init_y; pose[2] = 270.0;           // yaw = -90 % 360 (utils.py:718)
    if (T.rvo) {
        for (int k = 0; k < T.N; k++) {
            avel[2 * k] = k < s.agent_number ? 0.0 : apref[2 * k];
            avel[2 * k + 1] = k < s.agent_number ? 0.0 : apref[2 * k + 1];
        }
        for (int q = 0; q < D2D_WG_MAX_OBS; q++)
            for (int c = 0; c < 3; c++) obs[3 * q + c] = q < s.pillar_number ? (double)pil[q][c] : 0.0;
        *nobs = s.pillar_number;
    }
    return 0;
}
#endif

#if defined(__CUDACC__)
// ------------------------------------------------------------------------------------------------ device
static_assert(D2D_WG_GRID == D2D_GRID && D2D_WG_MAX_OBS == D2D_RVO_MAX_OBS, "d2d_worldgen.cuh and d2d_state.cuh disagree");
struct WgWarp {                          // per-warp shared memory
    uint32_t mt[D2D_MT_N];               // the Python stream, then the NumPy stream
    int pil[D2D_WORLD_MAX_PILLARS][3];
    double vel[D2D_WORLD_GROUPS][2];
    unsigned long long occ[D2D_WG_GRID], erase[D2D_WG_GRID];
};

// the in-place twist by the whole warp: 32 entries at a time, every lane reads before any lane writes.  Entry i reads
// mt[i], mt[i + 1] (not yet rewritten) and mt[(i + 397) % 624] (rewritten by an earlier group exactly when i >= 227), so the
// order of the sequential twist is kept.
__device__ __forceinline__ void wg_twist_warp(uint32_t *mt, int lane) {
    for (int i0 = 0; i0 < D2D_MT_N; i0 += 32) {
        const int i = i0 + lane;
        const uint32_t v = i < D2D_MT_N ? wg_twist_at(mt, i) : 0u;
        __syncwarp();
        if (i < D2D_MT_N) mt[i] = v;
        __syncwarp();
    }
}

// the next output of the Python stream; warp-uniform (every lane holds the same pos and gets the same value)
__device__ __forceinline__ uint32_t wg_next(uint32_t *mt, int &pos, int lane) {
    if (pos >= D2D_MT_N) { wg_twist_warp(mt, lane); pos = 0; }
    return wg_temper(mt[pos++]);
}

__device__ __forceinline__ int wg_randint(uint32_t *mt, int &pos, int lane, int a, int b) {
    const uint32_t n = (uint32_t)(b - a + 1);
    const int k = wg_bit_length(n);
    uint32_t r;
    do { r = wg_next(mt, pos, lane) >> (32 - k); } while (r >= n);
    return a + (int)r;
}

__device__ __forceinline__ double wg_random(uint32_t *mt, int &pos, int lane) {
    const uint32_t a = wg_next(mt, pos, lane);
    return wg_random53(a, wg_next(mt, pos, lane));
}

// A world given up: the first warp to claim the (device) claim word stores the env into fault[1] and then (1 << 63 | key)
// into fault[0] (mapped host words), so the host never pairs one world's key with another's env.  The host clears the words
// and the claim when it reports the failure.
__device__ __noinline__ void wg_report_fault(volatile unsigned long long *fault, unsigned int *claim, int env, long long key) {
    if (atomicCAS(claim, 0u, 1u) != 0u) return;
    fault[1] = (unsigned long long)env;
    __threadfence_system();
    fault[0] = (1ull << 63) | (unsigned long long)key;
}

// Blocks per SM the generation kernels are compiled for (__launch_bounds__): 8 for d2d_worldgen_kernel and 7 for
// d2d_worldgen_list_kernel cap them at 64 and 72 registers, the figures of the single-table kernels, so reading the table
// through the key costs no occupancy (the 22.7 KB of shared memory per block would allow 9).
#define D2D_WG_MIN_BLOCKS 8
#define D2D_WG_LIST_MIN_BLOCKS 7

// One warp per generated world: envs[w] gets the world of keys[w] (source << 32 | seed), built from the tables Tg[source].
// lazy: also mark the env pending_reset.  A placement that exceeds D2D_WORLD_MAX_REJECTS is reported (wg_report_fault) and
// the env abandoned.  The body is shared with d2d_worldgen_list_kernel through d2d_worldgen_body.inc.
__global__ void __launch_bounds__(D2D_WG_WARPS * 32, D2D_WG_MIN_BLOCKS) d2d_worldgen_kernel(const DevP P, const WgTables *__restrict__ Tg,
                                                                          const int *__restrict__ envs,
                                                                          const long long *__restrict__ keys, int count, int lazy,
                                                                          volatile unsigned long long *fault, unsigned int *claim) {
    __shared__ WgWarp sh[D2D_WG_WARPS];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int w = blockIdx.x * D2D_WG_WARPS + wid;
    if (w >= count) return;
#define WG_ABANDON return
#include "d2d_worldgen_body.inc"
#undef WG_ABANDON
}

// The worlds the seed queue handed out in the step just logged (d2d_episode_log_kernel): list and count are device data, so
// the launch needs no host round trip and can be captured in a graph.  Grid-stride over warps; always lazy.
__global__ void __launch_bounds__(D2D_WG_WARPS * 32, D2D_WG_LIST_MIN_BLOCKS) d2d_worldgen_list_kernel(const DevP P, const WgTables *__restrict__ Tg,
                                                                               const int *__restrict__ envs,
                                                                               const long long *__restrict__ keys,
                                                                               const int *__restrict__ count,
                                                                               volatile unsigned long long *fault,
                                                                               unsigned int *claim) {
    __shared__ WgWarp sh[D2D_WG_WARPS];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int lazy = 1;
    const int n = *count;
    for (int w = blockIdx.x * D2D_WG_WARPS + wid; w < n; w += gridDim.x * D2D_WG_WARPS) {
        __syncwarp();                    // every lane is done with the previous world's shared memory
        {
#define WG_ABANDON goto next_world
#include "d2d_worldgen_body.inc"
#undef WG_ABANDON
        }
    next_world:;
    }
}
#endif
