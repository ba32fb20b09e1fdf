// d2d_difficulty.cuh -- the survivability difficulty metrics (d2d_difficulty): agents stepped alone from each env's reset
// snapshot, and every position of a grid tested against them after every step.  Reads the snapshot, writes only the
// outputs (drone2d.h documents them).
//
// Under CVM no agent looks at the drone or at another agent, so one agent trajectory per world answers every position.
// One warp per (env, chunk of 64 grid positions):
//   1. lanes evaluate the five static probes of the chunk's positions (d2d_static_probe, the step kernels' arithmetic);
//   2. lanes take 32 agents at a time and step them K times in registers (d2d_cvm_agent_step); after each step an agent
//      finds the grid indices within r + drone_radius per axis by division and tests only those exactly; the warp ORs the
//      lanes' 64-bit hit masks (__reduce_or_sync), and lane l keeps the first hit of positions l and l + 32 in registers
//      and ORs slot bits into its own shared-memory words (no atomics);
//   3. the chunk's first_hit / static_hit are stored, and its collision_state bytes with 16-byte stores.
// Re-stepping the agents for every 64-position chunk keeps shared memory bounded (64 x ceil(n_slots / 32) words a warp).
#pragma once
#include "d2d_state.cuh"
#include "d2d_math.cuh"
#include "d2d_agent_math.cuh"
#include "d2d_step.cuh"

#define D2D_DIFF_WARPS 4

struct DiffOut {
    int16_t *first_hit;
    uint8_t *static_hit, *cs;
    int32_t first_env, count, nchunks, nwords;     // nwords = ceil(n_slots / 32): slot-bit words per position
};

__device__ __forceinline__ uint8_t d2d_diff_cs_byte(const uint32_t *bits, const uint8_t *stat, int nwords, int ns, int b) {
    const int p = b / ns, s = b - p * ns;
    return stat[p] ? (uint8_t)0 : (uint8_t)((bits[p * nwords + (s >> 5)] >> (s & 31)) & 1u);
}

__global__ void __launch_bounds__(D2D_DIFF_WARPS * 32) d2d_difficulty_kernel(const DevP P, const DiffOut O,
                                                                             const d2d_difficulty_spec S) {
    extern __shared__ uint32_t d2d_diff_bits[];                // [D2D_DIFF_WARPS][64][nwords]
    __shared__ uint8_t stat_s[D2D_DIFF_WARPS][64];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long task = (long long)blockIdx.x * D2D_DIFF_WARPS + warp;
    if (task >= (long long)O.count * O.nchunks) return;      // a whole warp leaves; the kernel has no block barrier
    const int w = (int)(task / O.nchunks), chunk = (int)(task - (long long)w * O.nchunks);
    const int e = O.first_env + w;
    const int ny = S.ny, npos = S.nx * ny, p0 = chunk * 64, pc = min(64, npos - p0);
    const int nwords = O.nwords;
    uint32_t *bits = d2d_diff_bits + (size_t)warp * 64 * nwords;
    uint8_t *stat = stat_s[warp];
    for (int q = lane; q < 64 * nwords; q += 32) bits[q] = 0u;

    // ---- 1. static probes (Drone2D.is_collide utils.py:766-771)
    const uint64_t *gt = P.gt_rows + (size_t)e * D2D_GRID;
    for (int p = lane; p < 64; p += 32) {
        int st = 0;
        if (p < pc) {
            const int i = (p0 + p) / ny, j = p0 + p - i * ny;
            const double x = S.x0 + (double)i * S.step, y = S.y0 + (double)j * S.step;
            for (int q = 0; q < 5; q++) st |= d2d_static_probe(P, gt, x, y, q);
        }
        stat[p] = (uint8_t)st;
    }
    __syncwarp();

    // ---- 2. agents, 32 at a time, K steps each
    const int ilo = p0 / ny, ihi = (p0 + pc - 1) / ny;         // grid rows the chunk touches
    const int N = P.N, K = S.steps;
    const double dt = P.dt, edge = P.scale, mw = P.map_w, mh = P.map_h;
    int first0 = 0, first1 = 0;                                // first hit step of positions p0 + lane, p0 + 32 + lane
    for (int a0 = 0; a0 < N; a0 += 32) {
        const bool on = a0 + lane < N;
        double2 pos = double2{0.0, 0.0}, pref = double2{0.0, 0.0};
        double r = 0.0;
        if (on) {
            const size_t g = (size_t)e * P.NP + a0 + lane;
            pos = P.apos0[g]; pref = P.apref0[g]; r = P.arad[g];
        }
        const double R = r + P.drone_r;
#pragma unroll 1
        for (int t = 1; t <= K; t++) {
            unsigned long long m = 0ull;
            if (on) {
                d2d_cvm_agent_step(pos.x, pos.y, pref.x, pref.y, r, dt, edge, mw, mh);
                int il, ih, jl, jh;
                d2d_grid_span(pos.x, R, S.x0, S.step, S.nx, &il, &ih);
                d2d_grid_span(pos.y, R, S.y0, S.step, ny, &jl, &jh);
                il = max(il, ilo); ih = min(ih, ihi);
                for (int i = il; i <= ih; i++) {
                    const double x = S.x0 + (double)i * S.step;
                    for (int j = jl; j <= jh; j++) {
                        const int p = i * ny + j - p0;
                        if (p >= 0 && p < pc && d2d_agent_hits(pos.x, pos.y, R, x, S.y0 + (double)j * S.step)) m |= 1ull << p;
                    }
                }
            }
            const unsigned lo = __reduce_or_sync(0xffffffffu, (unsigned)m);
            const unsigned hi = __reduce_or_sync(0xffffffffu, (unsigned)(m >> 32));
            if (lo | hi) {
                const unsigned sl = S.slot[t - 1];
                const bool rec = nwords != 0 && sl != D2D_DIFF_NO_SLOT;
                if ((lo >> lane) & 1u) {
                    if (first0 == 0 || t < first0) first0 = t;
                    if (rec) bits[lane * nwords + (sl >> 5)] |= 1u << (sl & 31);
                }
                if ((hi >> lane) & 1u) {
                    if (first1 == 0 || t < first1) first1 = t;
                    if (rec) bits[(lane + 32) * nwords + (sl >> 5)] |= 1u << (sl & 31);
                }
            }
        }
    }

    // ---- 3. outputs
    const size_t base = (size_t)w * npos + p0;
    if (lane < pc) { O.first_hit[base + lane] = (int16_t)first0; O.static_hit[base + lane] = stat[lane]; }
    if (lane + 32 < pc) { O.first_hit[base + 32 + lane] = (int16_t)first1; O.static_hit[base + 32 + lane] = stat[lane + 32]; }
    if (O.cs) {
        __syncwarp();
        const int ns = S.n_slots, nbytes = pc * ns;
        uint8_t *dst = O.cs + base * ns;
        // bytes up to the first 16-byte boundary of dst, 16-byte stores, bytes for the tail
        const int head = min((int)((16 - ((uintptr_t)dst & 15)) & 15), nbytes);
        const int nvec = (nbytes - head) >> 4, tail0 = head + (nvec << 4);
        if (lane < head) dst[lane] = d2d_diff_cs_byte(bits, stat, nwords, ns, lane);
        for (int v = lane; v < nvec; v += 32) {
            uint32_t wv[4];
            for (int q = 0; q < 4; q++) {
                uint32_t x = 0u;
                for (int b = 0; b < 4; b++)
                    x |= (uint32_t)d2d_diff_cs_byte(bits, stat, nwords, ns, head + (v << 4) + 4 * q + b) << (8 * b);
                wv[q] = x;
            }
            ((uint4 *)(dst + head))[v] = make_uint4(wv[0], wv[1], wv[2], wv[3]);
        }
        if (lane < nbytes - tail0) dst[tail0 + lane] = d2d_diff_cs_byte(bits, stat, nwords, ns, tail0 + lane);
    }
}
