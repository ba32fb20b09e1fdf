// d2d_episode.cuh -- the episode log (d2d_enable_episode_log / d2d_read_episode_log) and the seed queue
// (d2d_set_seed_queue): one kernel behind every logged step turns the step's `done` bytes into records.
#pragma once
#include "d2d_state.cuh"

#define D2D_EP_THREADS 1024                // per block: 16 done bytes per thread and pass, 16384 envs per pass

static_assert(sizeof(d2d_episode_record) == 48, "d2d_episode_record must be 48 bytes (drone2d.h)");

// Device side of the log (passed by value).  head: [0] records written since the last read, [1] steps logged, [2] seeds
// handed out by the queue, [3] queue length.
struct EpLog {
    d2d_episode_record *rec;     // [capacity]
    long long capacity;
    long long *head;             // [4]
    long long *world_seed;       // [B] world key of each env
    int *list;                   // [B] scratch: the envs that reported done this step, ascending (each block its own entries)
    int *gen_env;                // [B] worlds the queue handed out this step (read by d2d_worldgen_list_kernel) ...
    long long *gen_key;          // [B] ... their world keys
    int *gen_count;              // ... and their number
    unsigned int *ticket;        // blocks of d2d_episode_log_kernel done with this step (0 between launches)
    const long long *queue;      // [head[3]] world keys of the queue
};

// bit k of the result: byte k of the 16 bytes is non-zero
__device__ __forceinline__ unsigned ep_nonzero_bytes(uint4 v) {
    unsigned m = 0;
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const uint32_t t = __vcmpne4(w[k], 0u) & 0x01010101u;
        m |= ((t | (t >> 7) | (t >> 14) | (t >> 21)) & 0xfu) << (4 * k);
    }
    return m;
}

// One block per SM at most (grid G).  Phase 1: every block compacts done[0, B) with 16-byte loads and a block prefix sum
// per pass of 16384 envs (no inter-block scan: each block scans the whole byte array, which L2 serves), and keeps the
// positions it owns: record j belongs to block (j / 32) % G, warp j % 32.  Phase 2: each warp counts the explored cells
// of its finished env (as d2d_count_explored_warp does) and writes the record; while the queue has seeds, the env takes
// the next one in list order.  The last block to finish (ticket) advances the head.
__global__ void __launch_bounds__(D2D_EP_THREADS) d2d_episode_log_kernel(const DevP P, const EpLog L) {
    __shared__ int warp_sum[D2D_EP_THREADS / 32];
    __shared__ int total;
    __shared__ long long head[4];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, G = gridDim.x;
    if (tid < 4) head[tid] = L.head[tid];
    if (tid == 0) total = 0;
    __syncthreads();
    const int nw = (P.B + 15) / 16;                      // the done buffer is padded to a multiple of 16 bytes
    for (int w0 = 0; w0 < nw; w0 += D2D_EP_THREADS) {
        const int w = w0 + tid;
        unsigned m = 0;
        if (w < nw) {
            m = ep_nonzero_bytes(__ldcg((const uint4 *)P.done + w));
            const int left = P.B - 16 * w;
            if (left < 16) m &= (1u << left) - 1u;
        }
        const int c = __popc(m);
        int x = c;                                        // inclusive warp scan
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
        if (lane == 31) warp_sum[wid] = x;
        __syncthreads();
        if (wid == 0) {
            int y = warp_sum[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int z = __shfl_up_sync(0xffffffffu, y, o); if (lane >= o) y += z; }
            warp_sum[lane] = y;
        }
        __syncthreads();
        int pos = total + (wid ? warp_sum[wid - 1] : 0) + x - c;
        while (m) {
            const int b = __ffs(m) - 1;
            m &= m - 1u;
            if ((pos >> 5) % G == (int)blockIdx.x) L.list[pos] = 16 * w + b;
            pos++;
        }
        __syncthreads();                                  // every thread has read warp_sum and total
        if (tid == 0) total += warp_sum[D2D_EP_THREADS / 32 - 1];
        __syncthreads();
    }
    const int n = total;
    const long long h0 = head[0], step = head[1], q0 = head[2], qlen = head[3];
    const long long avail = qlen > q0 ? qlen - q0 : 0;
    const int taken = (long long)n < avail ? n : (int)avail;
    for (int j = ((int)blockIdx.x << 5) + wid; j < n; j += G << 5) {
        const int e = L.list[j];
        const uint8_t *bel = P.belief + (size_t)e * D2D_BELIEF_STRIDE;
        int cnt = 0;
        for (int q = lane; q < D2D_CELLS / 16; q += 32) {              // cells 0 .. 2495
            const uint4 v = __ldcg((const uint4 *)bel + q);
            cnt += __popc(ep_nonzero_bytes(v));
        }
        if (lane == 0) cnt += __popc(ep_nonzero_bytes(__ldcg((const uint4 *)bel + D2D_CELLS / 16)) & 0xfu);   // 2496 .. 2499
        cnt = __reduce_add_sync(0xffffffffu, cnt);
        if (lane == 0) {
            const long long slot = h0 + j;
            const EnvRec &r = P.rec[e];
            if (slot < L.capacity) {
                d2d_episode_record o;
                o.seed = L.world_seed[e]; o.step = step; o.tracked_steps = r.bufts;
                o.env = e; o.steps = r.steps; o.grid_discovered = cnt; o.trackers = r.bufc;
                o.state_machine = (uint8_t)r.sm; o.collision_flag = P.collision[e]; o.freezing_flag = P.freezing[e];
                o.dead_lock_flag = P.dead_lock[e]; o.reserved = 0;
                L.rec[slot] = o;
            }
            if (j < taken) {
                const long long s = L.queue[q0 + j];
                L.world_seed[e] = s;
                L.gen_env[j] = e; L.gen_key[j] = s;
            }
        }
    }
    // every block has read the head (above) before it takes its ticket; the last one advances it
    __syncthreads();
    if (tid == 0 && atomicAdd(L.ticket, 1u) == (unsigned)G - 1u) {
        L.head[0] = h0 + n; L.head[1] = step + 1; L.head[2] = q0 + taken; *L.gen_count = taken;
        *L.ticket = 0u;
    }
}
