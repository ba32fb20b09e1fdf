// d2d_clone.cuh -- per-env state copies: env -> env inside the arena (d2d_clone_envs), env -> packed row (d2d_save_state)
// and packed row -> env (d2d_load_state), all driven by one field table built from the per-env tags of add_buf.
#pragma once
#include <stdint.h>
#include <cuda_runtime.h>

#define D2D_CLONE_MAX_FIELDS 64
#define D2D_CLONE_THREADS 256
#define D2D_CLONE_UNROLL 4            // copy units a thread has in flight (loads issued before the first store)

// One per-env row: env e's `bytes` bytes start at arena + off + e * stride; in a packed state row they start at `pack`.
// A buffer with several per-env planes (rng_pos, rng_gauss) contributes one field per plane.
struct CloneField {
    unsigned long long off, stride;
    unsigned int bytes, pack;
};

struct CloneTable {
    int n;                            // fields in use
    unsigned int pack_bytes;          // bytes per packed state row (a multiple of 128)
    CloneField f[D2D_CLONE_MAX_FIELDS];
};

enum { D2D_CLONE_ARENA = 0, D2D_CLONE_SAVE = 1, D2D_CLONE_LOAD = 2 };

__device__ __forceinline__ uint4 d2d_clone_ld(const unsigned char *p, int lg) {
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    switch (lg) {
        case 4: v = *(const uint4 *)p; break;
        case 3: { const uint2 t = *(const uint2 *)p; v.x = t.x; v.y = t.y; } break;
        case 2: v.x = *(const unsigned int *)p; break;
        case 1: v.x = *(const unsigned short *)p; break;
        default: v.x = *p; break;
    }
    return v;
}

__device__ __forceinline__ void d2d_clone_st(unsigned char *p, uint4 v, int lg) {
    switch (lg) {
        case 4: *(uint4 *)p = v; break;
        case 3: *(uint2 *)p = make_uint2(v.x, v.y); break;
        case 2: *(unsigned int *)p = v.x; break;
        case 1: *(unsigned short *)p = (unsigned short)v.x; break;
        default: *p = (unsigned char)v.x; break;
    }
}

// Block b copies copy b.  ARENA: env src[b] -> env dst[b].  SAVE: env src[b] (src null: env b) -> packed row b.
// LOAD: packed row b -> env dst[b].  The host has checked every index, and that no env is written twice or both read and
// written.  Each field is cut into units of the widest access (16, 8, 4, 2 or 1 bytes) that both rows' addresses and its
// length allow; the units of all fields form one list that the block's threads walk D2D_CLONE_UNROLL units at a time.
__global__ void __launch_bounds__(D2D_CLONE_THREADS) d2d_clone_kernel(const CloneTable T, const int mode,
                                                                      unsigned char *arena,
                                                                      unsigned char *packed,
                                                                      const int *__restrict__ src, const int *__restrict__ dst) {
    __shared__ const unsigned char *s_src[D2D_CLONE_MAX_FIELDS];
    __shared__ unsigned char *s_dst[D2D_CLONE_MAX_FIELDS];
    __shared__ int s_lg[D2D_CLONE_MAX_FIELDS];
    __shared__ int s_first[D2D_CLONE_MAX_FIELDS + 1];       // first unit of each field; [n] = units in total
    const int b = blockIdx.x, tid = threadIdx.x;
    if (tid < 32) {
        const int es = mode == D2D_CLONE_LOAD ? 0 : (src ? src[b] : b);
        const int ed = mode == D2D_CLONE_SAVE ? 0 : dst[b];
        unsigned char *row = packed + (size_t)b * T.pack_bytes;
        int carry = 0;
        for (int j0 = 0; j0 < D2D_CLONE_MAX_FIELDS; j0 += 32) {
            const int j = j0 + tid;
            int units = 0;
            if (j < T.n) {
                const CloneField f = T.f[j];
                unsigned char *a = arena + f.off;
                const unsigned char *sp = mode == D2D_CLONE_LOAD ? row + f.pack : a + (size_t)es * f.stride;
                unsigned char *dp = mode == D2D_CLONE_SAVE ? row + f.pack : a + (size_t)ed * f.stride;
                const unsigned int al = (unsigned int)(uintptr_t)sp | (unsigned int)(uintptr_t)dp | f.bytes;
                const int lg = (al & 15u) == 0 ? 4 : (al & 7u) == 0 ? 3 : (al & 3u) == 0 ? 2 : (al & 1u) == 0 ? 1 : 0;
                s_src[j] = sp; s_dst[j] = dp; s_lg[j] = lg;
                units = (int)(f.bytes >> lg);
            }
            int incl = units;                                 // inclusive warp scan of the unit counts
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, incl, o);
                if (tid >= o) incl += y;
            }
            if (j <= T.n) s_first[j] = carry + incl - units;
            carry += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (tid == 0 && T.n == D2D_CLONE_MAX_FIELDS) s_first[T.n] = carry;
    }
    __syncthreads();
    const int total = s_first[T.n];
    int j = 0;                                                // this thread's units only increase: the field cursor too
    for (int base = tid; base < total; base += D2D_CLONE_THREADS * D2D_CLONE_UNROLL) {
        uint4 v[D2D_CLONE_UNROLL];
        unsigned char *dp[D2D_CLONE_UNROLL];
        int lg[D2D_CLONE_UNROLL];
#pragma unroll
        for (int k = 0; k < D2D_CLONE_UNROLL; k++) {
            const int u = base + k * D2D_CLONE_THREADS;
            lg[k] = -1;
            if (u < total) {
                while (s_first[j + 1] <= u) j++;
                lg[k] = s_lg[j];
                const size_t o = (size_t)(u - s_first[j]) << lg[k];
                dp[k] = s_dst[j] + o;
                v[k] = d2d_clone_ld(s_src[j] + o, lg[k]);
            }
        }
#pragma unroll
        for (int k = 0; k < D2D_CLONE_UNROLL; k++)
            if (lg[k] >= 0) d2d_clone_st(dp[k], v[k], lg[k]);
    }
}
