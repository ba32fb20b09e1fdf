// d2d_render.cuh -- RGB frames of envs drawn from the arena (d2d_render): the reference's Drone2DEnv2.render
// (drone_v2.py:263-303, utils.py:31-64, 550-558, 786-817) as rgb_array frames.  Reads the arena, writes only the frames.
//
// One block per (env, band of frame rows).  A band is a contiguous byte range of the C-contiguous [H][W][3] frame
// (at most D2D_RENDER_BAND_PIX pixels).  The block
//   1. stages the env's belief and ground-truth rows in shared memory;
//   2. rasterises the agents, trackers and waypoints whose bounding box touches the band: each warp ballots 32 items at a
//      time and then walks the boxes of the hits with all lanes; agents leave their index + 1 per pixel (atomicMax: the
//      highest index wins), rings and waypoints a bit;
//   3. composes every pixel of the band back to front (cells, view, plan, trackers, agents, drone) into a shared-memory copy
//      of the band that has the destination's alignment modulo 16;
//   4. stores the band with byte stores up to the first 16-byte boundary, 16-byte stores after it and byte stores for the
//      tail, so any alignment of the output works and a warp's stores are contiguous.
// Pixel rule (DESIGN.md section 2, "Rendering"): s = map_scale / ppc, pixel (row r, col c) has the centre ((c + 0.5) s,
// (r + 0.5) s); a disc holds it iff (x-cx)*(x-cx) + (y-cy)*(y-cy) <= R*R in fp64 (built with -fmad=false).
#pragma once
#include "d2d_state.cuh"
#include "d2d_math.cuh"
#include "d2d_step.cuh"

#define D2D_RENDER_THREADS 256
#define D2D_RENDER_BAND_PIX 4096     // pixels of one band: 12 KB of output per block

struct RenderList { int32_t e[D2D_RENDER_MAX_LIST]; };

struct RenderArgs {
    uint8_t *frames;
    int32_t first_env, count, use_list;
    int32_t ppc, layers, W, band_rows, nbands;
    double s;                        // map_scale / ppc
    double span;                     // ray_da * (n_rays - 1): angle from ray 0 to the last ray
};

// box of the pixels whose centre can lie within R of (cx, cy), clipped to columns [0, W) and rows [r0, r1); one pixel of
// slack on every side (the exact test decides).  Returns false when the box is empty.
__device__ __forceinline__ bool d2d_render_box(double cx, double cy, double R, double s, int W, int r0, int r1,
                                               int &c_lo, int &c_hi, int &y_lo, int &y_hi) {
    const double big = 1e6;
    double a = floor((cx - R) / s) - 1.0, b = floor((cx + R) / s) + 1.0;
    double u = floor((cy - R) / s) - 1.0, v = floor((cy + R) / s) + 1.0;
    if (!(a <= b && u <= v)) return false;       // NaN
    a = fmax(a, -1.0); b = fmin(b, big); u = fmax(u, -1.0); v = fmin(v, big);
    c_lo = max((int)a, 0); c_hi = min((int)fmin(b, (double)(W - 1)), W - 1);
    y_lo = max((int)u, r0); y_hi = min((int)fmin(v, (double)(r1 - 1)), r1 - 1);
    return c_lo <= c_hi && y_lo <= y_hi;
}

__device__ __forceinline__ double d2d_render_d2(int r, int c, double s, double cx, double cy) {
    const double x = ((double)c + 0.5) * s, y = ((double)r + 0.5) * s;
    const double dx = x - cx, dy = y - cy;
    return dx * dx + dy * dy;
}

__global__ void __launch_bounds__(D2D_RENDER_THREADS) d2d_render_kernel(const DevP P, const RenderArgs A, const RenderList L) {
    __shared__ __align__(16) uint8_t obuf[D2D_RENDER_BAND_PIX * 3 + 16];
    __shared__ unsigned int own[D2D_RENDER_BAND_PIX];                  // agent index + 1 (0: none)
    __shared__ unsigned int ring_bits[D2D_RENDER_BAND_PIX / 32], way_bits[D2D_RENDER_BAND_PIX / 32];
    __shared__ __align__(16) uint8_t bel[D2D_CELLS + 12];
    __shared__ uint64_t gt[D2D_GRID];
    __shared__ double wedge[4];                                        // cos / sin of ray 0 and of the last ray

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = D2D_RENDER_THREADS / 32;
    const int slot = blockIdx.x / A.nbands, band = blockIdx.x - slot * A.nbands;
    const int e = A.use_list ? L.e[slot] : A.first_env + slot;
    const int W = A.W, H = 50 * A.ppc, ppc = A.ppc, layers = A.layers;
    const int r0 = band * A.band_rows, r1 = min(r0 + A.band_rows, H);
    const int npix = (r1 - r0) * W;
    const double s = A.s;
    const EnvRec &rec = P.rec[e];
    const double px = rec.px, py = rec.py;

    uint8_t *dst = A.frames + (size_t)slot * ((size_t)H * W * 3) + (size_t)r0 * W * 3;
    const int shift = (int)((uintptr_t)dst & 15);

    for (int p = tid; p < npix; p += D2D_RENDER_THREADS) own[p] = 0u;
    for (int p = tid; p < D2D_RENDER_BAND_PIX / 32; p += D2D_RENDER_THREADS) { ring_bits[p] = 0u; way_bits[p] = 0u; }
    if (layers & (D2D_RENDER_GROUND_TRUTH | D2D_RENDER_BELIEF)) {
        const uint32_t *bsrc = (const uint32_t *)(P.belief + (size_t)e * D2D_BELIEF_STRIDE);
        for (int q = tid; q < D2D_CELLS / 4; q += D2D_RENDER_THREADS) ((uint32_t *)bel)[q] = __ldg(bsrc + q);
        for (int q = tid; q < D2D_GRID; q += D2D_RENDER_THREADS) gt[q] = __ldg(P.gt_rows + (size_t)e * D2D_GRID + q);
    }
    if ((layers & D2D_RENDER_VIEW) && tid < 2) {
        // the values of d2d_sincos, from its inline double-double core: a call of the shared non-inlined copy from one more
        // kernel would change how the compiler builds the existing kernels that call it
        d2d_dd sn, cs;
        d2d_sincos_dd(d2d_ray_angle(P, rec.yaw, tid == 0 ? 0 : P.n_rays - 1), &sn, &cs);
        wedge[2 * tid] = cs.h + cs.l;
        wedge[2 * tid + 1] = sn.h + sn.l;
    }
    __syncthreads();

    // ---- rasterise the culled items of this band (warp-level; no block barrier inside)
    const int N = P.N;
    if (layers & (D2D_RENDER_AGENTS | D2D_RENDER_TRACKERS)) {
        for (int pass = 0; pass < 2; pass++) {
            const bool agents = pass == 0;
            if (!(layers & (agents ? D2D_RENDER_AGENTS : D2D_RENDER_TRACKERS))) continue;
            for (int base = warp * 32; base < N; base += nwarps * 32) {
                const int k = base + lane;
                double cx = 0.0, cy = 0.0, R = 0.0;
                int cl = 0, ch = -1, yl = 0, yh = -1;
                bool on = false;
                if (k < N) {
                    const size_t ek = (size_t)e * P.NP + k;
                    if (agents) {
                        const double2 a = P.apos[ek];
                        cx = a.x; cy = a.y; R = P.arad[ek];
                        on = true;
                    } else if (P.trk_active[ek]) {
                        cx = P.trk_mu[ek * 4]; cy = P.trk_mu[ek * 4 + 1]; R = P.trk_radius[ek];
                        on = true;
                    }
                    on = on && d2d_render_box(cx, cy, R, s, W, r0, r1, cl, ch, yl, yh);
                }
                unsigned m = __ballot_sync(0xffffffffu, on);
                while (m) {
                    const int b = __ffs(m) - 1;
                    m &= m - 1;
                    const double bx = __shfl_sync(0xffffffffu, cx, b), by = __shfl_sync(0xffffffffu, cy, b);
                    const double bR = __shfl_sync(0xffffffffu, R, b);
                    const int bcl = __shfl_sync(0xffffffffu, cl, b), bch = __shfl_sync(0xffffffffu, ch, b);
                    const int byl = __shfl_sync(0xffffffffu, yl, b), byh = __shfl_sync(0xffffffffu, yh, b);
                    const int bw = bch - bcl + 1, n = bw * (byh - byl + 1);
                    const double R2 = bR * bR;
                    double Ri = bR - s;
                    Ri = Ri > 0.0 ? Ri : 0.0;
                    const double Ri2 = Ri * Ri;
                    for (int q = lane; q < n; q += 32) {
                        const int r = byl + q / bw, c = bcl + q % bw;
                        const double d2 = d2d_render_d2(r, c, s, bx, by);
                        const int p = (r - r0) * W + c;
                        if (agents) {
                            if (d2 <= R2) atomicMax(&own[p], (unsigned)(base + b + 1));
                        } else if (Ri2 < d2 && d2 <= R2) {
                            atomicOr(&ring_bits[p >> 5], 1u << (p & 31));
                        }
                    }
                }
            }
        }
    }
    if ((layers & D2D_RENDER_PLAN) && P.planner == D2D_PLANNER_PRIMITIVE) {
        const int n_way = P.n_way, total = rec.nseg * n_way, half = ppc / 4;
        const double *coeff = P.traj_coeff + (size_t)e * D2D_MAX_SEGMENTS * 6;
        for (int a = rec.cursor + tid; a < total; a += D2D_RENDER_THREADS) {
            const int seg = a / n_way, ws = a - seg * n_way, ti = n_way - 1 - ws;
            const double *cf = coeff + (size_t)seg * 6;
            const double t = P.tab->t_way[ti], t2 = P.tab->t_way2[ti];
            // the arithmetic of the step's waypoint pop (d2d_step.cuh) and of vec_env.trajectory_waypoints
            const double wx = rint(D2D_FMA(t2, cf[2], cf[0] + t * cf[1]));
            const double wy = rint(D2D_FMA(t2, cf[5], cf[3] + t * cf[4]));
            const double fc = floor(wx * (double)ppc / P.scale), fr = floor(wy * (double)ppc / P.scale);
            if (!(fc >= -64.0 && fc < (double)W + 64.0 && fr >= -64.0 && fr < (double)H + 64.0)) continue;
            const int col = (int)fc, row = (int)fr;
            const int c_lo = max(col - half, 0), c_hi = min(col + half, W - 1);
            const int y_lo = max(row - half, r0), y_hi = min(row + half, r1 - 1);
            for (int r = y_lo; r <= y_hi; r++)
                for (int c = c_lo; c <= c_hi; c++) {
                    const int p = (r - r0) * W + c;
                    atomicOr(&way_bits[p >> 5], 1u << (p & 31));
                }
        }
    }
    __syncthreads();

    // ---- compose every pixel of the band, back to front
    const bool gt_on = (layers & D2D_RENDER_GROUND_TRUTH) != 0, bel_on = (layers & D2D_RENDER_BELIEF) != 0;
    const double w0c = wedge[0], w0s = wedge[1], w1c = wedge[2], w1s = wedge[3];
    const double depth2 = P.depth2, dr2 = P.drone_r * P.drone_r;
    const double tgx = rec.tgx, tgy = rec.tgy;
    const bool wide = A.span > D2D_PI;
    uint8_t *ob = obuf + shift;
    for (int p = tid; p < npix; p += D2D_RENDER_THREADS) {
        const int rr = p / W, c = p - rr * W, r = r0 + rr;
        const int i = c / ppc, j = r / ppc;
        int R = 255, G = 255, Bc = 255;
        if (gt_on || bel_on) {
            const int wall = (int)((gt[i] >> j) & 1ull);
            const int b = bel[i * D2D_GRID + j];
            int v;                                            // 0 white, 1 black, 2 grey 128, 3 grey 64
            if (gt_on && bel_on) v = b == 0 ? (wall ? 3 : 2) : (b == 1 ? 1 : 0);
            else if (gt_on) v = wall;
            else v = b == 0 ? 2 : (b == 1 ? 1 : 0);
            R = G = Bc = v == 0 ? 255 : (v == 1 ? 0 : (v == 2 ? 128 : 64));
        }
        const double x = ((double)c + 0.5) * s, y = ((double)r + 0.5) * s;
        if (layers & D2D_RENDER_VIEW) {
            const double vx = x - px, vy = y - py;
            if (vx * vx + vy * vy <= depth2) {
                bool in = true;
                if (!(vx == 0.0 && vy == 0.0)) {
                    const double c0 = w0c * vy - w0s * vx;    // cross(d0, v)
                    const double c1 = vx * w1s - vy * w1c;    // cross(v, d1)
                    in = wide ? !(c0 < 0.0 && c1 < 0.0) : (c0 >= 0.0 && c1 >= 0.0);
                }
                if (in) { R = (3 * R + 255) >> 2; G = (3 * G + 255) >> 2; Bc = (3 * Bc) >> 2; }
            }
        }
        if (layers & D2D_RENDER_PLAN) {
            const double dx = x - tgx, dy = y - tgy;
            if (dx * dx + dy * dy <= dr2) { R = 255; G = 0; Bc = 255; }
            if ((way_bits[p >> 5] >> (p & 31)) & 1u) { R = 0; G = 160; Bc = 0; }
        }
        if ((layers & D2D_RENDER_TRACKERS) && ((ring_bits[p >> 5] >> (p & 31)) & 1u)) { R = 255; G = 140; Bc = 0; }
        if (layers & D2D_RENDER_AGENTS) {
            const unsigned o = own[p];
            if (o) {
                if (P.hit[(size_t)e * P.NP + (o - 1)]) { R = 220; G = 0; Bc = 0; } else { R = 0; G = 0; Bc = 220; }
            }
        }
        if (layers & D2D_RENDER_DRONE) {
            const double dx = x - px, dy = y - py;
            if (dx * dx + dy * dy <= dr2) { R = 0; G = 200; Bc = 0; }
        }
        ob[3 * p] = (uint8_t)R; ob[3 * p + 1] = (uint8_t)G; ob[3 * p + 2] = (uint8_t)Bc;
    }
    __syncthreads();

    // ---- store the band: bytes up to the first 16-byte boundary of dst, 16-byte stores, bytes for the tail
    const int nbytes = npix * 3;
    const int head = min((16 - shift) & 15, nbytes);
    const int nvec = (nbytes - head) >> 4;
    const int tail0 = head + (nvec << 4);
    if (tid < head) dst[tid] = ob[tid];
    const uint4 *vs = (const uint4 *)(ob + head);
    uint4 *vd = (uint4 *)(dst + head);
    for (int q = tid; q < nvec; q += D2D_RENDER_THREADS) vd[q] = vs[q];
    if (tid < nbytes - tail0) dst[tail0 + tid] = ob[tail0 + tid];
}
