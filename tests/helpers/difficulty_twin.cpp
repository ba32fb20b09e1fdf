// Host-compiled twin of the agent stepping and hit search of csrc/d2d_difficulty.cuh for the CPU test-suite
// (tests/test_difficulty_host.py), over the same D2D_HD helpers (csrc/d2d_agent_math.cuh).
// Build: g++ -O2 -ffp-contract=off -shared -fPIC (no FMA contraction: same arithmetic as nvcc -fmad=false).
#include <stddef.h>
#include "../../include/drone2d.h"
#include "../../gym_drone2d_activeperception_b200/csrc/d2d_agent_math.cuh"

extern "C" {
// n agents from (pos, pref) stepped `steps` times; the positions after step k go to out[k-1][n][2]
void dt_trajectory(long n, const double *pos, const double *pref, const double *rad, double dt, double edge, double map_w,
                   double map_h, long steps, double *out) {
    for (long a = 0; a < n; a++) {
        double px = pos[2 * a], py = pos[2 * a + 1], ux = pref[2 * a], uy = pref[2 * a + 1];
        for (long k = 0; k < steps; k++) {
            d2d_cvm_agent_step(px, py, ux, uy, rad[a], dt, edge, map_w, map_h);
            out[(k * n + a) * 2] = px;
            out[(k * n + a) * 2 + 1] = py;
        }
    }
}

// first_hit[nx * ny] of one world, searched as the kernel searches (d2d_grid_span per axis, then d2d_agent_hits)
void dt_first_hit(long n, const double *pos, const double *pref, const double *rad, double drone_r, double dt, double edge,
                  double map_w, double map_h, double x0, double y0, double step, int nx, int ny, int steps, short *first) {
    for (int p = 0; p < nx * ny; p++) first[p] = 0;
    for (long a = 0; a < n; a++) {
        double px = pos[2 * a], py = pos[2 * a + 1], ux = pref[2 * a], uy = pref[2 * a + 1];
        const double R = rad[a] + drone_r;
        for (int k = 1; k <= steps; k++) {
            d2d_cvm_agent_step(px, py, ux, uy, rad[a], dt, edge, map_w, map_h);
            int il, ih, jl, jh;
            d2d_grid_span(px, R, x0, step, nx, &il, &ih);
            d2d_grid_span(py, R, y0, step, ny, &jl, &jh);
            for (int i = il; i <= ih; i++)
                for (int j = jl; j <= jh; j++)
                    if (d2d_agent_hits(px, py, R, x0 + (double)i * step, y0 + (double)j * step) &&
                        (first[i * ny + j] == 0 || k < first[i * ny + j]))
                        first[i * ny + j] = (short)k;
        }
    }
}

long dt_sizeof_spec(void) { return (long)sizeof(d2d_difficulty_spec); }
long dt_offsetof_slot(void) { return (long)offsetof(d2d_difficulty_spec, slot); }

int dt_agent_hits(double ax, double ay, double R, double x, double y) { return d2d_agent_hits(ax, ay, R, x, y) ? 1 : 0; }
}
