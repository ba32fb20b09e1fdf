// d2d_agent_math.cuh -- one CVM Agent.step and the dynamic-collision test, as host/device helpers.  d2d_difficulty_kernel
// steps agents with them on the device; tests/helpers/difficulty_twin.cpp compiles the same code on the host (g++
// -ffp-contract=off) so the CPU tests hold it to the oracle.
//
// d2d_cvm_agent_step restates the CVM branch of d2d_phase_agents (d2d_step.cuh) operation for operation; the step kernel
// keeps its own copy so that its code is unchanged, and tests/test_difficulty_host.py holds the two together through the
// oracle, which the step kernels are held to.  The small-crowd form of the rollout kernel (d2d_agents_lane) steps its
// agents with this helper; tests/test_gpu_rollout.py holds it to the step kernels bit for bit.
#pragma once
#include "d2d_math.cuh"

// Agent.step under CVM (drone_v2.py:178, utils.py:470-486): velocity IS pref_velocity (the same ndarray), so a bounce is
// visible through the velocity unless the 30-degree rotation (speed <= 5) rebound pref_velocity to a new array first.
// (px, py): position, (ux, uy): pref_velocity; edge = map_scale.
D2D_HD void d2d_cvm_agent_step(double &px, double &py, double &ux, double &uy, double r, double dt, double edge,
                               double map_w, double map_h) {
    const double C6 = 0.8660254037844387, S6 = 0.49999999999999994;   // math.cos(pi/6), math.sin(pi/6) (glibc)
    double vx = ux, vy = uy;
    const double nx = px + vx * dt, ny = py + vy * dt;
    bool rebound = false;
    if (d2d_norm2_le(vx, vy, 5.0)) {   // utils.py:476-477: rotation by 30 deg rebinds pref_velocity
        const double qx = D2D_FMA(C6, ux, -S6 * uy);
        const double qy = D2D_FMA(S6, ux, C6 * uy);
        ux = qx; uy = qy;
        rebound = true;
    }
    if (nx < edge + r) ux = fabs(ux);
    else if (nx > map_w - edge - r) ux = -fabs(ux);
    if (ny < edge + r) uy = fabs(uy);
    else if (ny > map_h - edge - r) uy = -fabs(uy);
    if (!rebound) { vx = ux; vy = uy; }
    px = px + vx * dt;
    py = py + vy * dt;
}

// Drone2D.is_collide's agent test (utils.py:773-776): np.linalg.norm(agent.position - p) < agent.radius + drone.radius
D2D_HD bool d2d_agent_hits(double ax, double ay, double R, double x, double y) { return d2d_norm2_lt(ax - x, ay - y, R); }

// The grid indices i (x = x0 + i * step) that can lie within R of a: [*lo, *hi], clipped to [0, n); one index of slack on
// each side (the exact test decides).  Empty when *lo > *hi.
D2D_HD void d2d_grid_span(double a, double R, double x0, double step, int n, int *lo, int *hi) {
    double l = ceil((a - R - x0) / step) - 1.0, h = floor((a + R - x0) / step) + 1.0;
    l = l > 0.0 ? (l < (double)n ? l : (double)n) : 0.0;     // also maps NaN to 0 ...
    h = h < (double)(n - 1) ? h : (double)(n - 1);           // ... and to n - 1
    *lo = (int)l;
    *hi = h >= l ? (int)h : -1;
}
