"""NumPy twin of d2d_render_kernel: renders one env's frame from host copies of its buffers, following the pixel rules of
DESIGN.md ("Rendering") literally, so that every byte can be compared with the device.

sin / cos of the two wedge boundary angles are the correctly rounded values the device's d2d_sincos gives, evaluated here
with 90-digit decimal arithmetic.  `render` also returns the mask of wedge-edge pixels (cross product within 1e-9 * |v| of
0) whose verdict the glibc sin / cos the reference would call decide the other way: only those pixels depend on which of
the two 1-ulp-apart values a renderer uses.  A drone on the integer lattice with a boundary on the 45-degree lattice puts a
whole line of pixel centres exactly on the boundary; the sign of their cross product is that of cos - sin in the last ulp,
the same on both sides here, so they are compared like every other pixel."""
import math
from decimal import Decimal, localcontext

import numpy as np

GROUND_TRUTH, BELIEF, VIEW, PLAN, TRACKERS, AGENTS, DRONE, ALL = 1, 2, 4, 8, 16, 32, 64, 127
PI, TWO_PI = 3.141592653589793, 6.283185307179586
DEG2RAD = PI / 180.0
EDGE_TOL = 1e-9

STATE_KEYS = ("belief", "gt_rows", "agent_pos", "agent_radius", "hit", "tracker_active", "tracker_mu", "tracker_radius",
              "drone_x", "drone_y", "drone_yaw", "target_x", "target_y", "traj_coeff", "traj_nseg", "traj_cursor")


def ray_angle(cfg, yaw, ray):
    """d2d_ray_angle (d2d_step.cuh): the wrapped angle of ray `ray` at drone yaw `yaw` (degrees)."""
    fov = cfg.drone_view_range * DEG2RAD
    a0, da = -fov / 2, fov / float(cfg.n_rays)
    ray_a = a0 + da * float(ray)
    a = (TWO_PI - yaw * DEG2RAD) + ray_a
    a = math.copysign(math.fmod(abs(a), TWO_PI), a)
    if a < 0:
        a += TWO_PI
    return a


def sincos_cr(a):
    """(sin(a), cos(a)) correctly rounded to double, as d2d_sincos gives them: Taylor series of the exact binary value of `a`
    (|a| < 7) in 90-digit decimal arithmetic, then float(), which rounds a Decimal correctly."""
    with localcontext() as ctx:
        ctx.prec = 90
        x = Decimal(a)
        x2 = x * x
        tiny = Decimal(10) ** -88
        sn, cs = Decimal(0), Decimal(0)
        term, n = x, 1                  # x^n / n!, n odd
        while abs(term) > tiny:
            sn += term
            term = -term * x2 / ((n + 1) * (n + 2))
            n += 2
        term, n = Decimal(1), 0         # x^n / n!, n even
        while abs(term) > tiny:
            cs += term
            term = -term * x2 / ((n + 1) * (n + 2))
            n += 2
        return float(sn), float(cs)


def _wedge(cfg, sc0, sc1, vx, vy):
    """(inside, c0, c1) of the view-wedge rule for boundary directions (cos, sin) given as (sin, cos) pairs."""
    (d0s, d0c), (d1s, d1c) = sc0, sc1
    c0 = d0c * vy - d0s * vx                                 # cross(d0, v)
    c1 = vx * d1s - vy * d1c                                 # cross(v, d1)
    if wedge_span(cfg) > PI:
        inside = ~((c0 < 0) & (c1 < 0))
    else:
        inside = (c0 >= 0) & (c1 >= 0)
    return inside, c0, c1


def wedge_span(cfg):
    fov = cfg.drone_view_range * DEG2RAD
    return (fov / float(cfg.n_rays)) * float(cfg.n_rays - 1)


def env_state(env, e):
    """Host copies (.cpu()) of the buffers env `e` of a Drone2DVecEnv is rendered from."""
    b = env.buffer
    st = {k: b(k)[e].cpu().numpy() for k in STATE_KEYS if k not in ("traj_coeff",)}
    st["traj_coeff"] = b("traj_coeff")[e].cpu().numpy() if int(env.cfg.planner) == 1 else None
    return st


def _pixels(ppc, scale):
    H = 50 * ppc
    s = scale / ppc
    x = (np.arange(H, dtype=np.float64) + 0.5) * s          # column centres (world x)
    y = (np.arange(H, dtype=np.float64) + 0.5) * s          # row centres (world y)
    return H, s, x[None, :], y[:, None]


def _disc(x, y, cx, cy, R):
    dx, dy = x - cx, y - cy
    return dx * dx + dy * dy <= R * R


def render(st, cfg, ppc, layers=ALL):
    """(frame uint8 [H, W, 3], exempt bool [H, W]) of one env.  st: dict of host arrays named like d2d_get_buffer (one env's
    rows; see STATE_KEYS); cfg: d2d_config-like (map_scale, drone_radius, drone_view_depth, drone_view_range, n_rays, n_way,
    t_way, t_way2, t_way_x2, planner)."""
    from gym_drone2d_activeperception_b200.vec_env import trajectory_waypoints
    scale = float(cfg.map_scale)
    H, s, x, y = _pixels(ppc, scale)
    img = np.full((H, H, 3), 255, dtype=np.int64)
    exempt = np.zeros((H, H), dtype=bool)
    ci = np.arange(H) // ppc                                 # cell index of a column (x) / of a row (y)
    if layers & (GROUND_TRUTH | BELIEF):
        bel = np.asarray(st["belief"], dtype=np.int64).reshape(50, 50)
        gtr = np.asarray(st["gt_rows"]).astype(np.int64).view(np.uint64).reshape(50)
        wall = ((gtr[:, None] >> np.arange(50, dtype=np.uint64)[None, :]) & np.uint64(1)).astype(np.int64)   # [i][j]
        b = bel[ci[None, :], ci[:, None]]                    # pixel (r, c) -> belief[c // ppc][r // ppc]
        w = wall[ci[None, :], ci[:, None]]
        if (layers & GROUND_TRUTH) and (layers & BELIEF):
            v = np.where(b == 0, np.where(w == 1, 64, 128), np.where(b == 1, 0, 255))
        elif layers & GROUND_TRUTH:
            v = np.where(w == 1, 0, 255)
        else:
            v = np.where(b == 0, 128, np.where(b == 1, 0, 255))
        img[:] = v[:, :, None]
    px, py = float(st["drone_x"]), float(st["drone_y"])
    if layers & VIEW:
        a0, a1 = ray_angle(cfg, float(st["drone_yaw"]), 0), ray_angle(cfg, float(st["drone_yaw"]), int(cfg.n_rays) - 1)
        vx, vy = np.broadcast_arrays(x - px, y - py)
        depth = float(cfg.drone_view_depth)
        rng = vx * vx + vy * vy <= depth * depth
        inside, c0, c1 = _wedge(cfg, sincos_cr(a0), sincos_cr(a1), vx, vy)
        zero = (vx == 0) & (vy == 0)
        m = rng & (inside | zero)
        img[m] = (3 * img[m] + np.array([255, 255, 0])) >> 2
        inside_glibc, _, _ = _wedge(cfg, (math.sin(a0), math.cos(a0)), (math.sin(a1), math.cos(a1)), vx, vy)
        nv = np.sqrt(vx * vx + vy * vy)
        edge = (np.abs(c0) <= EDGE_TOL * nv) | (np.abs(c1) <= EDGE_TOL * nv)
        exempt |= rng & ~zero & edge & (inside != inside_glibc)
    dr = float(cfg.drone_radius)
    if layers & PLAN:
        img[_disc(x, y, float(st["target_x"]), float(st["target_y"]), dr)] = (255, 0, 255)
        if int(cfg.planner) == 1 and st.get("traj_coeff") is not None:
            wp, _ = trajectory_waypoints(cfg, st["traj_coeff"], int(st["traj_nseg"]), int(st["traj_cursor"]))
            h = ppc // 4
            for wx, wy in wp:
                col, row = int(math.floor(wx * ppc / scale)), int(math.floor(wy * ppc / scale))
                r_lo, r_hi, c_lo, c_hi = max(row - h, 0), min(row + h, H - 1), max(col - h, 0), min(col + h, H - 1)
                if r_lo <= r_hi and c_lo <= c_hi:
                    img[r_lo:r_hi + 1, c_lo:c_hi + 1] = (0, 160, 0)
    if layers & TRACKERS:
        act, mu, rad = np.asarray(st["tracker_active"]), np.asarray(st["tracker_mu"]), np.asarray(st["tracker_radius"])
        for k in range(len(act)):
            if act[k]:
                R = float(rad[k])
                dx, dy = x - float(mu[k][0]), y - float(mu[k][1])
                d2 = dx * dx + dy * dy
                Ri = max(R - s, 0.0)
                img[(Ri * Ri < d2) & (d2 <= R * R)] = (255, 140, 0)
    if layers & AGENTS:
        pos, rad, hit = np.asarray(st["agent_pos"]), np.asarray(st["agent_radius"]), np.asarray(st["hit"])
        for k in range(len(rad)):
            img[_disc(x, y, float(pos[k][0]), float(pos[k][1]), float(rad[k]))] = (220, 0, 0) if hit[k] else (0, 0, 220)
    if layers & DRONE:
        img[_disc(x, y, px, py, dr)] = (0, 200, 0)
    return img.astype(np.uint8), exempt
