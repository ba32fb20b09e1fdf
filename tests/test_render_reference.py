"""The NumPy twin of d2d_render (tests/render_reference.py) on hand-built states: disc and ring pixels against direct
enumeration of pixel centres, layer order, the cell palette, clipping at the frame edge, several pixel densities; the view
wedge against the cells the oracle's rays mark; the header's render constants against _native.  CPU only."""
import os
import shutil
import subprocess
from types import SimpleNamespace

import numpy as np
import pytest

import render_reference as rr
import util

PPCS = (1, 3, 7, 10)


def _cfg(**kw):
    d = dict(map_scale=10.0, drone_radius=10.0, drone_view_depth=80.0, drone_view_range=90.0, n_rays=50, n_way=0,
             planner=0, t_way=[], t_way2=[], t_way_x2=[])
    d.update(kw)
    return SimpleNamespace(**d)


def _state(agents=(), trackers=(), drone=(250.0, 250.0, 0.0), target=(50.0, 460.0)):
    """agents: (x, y, radius, hit); trackers: (x, y, radius)."""
    n = max(len(agents), len(trackers), 1)
    st = dict(belief=np.zeros((50, 50), np.uint8), gt_rows=np.zeros(50, np.int64),
              agent_pos=np.full((n, 2), -1e4), agent_radius=np.zeros(n), hit=np.zeros(n, np.int8),
              tracker_active=np.zeros(n, np.uint8), tracker_mu=np.zeros((n, 4)), tracker_radius=np.zeros(n),
              drone_x=drone[0], drone_y=drone[1], drone_yaw=drone[2], target_x=target[0], target_y=target[1],
              traj_coeff=None, traj_nseg=0, traj_cursor=0)
    for k, (x, y, r, h) in enumerate(agents):
        st["agent_pos"][k] = (x, y); st["agent_radius"][k] = r; st["hit"][k] = h
    for k, (x, y, r) in enumerate(trackers):
        st["tracker_active"][k] = 1; st["tracker_mu"][k, :2] = (x, y); st["tracker_radius"][k] = r
    return st


def _enumerate(ppc, inside):
    """Pixels (r, c) whose centre satisfies inside(x, y), by a plain loop over Python floats."""
    s = 10.0 / ppc
    H = 50 * ppc
    return {(r, c) for r in range(H) for c in range(H) if inside((c + 0.5) * s, (r + 0.5) * s)}


def _where(img, rgb):
    return set(zip(*np.nonzero((img == np.array(rgb, np.uint8)).all(2))))


@pytest.mark.parametrize("ppc", PPCS)
def test_disc_and_ring_pixels_match_enumeration(ppc):
    cx, cy, R = 123.4, 301.7, 15.0
    tx, ty, TR = 380.25, 90.5, 37.3
    st = _state(agents=[(cx, cy, R, 0)], trackers=[(tx, ty, TR)])
    img, ex = rr.render(st, _cfg(), ppc, rr.AGENTS | rr.TRACKERS)
    assert not ex.any()
    disc = _enumerate(ppc, lambda x, y: (x - cx) * (x - cx) + (y - cy) * (y - cy) <= R * R)
    s = 10.0 / ppc
    Ri = max(TR - s, 0.0)
    ring = _enumerate(ppc, lambda x, y: Ri * Ri < (x - tx) * (x - tx) + (y - ty) * (y - ty) <= TR * TR)
    assert _where(img, (0, 0, 220)) == disc and len(disc) > 0
    assert _where(img, (255, 140, 0)) == ring and len(ring) > 0
    assert (img.reshape(-1, 3) == 255).all(1).sum() == (50 * ppc) ** 2 - len(disc) - len(ring)


@pytest.mark.parametrize("ppc", PPCS)
def test_clipping_at_the_frame_edge(ppc):
    cx, cy, R = -4.0, 497.0, 15.0
    st = _state(agents=[(cx, cy, R, 1)], drone=(1000.0, 1000.0, 0.0))
    img, _ = rr.render(st, _cfg(), ppc, rr.AGENTS | rr.DRONE)
    want = _enumerate(ppc, lambda x, y: (x - cx) * (x - cx) + (y - cy) * (y - cy) <= R * R)
    assert _where(img, (220, 0, 0)) == want and len(want) > 0
    assert img.shape == (50 * ppc, 50 * ppc, 3)


def test_layer_order():
    # agent 1 over agent 0, the drone over both, agents over the tracker ring and the target, the ring over the view
    st = _state(agents=[(250.0, 250.0, 15.0, 1), (262.0, 250.0, 15.0, 0)], trackers=[(250.0, 250.0, 20.0)],
                drone=(255.0, 250.0, 0.0), target=(250.0, 250.0))
    img, _ = rr.render(st, _cfg(), 10, rr.ALL)
    assert tuple(img[250, 255]) == (0, 200, 0)          # drone centre
    assert tuple(img[250, 270]) == (0, 0, 220)          # only agent 1 (not seen)
    assert tuple(img[250, 236]) == (220, 0, 0)          # only agent 0 (seen)
    assert tuple(img[250, 268]) == (0, 0, 220)          # both agents: the higher index wins
    assert tuple(img[250, 230]) == (255, 140, 0)        # ring outside the agents
    img2, _ = rr.render(st, _cfg(), 10, rr.PLAN)
    assert tuple(img2[250, 240]) == (255, 0, 255)
    img3, _ = rr.render(st, _cfg(), 10, rr.PLAN | rr.AGENTS)
    assert tuple(img3[250, 240]) == (220, 0, 0)         # agent 0 only, over the target


def test_cell_palette_all_four_bit_combinations():
    st = _state(drone=(1000.0, 1000.0, 0.0))
    st["gt_rows"][3] = np.int64(1 << 7) | np.int64(1 << 8)     # walls (3, 7), (3, 8)
    st["belief"][3, 7] = 1          # seen wall
    st["belief"][3, 9] = 2          # seen free
    st["belief"][4, 7] = 1
    cells = {(3, 7): None, (3, 8): None, (3, 9): None, (4, 7): None, (5, 5): None}
    want = {
        rr.GROUND_TRUTH | rr.BELIEF: {(3, 7): 0, (3, 8): 64, (3, 9): 255, (4, 7): 0, (5, 5): 128},
        rr.GROUND_TRUTH: {(3, 7): 0, (3, 8): 0, (3, 9): 255, (4, 7): 255, (5, 5): 255},
        rr.BELIEF: {(3, 7): 0, (3, 8): 128, (3, 9): 255, (4, 7): 0, (5, 5): 128},
        0: {(3, 7): 255, (3, 8): 255, (3, 9): 255, (4, 7): 255, (5, 5): 255},
    }
    for layers, table in want.items():
        for ppc in (1, 3):
            img, _ = rr.render(st, _cfg(), ppc, layers)
            for (i, j) in cells:
                block = img[j * ppc:(j + 1) * ppc, i * ppc:(i + 1) * ppc]     # cell (i, j): columns i*ppc.., rows j*ppc..
                assert (block == table[(i, j)]).all(), (layers, ppc, i, j, block[0, 0])


def test_view_blend_and_range():
    st = _state(drone=(250.0, 250.0, 0.0))
    img, _ = rr.render(st, _cfg(drone_view_range=360.0), 10, rr.VIEW)
    inside = _enumerate(10, lambda x, y: (x - 250.0) * (x - 250.0) + (y - 250.0) * (y - 250.0) <= 6400.0)
    got = _where(img, ((3 * 255 + 255) >> 2, (3 * 255 + 255) >> 2, (3 * 255) >> 2))
    # FOV 360 with 50 rays spans 352.8 degrees: the pixels missing from the disc form the thin gap behind the drone
    assert got <= inside and 0 < len(inside - got) < 0.03 * len(inside)


@pytest.mark.parametrize("ppc", PPCS)
def test_waypoints_square_and_clip(ppc):
    # one Primitive segment whose waypoints are constants: coefficient rows (p, v, h) per axis, t tables of n_way entries
    n_way = 3
    cfg = _cfg(planner=1, n_way=n_way, t_way=[0.1, 0.2, 0.3], t_way2=[0.01, 0.04, 0.09], t_way_x2=[0.2, 0.4, 0.6])
    coeff = np.zeros((100, 6))
    coeff[0] = (3.0, 0.0, 0.0, 122.0, 0.0, 0.0)         # (3, 122): near the left edge
    coeff[1] = (250.0, 0.0, 0.0, 250.0, 0.0, 0.0)
    st = _state(drone=(1000.0, 1000.0, 0.0), target=(-1e4, -1e4))
    st.update(traj_coeff=coeff, traj_nseg=2, traj_cursor=1)
    img, _ = rr.render(st, cfg, ppc, rr.PLAN)
    h = ppc // 4
    want = set()
    for x, y in ((3.0, 122.0), (250.0, 250.0)):
        col, row = int(np.floor(x * ppc / 10.0)), int(np.floor(y * ppc / 10.0))
        want |= {(r, c) for r in range(row - h, row + h + 1) for c in range(col - h, col + h + 1)
                 if 0 <= r < 50 * ppc and 0 <= c < 50 * ppc}
    assert _where(img, (0, 160, 0)) == want


# ---------------------------------------------------------------------------------------------- wedge orientation (oracle)
@pytest.mark.parametrize("fov", [90, 180, 360])
def test_wedge_covers_the_cells_the_oracle_marks(fov):
    from gym_drone2d_activeperception_b200.params import Params
    from gym_drone2d_activeperception_b200.vec_env import make_config
    from gym_drone2d_activeperception_b200.world import generate_worlds
    B = 24
    p = Params(debug=False, planner="NoMove", gaze_method="NoControl", static_map="maps/empty_map.npy", agent_number=10,
               agent_radius=15, agent_max_speed=20, drone_view_range=fov, map_id=1)
    worlds = generate_worlds(p, 1 + np.arange(B))
    rng = np.random.RandomState(fov)
    poses = worlds["drone_pose"].copy()
    poses[:, 0] = rng.uniform(100, 400, B); poses[:, 1] = rng.uniform(100, 400, B)
    poses[:, 2] = np.where(np.arange(B) % 2 == 0, 45.0 * (np.arange(B) % 8), rng.uniform(0, 360, B))   # on / off the 45° lattice
    poses[::5, :2] = np.round(poses[::5, :2])
    ob = util.oracle_batch(p, worlds, poses)
    before = ob.gather(trackers=False)["belief"].copy()
    ob.step(np.zeros(B), auto_reset=False)
    g = ob.gather(trackers=False)
    ob.close()
    cfg = make_config(p, B, 10, 0)
    blended = np.array([(3 * 255 + 255) >> 2, (3 * 255 + 255) >> 2, (3 * 255) >> 2], np.uint8)
    checked = 0
    for e in range(B):
        st = _state(drone=(g["drone_x"][e], g["drone_y"][e], g["drone_yaw"][e]))
        img, _ = rr.render(st, cfg, 10, rr.VIEW)
        wedge = (img == blended).all(2)
        cell_has = wedge.reshape(50, 10, 50, 10).any((1, 3)).T           # [i][j]: any wedge pixel in cell (i, j)
        near = np.zeros_like(cell_has)
        padded = np.pad(cell_has, 1)
        for di in (0, 1, 2):
            for dj in (0, 1, 2):
                near |= padded[di:di + 50, dj:dj + 50]
        marked = (g["belief"][e] != before[e])
        if g["done"][e]:            # a drone placed on an agent: the episode ends before anything is seen
            continue
        checked += 1
        miss = np.argwhere(marked & ~near)
        assert len(miss) == 0, (fov, e, poses[e].tolist(), miss[:5].tolist())
        # and the wedge points the right way: most of its cells are marked (no walls in the empty map's interior)
        assert (marked & cell_has).sum() >= 0.5 * marked.sum() > 0
    assert checked >= B // 2


# ---------------------------------------------------------------------------------------------- header constants
@pytest.mark.skipif(shutil.which("gcc") is None, reason="needs a C compiler")
def test_render_constants_match_header(tmp_path):
    from gym_drone2d_activeperception_b200 import _native
    names = ["D2D_RENDER_MAX_PPC", "D2D_RENDER_MAX_LIST", "D2D_RENDER_GROUND_TRUTH", "D2D_RENDER_BELIEF", "D2D_RENDER_VIEW",
             "D2D_RENDER_PLAN", "D2D_RENDER_TRACKERS", "D2D_RENDER_AGENTS", "D2D_RENDER_DRONE", "D2D_RENDER_ALL"]
    src = tmp_path / "consts.c"
    src.write_text("#include <stdio.h>\n#include \"drone2d.h\"\nint main(void) {\n" +
                   "".join("    printf(\"%%d\\n\", (int)%s);\n" % n for n in names) + "    return 0;\n}\n")
    exe = str(tmp_path / "consts")
    subprocess.run(["gcc", "-Wall", "-Werror", "-I", os.path.join(util.ROOT, "include"), str(src), "-o", exe], check=True)
    got = [int(x) for x in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [getattr(_native, n[4:]) for n in names]
    assert sum(_native.RENDER_LAYERS.values()) == _native.RENDER_ALL
    for k, v in _native.RENDER_LAYERS.items():
        assert v == getattr(rr, k.upper())


# ---------------------------------------------------------------------------------------------- montage / PNG (render.py)
def test_montage_and_png_round_trip(tmp_path):
    import struct
    import zlib
    torch = pytest.importorskip("torch")
    from gym_drone2d_activeperception_b200.render import montage, write_png
    frames = torch.arange(5 * 4 * 6 * 3, dtype=torch.int64).remainder(251).to(torch.uint8).view(5, 4, 6, 3)
    img = montage(frames, cols=2)
    assert img.shape == (12, 12, 3)
    for k in range(5):
        r, c = divmod(k, 2)
        assert torch.equal(img[4 * r:4 * r + 4, 6 * c:6 * c + 6], frames[k])
    assert (img[8:, 6:] == 255).all()
    path = tmp_path / "m.png"
    write_png(str(path), img)
    data = path.read_bytes()
    assert data[:8] == b"\x89PNG\r\n\x1a\n"
    w, h, depth, ctype = struct.unpack(">IIBB", data[16:26])
    assert (w, h, depth, ctype) == (12, 12, 8, 2)
    pos, idat = 8, b""
    while pos < len(data):
        n, tag = struct.unpack(">I4s", data[pos:pos + 8])
        body = data[pos + 8:pos + 8 + n]
        assert struct.unpack(">I", data[pos + 8 + n:pos + 12 + n])[0] == zlib.crc32(tag + body) & 0xffffffff
        if tag == b"IDAT":
            idat += body
        pos += 12 + n
    raw = np.frombuffer(zlib.decompress(idat), np.uint8).reshape(12, 1 + 36)
    assert (raw[:, 0] == 0).all() and np.array_equal(raw[:, 1:].reshape(12, 12, 3), img.numpy())


def test_sincos_is_correctly_rounded():
    import math
    mpmath = pytest.importorskip("mpmath")
    mpmath.mp.prec = 200
    rng = np.random.RandomState(5)
    angles = list(rng.uniform(0, 2 * math.pi, 2000)) + [rr.ray_angle(_cfg(), yaw, 0) for yaw in range(0, 360, 45)]
    for a in angles:
        s, c = rr.sincos_cr(float(a))
        assert s == float(mpmath.sin(mpmath.mpf(float(a)))) and c == float(mpmath.cos(mpmath.mpf(float(a)))), a


@pytest.mark.parametrize("ppc", PPCS)
def test_lattice_pose_boundary_pixels_are_decided_not_exempt(ppc):
    # drone on the integer lattice, yaw 270, FOV 90: ray 0 points along the 45-degree diagonal, so the pixel centres of the
    # diagonal lie on that boundary; their side is decided by the correctly rounded sin / cos, the same as the device's
    st = _state(drone=(50.0, 50.0, 270.0))
    img, ex = rr.render(st, _cfg(), ppc, rr.VIEW)
    assert not ex.any()
    s, c = rr.sincos_cr(rr.ray_angle(_cfg(), 270.0, 0))
    blended = (img == np.array([(3 * 255 + 255) >> 2, (3 * 255 + 255) >> 2, (3 * 255) >> 2], np.uint8)).all(2)
    k = (50 * ppc) // 10 + 3            # a diagonal pixel (row == col) ahead of the drone, within the view depth
    assert blended[k, k] == (c * 1.0 - s * 1.0 >= 0)
