"""Helpers around Drone2DVecEnv.render: tile frames into one image on the device, and write a PNG with the standard library
only (no imaging package is needed).

    frames = env.render(range(16), pixels_per_cell=4)          # uint8 CUDA [16, 200, 200, 3]
    write_png("step_0042.png", montage(frames, cols=4))        # one 800 x 800 image
"""
import struct
import zlib

import numpy as np
import torch


def montage(frames, cols, pad=0, pad_value=255):
    """Tiles frames [count, H, W, 3] row-major into one frame [rows*(H+pad)-pad, cols*(W+pad)-pad, 3] with torch ops on the
    frames' device; cells past the last frame are `pad_value`."""
    if frames.dim() != 4 or frames.shape[3] != 3:
        raise ValueError("montage: expected frames [count, H, W, 3], got %s" % (tuple(frames.shape),))
    cols = int(cols)
    if cols < 1:
        raise ValueError("montage: cols must be >= 1")
    count, H, W, _ = frames.shape
    rows = max(1, -(-count // cols))
    grid = torch.full((rows * cols, H + pad, W + pad, 3), pad_value, dtype=frames.dtype, device=frames.device)
    grid[:count, :H, :W] = frames
    img = grid.view(rows, cols, H + pad, W + pad, 3).permute(0, 2, 1, 3, 4).reshape(rows * (H + pad), cols * (W + pad), 3)
    return img[:rows * (H + pad) - pad, :cols * (W + pad) - pad]


def _chunk(tag, data):
    return struct.pack(">I", len(data)) + tag + data + struct.pack(">I", zlib.crc32(tag + data) & 0xffffffff)


def encode_png(frame, level=6):
    """PNG bytes of one uint8 RGB frame [H, W, 3] (tensor on any device, or numpy array): 8-bit truecolour, filter 0."""
    a = frame.cpu().numpy() if torch.is_tensor(frame) else np.asarray(frame)
    if a.dtype != np.uint8 or a.ndim != 3 or a.shape[2] != 3:
        raise ValueError("encode_png: expected a uint8 frame [H, W, 3], got %s %s" % (a.dtype, a.shape))
    H, W = a.shape[:2]
    raw = np.zeros((H, 1 + 3 * W), dtype=np.uint8)          # each scanline starts with filter type 0 (None)
    raw[:, 1:] = a.reshape(H, 3 * W)
    return (b"\x89PNG\r\n\x1a\n" + _chunk(b"IHDR", struct.pack(">IIBBBBB", W, H, 8, 2, 0, 0, 0)) +
            _chunk(b"IDAT", zlib.compress(raw.tobytes(), level)) + _chunk(b"IEND", b""))


def write_png(path, frame, level=6):
    """Writes one uint8 RGB frame [H, W, 3] as a PNG file (zlib + struct only)."""
    with open(path, "wb") as f:
        f.write(encode_png(frame, level))
