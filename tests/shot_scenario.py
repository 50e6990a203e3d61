"""Deterministic clips for shot boundary detection (numpy only; regenerated from their parameters by the GPU tests
and by tests/golden/make_shot_golden.py).  A clip is a list of scenes; each scene is a smooth random colour texture
(or a flat colour) seen through a window that translates by (dx, dy) pixels per frame, so consecutive frames of a
scene differ by motion and a scene change is a hard cut."""
import hashlib

import numpy as np

# name: (H, W, frames, seed, scene starts, (dx, dy) per frame, kind, height)
CLIPS = {
    "hd": (1080, 1920, 64, 1, (0, 20, 45), (6, 2), "texture", 50),
    "sd": (360, 640, 160, 2, (0, 50, 110), (2, 1), "texture", 50),
    "odd": (333, 517, 40, 3, (0, 25), (1, 1), "texture", 50),
    "h100": (360, 640, 40, 4, (0, 20), (2, 1), "texture", 100),
    "static": (120, 200, 30, 5, (0,), (0, 0), "flat", 50),
    "static_cut": (120, 200, 30, 6, (0, 15), (0, 0), "flat", 50),
    "run": (240, 320, 50, 7, (0, 20, 21, 22, 23), (1, 0), "texture", 50),
}


def _texture(rng, rows, cols, cell):
    """smooth colour texture: coarse random grid, bilinearly upsampled, plus a diagonal ramp"""
    gy, gx = rows // cell + 2, cols // cell + 2
    grid = rng.random((gy, gx, 3)) * 255.0
    y = np.arange(rows) / cell
    x = np.arange(cols) / cell
    y0, x0 = y.astype(np.int64), x.astype(np.int64)
    fy, fx = (y - y0)[:, None, None], (x - x0)[None, :, None]
    a = grid[y0][:, x0]
    b = grid[y0][:, x0 + 1]
    c = grid[y0 + 1][:, x0]
    d = grid[y0 + 1][:, x0 + 1]
    img = a * (1 - fy) * (1 - fx) + b * (1 - fy) * fx + c * fy * (1 - fx) + d * fy * fx
    ramp = (np.arange(rows)[:, None] + np.arange(cols)[None, :]) * (40.0 / (rows + cols))
    return np.clip(img * 0.8 + ramp[..., None], 0, 255).astype(np.uint8)


def make_clip(name):
    """uint8 [T,H,W,3] frames of clip `name`"""
    H, W, T, seed, starts, (dx, dy), kind, _ = CLIPS[name]
    frames = np.empty((T, H, W, 3), np.uint8)
    bounds = list(starts) + [T]
    for s in range(len(starts)):
        rng = np.random.default_rng(seed * 100 + s)
        n = bounds[s + 1] - bounds[s]
        if kind == "flat":
            frames[bounds[s]:bounds[s + 1]] = rng.integers(30, 220, 3, dtype=np.uint8)
            continue
        tex = _texture(rng, H + abs(dy) * n + 1, W + abs(dx) * n + 1, max(24, W // 16))
        for i in range(n):
            oy = i * dy if dy >= 0 else (n - 1 - i) * -dy
            ox = i * dx if dx >= 0 else (n - 1 - i) * -dx
            frames[bounds[s] + i] = tex[oy:oy + H, ox:ox + W]
    return frames


def height_of(name):
    return CLIPS[name][7]


def sha256(frames):
    return hashlib.sha256(np.ascontiguousarray(frames).tobytes()).hexdigest()


def translating(H, W, n, seed, dx=2, dy=1):
    """uint8 [n,H,W,3]: one scene of the texture above, moving by (dx, dy) >= 0 pixels per frame"""
    tex = _texture(np.random.default_rng(seed), H + dy * n + 1, W + dx * n + 1, max(24, W // 16))
    return np.stack([tex[i * dy:i * dy + H, i * dx:i * dx + W] for i in range(n)])
