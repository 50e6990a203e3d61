"""Deterministic clips for shot threading (numpy only; regenerated from their parameters by the GPU tests and by
tests/golden/make_thread_golden.py, which stores only their sha256).  A scene is a random mosaic of flat colour
blocks (corners everywhere, so FAST finds plenty of points); a shot shows its scene through a window shifted by a
few pixels, so two shots of one scene share most of their ORB features while different scenes share almost none."""
import hashlib

import numpy as np

FPS = 25.0
# name: (H, W, seed, lookahead, shots as (scene, frames, dx, dy); scene -1 is a flat grey frame)
CLIPS = {
    # recurring scenes through shifted windows, with a short first shot whose end - collar falls before t = 0
    "abab": (180, 320, 1, 5, [(0, 6, 0, 0), (1, 24, 3, 2), (0, 24, 6, 1), (1, 24, 0, 4), (2, 24, 2, 2), (0, 24, 4, 3)]),
    # over-segmented: one scene cut in three touching shots, then a new scene, a flat shot and a 4-frame shot
    "overseg": (180, 320, 2, 5, [(0, 24, 0, 0), (0, 24, 2, 1), (0, 24, 4, 2), (1, 24, 1, 1), (-1, 24, 0, 0),
                                 (1, 4, 3, 0), (2, 24, 0, 0)]),
    # a recurrence farther apart than lookahead (must not link), more shots than lookahead
    "far": (160, 288, 3, 3, [(0, 24, 0, 0), (1, 24, 0, 0), (2, 24, 0, 0), (3, 24, 0, 0), (4, 24, 0, 0),
                             (0, 24, 3, 3), (1, 24, 2, 2), (5, 24, 0, 0)]),
    # 1080p: A B A
    "hd": (1080, 1920, 4, 5, [(0, 12, 0, 0), (1, 12, 0, 0), (0, 12, 9, 6)]),
}
PAD = 16


def _mosaic(rng, rows, cols):
    img = np.empty((rows, cols, 3), np.uint8)
    img[...] = rng.integers(0, 256, 3, dtype=np.uint8)
    cell = max(8, min(rows, cols) // 12)
    for _ in range(rows * cols // (cell * cell) * 3):
        h, w = rng.integers(cell // 2, 2 * cell, 2)
        y, x = rng.integers(0, rows), rng.integers(0, cols)
        img[y:y + h, x:x + w] = rng.integers(0, 256, 3, dtype=np.uint8)
    return img


def make_clip(name):
    """(uint8 [T,H,W,3] frames, [(start, end)] shot segments in seconds) of clip `name`"""
    H, W, seed, _, shots = CLIPS[name]
    scenes = {}
    frames, segments, t = [], [], 0
    for scene, n, dx, dy in shots:
        if scene < 0:
            frames.append(np.full((n, H, W, 3), 128, np.uint8))
        else:
            if scene not in scenes:
                scenes[scene] = _mosaic(np.random.default_rng(seed * 100 + scene), H + PAD, W + PAD)
            frames.append(np.repeat(scenes[scene][None, dy:dy + H, dx:dx + W], n, axis=0))
        segments.append((t / FPS, (t + n) / FPS))
        t += n
    return np.concatenate(frames), segments


def lookahead_of(name):
    return CLIPS[name][3]


def sha256(frames):
    return hashlib.sha256(np.ascontiguousarray(frames).tobytes()).hexdigest()
