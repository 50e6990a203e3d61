"""Oracle for shot threading (pyannote/video/structure/thread.py): the reference's cv2 calls, and numpy restatements
of the ORB stages cv2 does not expose one by one (FAST scores with non-max suppression, retain-best with ties, Harris
responses at given points, intensity-centroid angles, rBRIEF with the recovered pattern) plus the exact Hamming 2-NN
ratio count.  The restatements are pinned against cv2 on CPU (tests/test_thread_cpu.py); the GPU kernels
(csrc/orb.cu) follow them operation for operation.

cv2 4.13 `ORB_create()` defaults: 500 features, scale factor 1.2, 8 levels, edge threshold 31, first level 0,
WTA_K 2, Harris score, patch size 31, FAST threshold 20.
"""
import os

import cv2
import numpy as np

N_FEATURES = 500
SCALE_FACTOR = float(np.float32(1.2))               # ORB_create takes a float; levels use it as a double
N_LEVELS = 8
EDGE = 31
PATCH = 31
HALF_PATCH = PATCH // 2
FAST_T = 20
HARRIS_K = np.float32(0.04)
HARRIS_BLOCK = 7
RATIO = 0.7
f32 = np.float32

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PATTERN_H = os.path.join(ROOT, "pyannote_video_b200", "csrc", "orb_pattern.cuh")

# FAST-9/16 circle (x, y), in OpenCV's order; an arc is 9 consecutive entries (wrapping)
CIRCLE = ((0, 3), (1, 3), (2, 2), (3, 1), (3, 0), (3, -1), (2, -2), (1, -3),
          (0, -3), (-1, -3), (-2, -2), (-3, -1), (-3, 0), (-3, 1), (-2, 2), (-1, 3))


# ----------------------------------------------------------------------------------------------------- reference calls
def resize_dsize(frame_size, height):
    """the reference's cv2.resize dsize (width, height) = (height, int(w * height / h)) for a (w, h) video"""
    w, h = frame_size
    return int(height), int(w * height / h)


def cv2_gray(rgb, dsize):
    """Thread._compute_orb's preprocessing: resize the RGB frame, then convert to gray"""
    return cv2.cvtColor(cv2.resize(rgb, dsize), cv2.COLOR_RGB2GRAY)


def kp_array(kps):
    """float64 [n, 5]: x, y, octave, response, angle (float32 values widened)"""
    return np.array([[k.pt[0], k.pt[1], k.octave, k.response, k.angle] for k in kps], np.float64).reshape(-1, 5)


def cv2_orb(gray):
    """(keypoints [n,5], descriptors uint8 [n,32]) of cv2.ORB_create().detectAndCompute"""
    kps, desc = cv2.ORB_create().detectAndCompute(gray, None)
    return kp_array(kps), (desc if desc is not None else np.zeros((0, 32), np.uint8))


def cv2_bf_count(q, t):
    """BFMatcher(NORM_HAMMING).knnMatch(k=2) + the reference's ratio test; 0 when a side has < 2 descriptors"""
    if q is None or t is None or len(q) < 2 or len(t) < 2:
        return 0
    m = cv2.BFMatcher(cv2.NORM_HAMMING).knnMatch(q, t, k=2)
    return sum(1 for p in m if len(p) == 2 and p[0].distance < RATIO * p[1].distance)


# ----------------------------------------------------------------------------------------------------- geometry
def cv_round(v):
    return int(np.rint(v))                                    # round half to even, as cvRound


def level_scales():
    """float32 level scales: getScale returns (float)pow(scaleFactor, level)"""
    return [f32(SCALE_FACTOR ** k) for k in range(N_LEVELS)]


def level_sizes(rows, cols):
    """[(rows, cols)] of the ORB pyramid: cvRound(size / scale), an int divided by a float, so in float32"""
    return [(cv_round(f32(rows) / s), cv_round(f32(cols) / s)) for s in level_scales()]


def level_quotas(n=N_FEATURES):
    """features per level: cvRound of a geometric series in float32, the last level takes the remainder"""
    factor = f32(1.0 / SCALE_FACTOR)
    per = f32(n * (f32(1) - factor) / (f32(1) - f32(np.float64(factor) ** N_LEVELS)))
    out = []
    for _ in range(N_LEVELS - 1):
        out.append(cv_round(per))
        per = f32(per * factor)
    out.append(max(n - sum(out), 0))
    return out


def pyramid(gray):
    """uint8 level images; level k is resized from level k - 1 with INTER_LINEAR_EXACT"""
    levels = [gray]
    for r, c in level_sizes(*gray.shape)[1:]:
        levels.append(cv2.resize(levels[-1], (c, r), interpolation=cv2.INTER_LINEAR_EXACT))
    return levels


def umax():
    """row half-widths of the radius-15 circular patch (OpenCV's symmetric construction)"""
    hp = HALF_PATCH
    u = [0] * (hp + 2)
    vmax = int(np.floor(hp * np.sqrt(f32(2)) / 2 + 1))
    vmin = int(np.ceil(hp * np.sqrt(f32(2)) / 2))
    for v in range(vmax + 1):
        u[v] = cv_round(hp * np.sqrt(1 - v * v / float(hp * hp)))
    v0 = 0
    for v in range(hp, vmin - 1, -1):
        while u[v0] == u[v0 + 1]:
            v0 += 1
        u[v] = v0
        v0 += 1
    return u[:hp + 1]


# ----------------------------------------------------------------------------------------------------- FAST
def fast_scores(img, t=FAST_T):
    """int32 map: the FAST-9/16 corner score (the largest threshold at which the pixel is still a corner, minus 1)
    where the pixel is a corner at threshold t, else 0; pixels within 3 of the edge are 0"""
    img = img.astype(np.int32)
    R, C = img.shape
    out = np.zeros((R, C), np.int32)
    if R < 7 or C < 7:
        return out
    c = img[3:R - 3, 3:C - 3]
    d = np.stack([c - img[3 + dy:R - 3 + dy, 3 + dx:C - 3 + dx] for dx, dy in CIRCLE])      # v - ring
    ring = np.concatenate([d, d[:8]])
    arc_min = np.stack([ring[k:k + 9].min(0) for k in range(16)]).max(0)                  # darker ring: d > 0
    arc_max = np.stack([ring[k:k + 9].max(0) for k in range(16)]).min(0)                  # brighter ring: d < 0
    best = np.maximum(arc_min, -arc_max)
    score = np.maximum(best, t) - 1
    out[3:R - 3, 3:C - 3] = np.where(best > t, score, 0)
    return out


def fast_keypoints(img, t=FAST_T):
    """(x, y, score) int arrays of FAST corners surviving 3 x 3 non-max suppression (strictly greater than all
    8 neighbours), as cv2.FastFeatureDetector_create(t, True, TYPE_9_16)"""
    s = fast_scores(img, t)
    p = np.pad(s, 1)
    R, C = s.shape
    keep = s > 0
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            if dx or dy:
                keep &= s > p[1 + dy:1 + dy + R, 1 + dx:1 + dx + C]
    y, x = np.nonzero(keep)
    return x, y, s[y, x]


def retain_best(score, n):
    """mask of cv2.KeyPointsFilter.retainBest: every point whose score reaches the n-th best (ties kept)"""
    score = np.asarray(score)
    if len(score) <= n:
        return np.ones(len(score), bool)
    if n == 0:
        return np.zeros(len(score), bool)
    cut = np.sort(score)[::-1][n - 1]
    return score >= cut


# ----------------------------------------------------------------------------------------------------- Harris / angle
def harris(img, xs, ys):
    """float32 Harris responses at integer points: integer Sobel over the 7 x 7 block, then cv2's float32 formula"""
    img = img.astype(np.int32)
    r = HARRIS_BLOCK // 2
    out = np.empty(len(xs), f32)
    scale = f32(1.0) / f32(4 * HARRIS_BLOCK * 255.0)
    s4 = f32(f32(f32(scale * scale) * scale) * scale)
    for i, (x, y) in enumerate(zip(xs, ys)):
        P = img[y - r - 1:y + r + 2, x - r - 1:x + r + 2]
        Ix = (P[1:-1, 2:] - P[1:-1, :-2]) * 2 + (P[:-2, 2:] - P[:-2, :-2]) + (P[2:, 2:] - P[2:, :-2])
        Iy = (P[2:, 1:-1] - P[:-2, 1:-1]) * 2 + (P[2:, :-2] - P[:-2, :-2]) + (P[2:, 2:] - P[:-2, 2:])
        a, b, c = f32((Ix * Ix).sum()), f32((Iy * Iy).sum()), f32((Ix * Iy).sum())
        ab = f32(a + b)
        v = f32(f32(a * b) - f32(c * c))
        v = f32(v - f32(f32(HARRIS_K * ab) * ab))
        out[i] = f32(v * s4)
    return out


_P1 = f32(0.9997878412794807 * f32(180 / np.pi))
_P3 = f32(-0.3258083974640975 * f32(180 / np.pi))
_P5 = f32(0.1555786518463281 * f32(180 / np.pi))
_P7 = f32(-0.04432655554792128 * f32(180 / np.pi))
_EPS = f32(np.finfo(np.float64).eps)


def fast_atan2(y, x):
    """cv2.fastAtan2 in float32, degrees in [0, 360)"""
    y, x = f32(y), f32(x)
    ax, ay = abs(x), abs(y)
    if ax >= ay:
        c = f32(ay / f32(ax + _EPS))
    else:
        c = f32(ax / f32(ay + _EPS))
    c2 = f32(c * c)
    a = f32(f32(f32(f32(f32(f32(f32(_P7 * c2) + _P5) * c2) + _P3) * c2) + _P1) * c)
    if not ax >= ay:
        a = f32(f32(90) - a)
    if x < 0:
        a = f32(f32(180) - a)
    if y < 0:
        a = f32(f32(360) - a)
    return a


def moments(img, x, y):
    """(m01, m10) intensity moments over the radius-15 circular patch centred on integer (x, y)"""
    u = umax()
    m01 = m10 = 0
    img = img.astype(np.int64)
    for v in range(-HALF_PATCH, HALF_PATCH + 1):
        d = u[abs(v)]
        row = img[y + v, x - d:x + d + 1]
        m10 += int((np.arange(-d, d + 1) * row).sum())
        m01 += v * int(row.sum())
    return m01, m10


def ic_angle(img, x, y):
    m01, m10 = moments(img, x, y)
    return fast_atan2(f32(m01), f32(m10))


# ----------------------------------------------------------------------------------------------------- rBRIEF
def orb_blur(img):
    """ORB's 7 x 7, sigma 2 smoothing of a level: float32 separable Gaussian, rounded to uint8 (reflect-101)"""
    k = cv2.getGaussianKernel(7, 2, cv2.CV_32F)
    return cv2.sepFilter2D(img, -1, k, k, borderType=cv2.BORDER_REFLECT_101)


def pattern():
    """int32 [256, 4]: (x0, y0, x1, y1) of every test, from the generated csrc/orb_pattern.cuh"""
    import re
    body = open(PATTERN_H).read().split("{", 1)[1].split("}", 1)[0]
    return np.array([int(v) for v in re.findall(r"-?\d+", body)], np.int32).reshape(256, 4)


_DEG2RAD = f32(np.pi / f32(180.0))


def brief(blurred, cx, cy, angle, pat=None):
    """32-byte rBRIEF descriptor at the integer level centre (cx, cy) for a float32 angle in degrees"""
    pat = pattern() if pat is None else pat
    a_rad = f32(f32(angle) * _DEG2RAD)
    ca, sa = f32(np.cos(np.float64(a_rad))), f32(np.sin(np.float64(a_rad)))
    px = pat[:, [0, 2]].astype(f32)
    py = pat[:, [1, 3]].astype(f32)
    x = (px * ca).astype(f32) - (py * sa).astype(f32)
    y = (px * sa).astype(f32) + (py * ca).astype(f32)
    ix, iy = np.rint(x).astype(np.int64), np.rint(y).astype(np.int64)
    v = blurred[cy + iy, cx + ix].astype(np.int32)
    bits = (v[:, 0] < v[:, 1]).astype(np.uint8)
    return np.packbits(bits, bitorder="little")


# ----------------------------------------------------------------------------------------------------- whole ORB
def orb(gray, n_features=N_FEATURES):
    """(keypoints [n,5], descriptors [n,32]) restating cv2.ORB_create().detectAndCompute, in level order"""
    levels = pyramid(gray)
    quotas = level_quotas(n_features)
    pat = pattern()
    kps, descs = [], []
    for lv, img in enumerate(levels):
        R, C = img.shape
        if R <= 2 * EDGE or C <= 2 * EDGE:
            continue
        x, y, s = fast_keypoints(img)
        inside = (x >= EDGE) & (x < C - EDGE) & (y >= EDGE) & (y < R - EDGE)
        x, y, s = x[inside], y[inside], s[inside]
        keep = retain_best(s, 2 * quotas[lv])
        x, y = x[keep], y[keep]
        h = harris(img, x, y)
        keep = retain_best(h, quotas[lv])
        x, y, h = x[keep], y[keep], h[keep]
        blurred = orb_blur(img)
        scale = f32(SCALE_FACTOR ** lv)
        for xi, yi, hi in zip(x, y, h):
            a = ic_angle(img, xi, yi)
            kps.append([f32(f32(xi) * scale), f32(f32(yi) * scale), lv, hi, a])
            descs.append(brief(blurred, xi, yi, a, pat))
    return np.array(kps, np.float64).reshape(-1, 5), np.array(descs, np.uint8).reshape(-1, 32)


# ----------------------------------------------------------------------------------------------------- matching
def popcount_distances(q, t):
    """int32 [nq, nt] Hamming distances of uint8 [n, 32] descriptor sets"""
    x = np.bitwise_xor(q[:, None, :], t[None, :, :])
    return np.unpackbits(x, axis=2).sum(2).astype(np.int32)


def match_count(q, t):
    """exact 2-NN ratio count: queries whose best distance < 0.7 * second best (float64); 0 if a side has < 2"""
    if len(q) < 2 or len(t) < 2:
        return 0
    d = np.sort(popcount_distances(q, t), axis=1)
    return int(np.count_nonzero(d[:, 0].astype(np.float64) < RATIO * d[:, 1].astype(np.float64)))


def as_set(kps, desc):
    """set of (x, y, octave, response, angle, descriptor bytes) rows for order-free comparison"""
    return set(tuple(k) + (bytes(d),) for k, d in zip(kps.tolist(), desc))


# ----------------------------------------------------------------------------------------------------- exact resize
def linear_exact_taps(src, dst):
    """(offset, c1) per destination index of cv2's INTER_LINEAR_EXACT: fval = src/dst * (d + 0.5) - 0.5 in double,
    c1 = cvRound(frac * 256), c0 = 256 - c1.  Downscales by < 2 never reach the replicated borders; other geometries
    are refused."""
    scale = 1.0 / (dst / src)
    ofs, c1 = [], []
    for d in range(dst):
        f = scale * (d + 0.5) - 0.5
        i = int(np.floor(f))
        if i < 0 or i >= src - 1:
            raise ValueError("INTER_LINEAR_EXACT border taps (%d -> %d) are not supported" % (src, dst))
        ofs.append(i)
        c1.append(cv_round((f - i) * 256))
    return np.array(ofs, np.int32), np.array(c1, np.int32)


def resize_exact(img, rows, cols):
    """numpy restatement of cv2.resize(img, (cols, rows), interpolation=INTER_LINEAR_EXACT) for uint8 downscales:
    8-bit fixed-point horizontal pass, then vertical pass rounded from 16 fractional bits"""
    xo, xc = linear_exact_taps(img.shape[1], cols)
    yo, yc = linear_exact_taps(img.shape[0], rows)
    s = img.astype(np.int64)
    h = s[:, xo] * (256 - xc) + s[:, xo + 1] * xc
    v = h[yo] * (256 - yc)[:, None] + h[yo + 1] * yc[:, None]
    return ((v + (1 << 15)) >> 16).astype(np.uint8)


def orb_blur_restated(img):
    """orb_blur in float32: horizontal taps accumulated in order with fused multiply-adds, vertical taps folded
    symmetrically (centre first, then the pairs 1, 2, 3 apart) with fused multiply-adds, rounded half to even"""
    k = cv2.getGaussianKernel(7, 2, cv2.CV_32F).ravel()

    def fma(a, b, c):
        return (a.astype(np.float64) * np.float64(b) + c.astype(np.float64)).astype(f32)

    P = np.pad(img, 3, mode="reflect").astype(f32)
    R, C = img.shape
    row = (P[:, 0:C] * k[0]).astype(f32)
    for j in range(1, 7):
        row = fma(P[:, j:j + C], k[j], row)
    col = (row[3:3 + R] * k[3]).astype(f32)
    for j in (1, 2, 3):
        col = fma((row[3 - j:3 - j + R] + row[3 + j:3 + j + R]).astype(f32), k[3 - j], col)
    return np.clip(np.rint(col), 0, 255).astype(np.uint8)
