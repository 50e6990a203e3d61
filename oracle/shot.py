"""ORACLE (test infrastructure — never imported by the product path).

Shot boundary detection as pyannote-video's `Shot` computes it (pyannote/video/structure/shot.py): per frame
RGB -> gray -> resize to (height columns x int(W*height/H) rows); per consecutive pair the Farneback optical flow
(pyr_scale 0.5, 3 levels, winsize 15, 3 iterations, poly_n 5, poly_sigma 1.1, box-filter update) and the displaced
frame difference (DFD); over the clip a zero-padded median filter, normalisation and thresholding.

Two legs:
  * `cv2_*`: the reference's own OpenCV calls (imports cv2 lazily; only the CPU tests and the golden generator use them);
  * `farneback()`: a numpy float32 restatement of OpenCV's Farneback (polynomial expansion, update matrices,
    box-filter flow update with running double sums, pyramid), written from the published algorithm
    (Farneback 2003) and OpenCV's documented behaviour.  Its intermediates (R, M, per-level flow) are what the
    GPU kernels are tested against stage by stage.  Measured |flow - cv2 flow|: DESIGN.md §5.
"""
import numpy as np

f32 = np.float32

PYR_SCALE = 0.5
LEVELS = 3
WINSIZE = 15
ITERATIONS = 3
POLY_N = 5
POLY_SIGMA = 1.1
MIN_SIZE = 32                              # levels whose size would fall below this are skipped
BORDER_W = (f32(0.14), f32(0.14), f32(0.4472), f32(0.8), f32(1.0))   # update-matrix weights of the 5 outer pixels


# ----------------------------------------------------------------------------------------------------- the reference's calls
def cv2_convert(rgb, height):
    import cv2
    h, w = rgb.shape[:2]
    return cv2.resize(cv2.cvtColor(rgb, cv2.COLOR_RGB2GRAY), (height, int(w * height / h)))


def cv2_flow(prev, cur):
    import cv2
    return cv2.calcOpticalFlowFarneback(prev, cur, None, PYR_SCALE, LEVELS, WINSIZE, ITERATIONS, POLY_N, POLY_SIGMA, 0)


def dfd(prev, cur, flow):
    """the reference's per-pixel displaced frame difference, vectorised: reconstruct[y,x] = cur[ry,rx] with
    r = int(max(0, min(p + d, size-1))).  The reference unpacks the flow vector as `dy, dx = flow[y, x]`
    while OpenCV stores (dx, dy): the column moves by the flow's y component and the row by its x component.
    Under NumPy >= 2 a Python int plus a float32 scalar stays float32, so p + d is rounded to float32."""
    h, w = prev.shape
    xs = (np.arange(w, dtype=f32)[None, :] + flow[..., 1].astype(f32)).astype(np.float64)
    ys = (np.arange(h, dtype=f32)[:, None] + flow[..., 0].astype(f32)).astype(np.float64)

    def clamp(v, hi):
        v = np.where(hi < v, float(hi), v)                    # Python min(v, hi) keeps v unless hi < v (NaN stays)
        v = np.where(v > 0, v, 0.0)                           # Python max(0, v) keeps 0 unless v > 0 (NaN -> 0)
        return v.astype(np.int64)

    rec = cur[clamp(ys, h - 1), clamp(xs, w - 1)].astype(np.float64)
    return float(np.mean(np.abs(prev.astype(np.float64) - rec)))


def reference_dfds(frames, height):
    """(gray frames, DFDs) of a uint8 [T,H,W,3] clip through the reference's calls"""
    gray = [cv2_convert(f, height) for f in frames]
    return np.stack(gray), np.array([dfd(gray[i - 1], gray[i], cv2_flow(gray[i - 1], gray[i]))
                                     for i in range(1, len(gray))])


# ----------------------------------------------------------------------------------------------------- numpy Farneback
def pyramid_sizes(h, w):
    """[(rows, cols)] from the coarsest level used down to level 0"""
    scale, k = 1.0, 0
    while k < LEVELS:
        scale *= PYR_SCALE
        if w * scale < MIN_SIZE or h * scale < MIN_SIZE:
            break
        k += 1
    out = []
    for lv in range(k, -1, -1):
        s = PYR_SCALE ** lv
        out.append((int(np.rint(h * s)), int(np.rint(w * s)), s))
    return out


def gaussian_taps(scale):
    """separable pre-blur of a pyramid level: (taps float32, radius); scale 1 -> OpenCV's fixed 3-tap [1 2 1]/4"""
    sigma = (1.0 / scale - 1.0) * 0.5
    ksize = max(int(np.rint(sigma * 5)) | 1, 3)
    if sigma <= 0:
        assert ksize == 3
        return np.array([0.25, 0.5, 0.25], f32), 1
    x = np.arange(ksize) - (ksize - 1) * 0.5
    k = np.exp(-x * x / (2 * sigma * sigma))
    return (k / k.sum()).astype(f32), ksize // 2


def _reflect101(n, r):
    idx = np.arange(-r, n + r)
    idx = np.abs(idx)
    return np.where(idx > n - 1, 2 * (n - 1) - idx, idx)


def blur(img, taps, r):
    """float32 separable filter, rows then columns, reflect-101 border, each tap product and sum rounded to float32"""
    h, w = img.shape
    src = img[:, _reflect101(w, r)]
    tmp = np.zeros((h, w), f32)
    for j in range(2 * r + 1):
        tmp = (tmp + taps[j] * src[:, j:j + w]).astype(f32)
    src = tmp[_reflect101(h, r), :]
    out = np.zeros((h, w), f32)
    for j in range(2 * r + 1):
        out = (out + taps[j] * src[j:j + h, :]).astype(f32)
    return out


def linear_taps(src, dst, zero_edges):
    """OpenCV INTER_LINEAR source indices and float weights (half-pixel centres, float32 fraction).  Along x a tap
    outside the image gets weight 0 (`zero_edges`); along y the rows are clamped and the weights kept."""
    scale = 1.0 / (dst / src)
    i0, i1, a0, a1 = [], [], [], []
    for d in range(dst):
        f = f32((d + 0.5) * scale - 0.5)
        s = int(np.floor(f))
        f = f32(f - f32(s))
        if zero_edges and s < 0:
            s, f = 0, f32(0)
        if zero_edges and s >= src - 1:
            s, f = src - 1, f32(0)
        i0.append(min(max(s, 0), src - 1))
        i1.append(min(max(s + 1, 0), src - 1))
        a0.append(f32(1) - f)
        a1.append(f)
    return np.array(i0), np.array(i1), np.array(a0, f32), np.array(a1, f32)


def resize_float(img, rows, cols):
    """float32 INTER_LINEAR resize (exact 2x downscale becomes the 2x2 mean, as OpenCV does)"""
    h, w = img.shape
    if (h, w) == (rows, cols):
        return img.copy()
    if h == 2 * rows and w == 2 * cols:
        return ((img[0::2, 0::2] + img[0::2, 1::2] + img[1::2, 0::2] + img[1::2, 1::2]) * f32(0.25)).astype(f32)
    x0, x1, ax0, ax1 = linear_taps(w, cols, True)
    y0, y1, ay0, ay1 = linear_taps(h, rows, False)
    t = (img[:, x0] * ax0 + img[:, x1] * ax1).astype(f32)
    return (t[y0] * ay0[:, None] + t[y1] * ay1[:, None]).astype(f32)


def poly_gaussian(n=POLY_N, sigma=POLY_SIGMA):
    """(g, xg, xxg float32 [2n+1], ig11, ig03, ig33, ig55 float64): the polynomial-expansion taps and the entries of
    the inverse of the 6x6 Gaussian-weighted normal matrix the expansion needs"""
    x = np.arange(-n, n + 1)
    g = np.exp(-(x * x) / (2 * sigma * sigma))
    g = (g / g.sum()).astype(f32)
    xg = (x.astype(f32) * g).astype(f32)
    xxg = ((x * x).astype(f32) * g).astype(f32)
    gg = (g[:, None] * g[None, :]).astype(f32)                 # [y, x]
    xf = x.astype(f32)[None, :]
    yf = x.astype(f32)[:, None]
    G = np.zeros((6, 6))
    G[0, 0] = gg.astype(np.float64).sum()
    G[1, 1] = (gg * xf * xf).astype(np.float64).sum()
    G[3, 3] = (gg * xf * xf * xf * xf).astype(np.float64).sum()
    G[5, 5] = (gg * xf * xf * yf * yf).astype(np.float64).sum()
    G[2, 2] = G[0, 3] = G[0, 4] = G[3, 0] = G[4, 0] = G[1, 1]
    G[4, 4] = G[3, 3]
    G[3, 4] = G[4, 3] = G[5, 5]
    iG = np.linalg.inv(G)
    return g, xg, xxg, iG[1, 1], iG[0, 3], iG[3, 3], iG[5, 5]


def poly_exp(img):
    """float32 [h,w] -> R float32 [5,h,w]: planes (y, x, xx, yy, xy) coefficients.  Columns first in float32 with
    clamped rows, then rows in float64 with replicated columns."""
    n = POLY_N
    g, xg, xxg, ig11, ig03, ig33, ig55 = poly_gaussian()
    h, w = img.shape
    r0 = (img * g[n]).astype(f32)
    r1 = np.zeros_like(r0)
    r2 = np.zeros_like(r0)
    for k in range(1, n + 1):
        up = img[np.maximum(np.arange(h) - k, 0)]
        dn = img[np.minimum(np.arange(h) + k, h - 1)]
        p = (up + dn).astype(f32)
        r0 = (r0 + (g[n + k] * p).astype(f32)).astype(f32)
        r1 = (r1 + (xg[n + k] * (dn - up).astype(f32)).astype(f32)).astype(f32)
        r2 = (r2 + (xxg[n + k] * p).astype(f32)).astype(f32)
    cols = np.clip(np.arange(-n, w + n), 0, w - 1)
    c0, c1, c2 = (r.astype(np.float64)[:, cols] for r in (r0, r1, r2))
    b1 = c0[:, n:n + w] * float(g[n])
    b3 = c1[:, n:n + w] * float(g[n])
    b5 = c2[:, n:n + w] * float(g[n])
    b2 = np.zeros((h, w))
    b4 = np.zeros((h, w))
    b6 = np.zeros((h, w))
    for k in range(1, n + 1):
        L, Rr = slice(n - k, n - k + w), slice(n + k, n + k + w)
        tg = c0[:, Rr] + c0[:, L]
        b1 = b1 + tg * float(g[n + k])
        b4 = b4 + tg * float(xxg[n + k])
        b2 = b2 + (c0[:, Rr] - c0[:, L]) * float(xg[n + k])
        b3 = b3 + (c1[:, Rr] + c1[:, L]) * float(g[n + k])
        b6 = b6 + (c1[:, Rr] - c1[:, L]) * float(xg[n + k])
        b5 = b5 + (c2[:, Rr] + c2[:, L]) * float(g[n + k])
    return np.stack([b3 * ig11, b2 * ig11, b1 * ig03 + b5 * ig33, b1 * ig03 + b4 * ig33, b6 * ig55]).astype(f32)


def update_matrices(R0, R1, flow):
    """M float32 [5,h,w] = (G11, G12, G22, h1, h2) of every pixel, R1 sampled bilinearly at x + flow"""
    _, h, w = R0.shape
    dx, dy = flow[..., 0], flow[..., 1]
    fx = (np.arange(w, dtype=f32)[None, :] + dx).astype(f32)
    fy = (np.arange(h, dtype=f32)[:, None] + dy).astype(f32)
    x1 = np.floor(fx).astype(np.int64)
    y1 = np.floor(fy).astype(np.int64)
    fx = (fx - x1.astype(f32)).astype(f32)
    fy = (fy - y1.astype(f32)).astype(f32)
    inside = (x1 >= 0) & (x1 < w) & (y1 >= 0) & (y1 < h)
    xa, ya = np.clip(x1, 0, w - 1), np.clip(y1, 0, h - 1)
    xb, yb = np.minimum(xa + 1, w - 1), np.minimum(ya + 1, h - 1)
    one = f32(1)
    a00, a01 = ((one - fx) * (one - fy)).astype(f32), (fx * (one - fy)).astype(f32)
    a10, a11 = ((one - fx) * fy).astype(f32), (fx * fy).astype(f32)

    def samp(c):
        P = R1[c]
        v = (a00 * P[ya, xa]).astype(f32)
        v = (v + (a01 * P[ya, xb]).astype(f32)).astype(f32)
        v = (v + (a10 * P[yb, xa]).astype(f32)).astype(f32)
        return (v + (a11 * P[yb, xb]).astype(f32)).astype(f32)

    half, quarter = f32(0.5), f32(0.25)
    r2 = np.where(inside, samp(0), f32(0))
    r3 = np.where(inside, samp(1), f32(0))
    r4 = np.where(inside, ((R0[2] + samp(2)) * half).astype(f32), R0[2])
    r5 = np.where(inside, ((R0[3] + samp(3)) * half).astype(f32), R0[3])
    r6 = np.where(inside, ((R0[4] + samp(4)) * quarter).astype(f32), (R0[4] * half).astype(f32))
    r2 = ((R0[0] - r2) * half).astype(f32)
    r3 = ((R0[1] - r3) * half).astype(f32)
    r2 = (r2 + ((r4 * dy).astype(f32) + (r6 * dx).astype(f32)).astype(f32)).astype(f32)
    r3 = (r3 + ((r6 * dy).astype(f32) + (r5 * dx).astype(f32)).astype(f32)).astype(f32)
    bw = np.array(BORDER_W, f32)
    # per-pixel scale = wx_left * wx_right * wy_top * wy_bottom in that order (1 where not at a border)
    sxl = np.where(np.arange(w) < 5, bw[np.minimum(np.arange(w), 4)], f32(1))
    sxr = np.where(np.arange(w) >= w - 5, bw[np.minimum(w - 1 - np.arange(w), 4)], f32(1))
    syt = np.where(np.arange(h) < 5, bw[np.minimum(np.arange(h), 4)], f32(1))
    syb = np.where(np.arange(h) >= h - 5, bw[np.minimum(h - 1 - np.arange(h), 4)], f32(1))
    scale = (((sxl[None, :] * sxr[None, :]).astype(f32) * syt[:, None]).astype(f32) * syb[:, None]).astype(f32)
    r2, r3, r4, r5, r6 = ((r * scale).astype(f32) for r in (r2, r3, r4, r5, r6))
    M = np.empty((5, h, w), f32)
    M[0] = ((r4 * r4).astype(f32) + (r6 * r6).astype(f32))
    M[1] = ((r4 + r5).astype(f32) * r6)
    M[2] = ((r5 * r5).astype(f32) + (r6 * r6).astype(f32))
    M[3] = ((r4 * r2).astype(f32) + (r6 * r3).astype(f32))
    M[4] = ((r6 * r2).astype(f32) + (r5 * r3).astype(f32))
    return M


def box_solve(M, winsize=WINSIZE):
    """flow float32 [h,w,2] from the winsize x winsize box sums of M (replicated borders).  Column sums run down the
    image as OpenCV's do (float32 difference added to a float64 running sum); row sums run along each row in float64."""
    _, h, w = M.shape
    m = winsize // 2
    Mf = M.reshape(5, h, w)
    vs = np.empty((h, 5, w))
    v = (Mf[:, 0, :] * f32(m + 2)).astype(np.float64)
    for y in range(1, m):
        v = v + Mf[:, min(y, h - 1), :]
    for y in range(h):
        v = v + (Mf[:, min(y + m, h - 1), :] - Mf[:, max(y - m - 1, 0), :]).astype(f32)
        vs[y] = v
    cols = np.clip(np.arange(-m - 1, w + m), 0, w - 1)        # vsum[-1-x] mirrors vsum[x]: replicated ends
    vp = vs[:, :, cols]                                        # index j <-> column j - m - 1
    acc = vs[:, :, 0] * (m + 2)
    for x in range(1, m):
        acc = acc + vs[:, :, min(x, w - 1)]
    scale = 1.0 / (winsize * winsize)
    flow = np.empty((h, w, 2), f32)
    for x in range(w):
        acc = acc + (vp[:, :, x + 2 * m + 1] - vp[:, :, x])
        g11, g12, g22, h1, h2 = (acc[:, c] * scale for c in range(5))
        idet = 1.0 / (g11 * g22 - g12 * g12 + 1e-3)
        flow[:, x, 0] = (g11 * h2 - g12 * h1) * idet
        flow[:, x, 1] = (g22 * h1 - g12 * h2) * idet
    return flow


def level_images(gray):
    """[(R float32 [5,rows,cols], image float32)] for each pyramid level, coarsest first"""
    h, w = gray.shape
    out = []
    img = gray.astype(f32)
    for rows, cols, s in pyramid_sizes(h, w):
        taps, r = gaussian_taps(s)
        I = resize_float(blur(img, taps, r), rows, cols)
        out.append((poly_exp(I), I))
    return out


def resize_flow(flow, rows, cols):
    f = np.stack([resize_float(flow[..., c], rows, cols) for c in range(2)], -1)
    return (f * f32(1.0 / PYR_SCALE)).astype(f32)


def farneback(prev, cur, trace=None):
    """numpy float32 Farneback flow [h,w,2] of two uint8 frames; `trace` (a list) receives per level
    dict(R0, R1, M0 (first update matrices), flow)"""
    L0, L1 = level_images(prev), level_images(cur)
    flow = None
    for (R0, _), (R1, _) in zip(L0, L1):
        _, rows, cols = R0.shape
        flow = np.zeros((rows, cols, 2), f32) if flow is None else resize_flow(flow, rows, cols)
        M = update_matrices(R0, R1, flow)
        M0 = M
        for it in range(ITERATIONS):
            flow = box_solve(M)
            if it < ITERATIONS - 1:
                M = update_matrices(R0, R1, flow)
        if trace is not None:
            trace.append(dict(R0=R0, R1=R1, M0=M0, flow=flow.copy()))
    return flow
