"""Shot boundary detection on the GPU — a drop-in for pyannote.video.Shot (pyannote/video/structure/shot.py).

Per frame: RGB -> gray -> resize to `height` columns x int(W * height / H) rows (the reference passes
(height, int(w * height / h)) to cv2.resize, which reads it as (width, height)).  Per consecutive pair: Farneback
optical flow and the displaced frame difference (DFD).  Over the clip: a zero-padded median filter of the DFDs,
normalisation (y - filtered) / filtered and thresholding; a run of consecutive over-threshold pairs keeps only its
first one.  The per-frame and per-pair work runs in csrc/shot.cu, many frames per launch; this module builds the
geometry and tables, carries the last frame of a batch into the next and does the (tiny) per-clip arithmetic.
"""
import ctypes as C

import numpy as np

from .annotation import Segment

PYR_SCALE = 0.5
LEVELS = 3
MIN_SIZE = 32
POLY_N = 5
POLY_SIGMA = 1.1
MAX_LEVELS = 4
MAX_TAPS = 19
f32 = np.float32


class PvShotLevel(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("rows", "cols", "r_off", "radius", "area2x", "dn_off", "up_off")] \
        + [("taps", C.c_float * MAX_TAPS)]


class PvShotGeo(C.Structure):
    _fields_ = [("h", C.c_int32), ("w", C.c_int32), ("n_levels", C.c_int32), ("r_stride", C.c_int32),
                ("lv", PvShotLevel * MAX_LEVELS),
                ("pg", C.c_float * (2 * POLY_N + 1)), ("pxg", C.c_float * (2 * POLY_N + 1)),
                ("pxxg", C.c_float * (2 * POLY_N + 1)), ("pad_", C.c_int32),
                ("ig11", C.c_double), ("ig03", C.c_double), ("ig33", C.c_double), ("ig55", C.c_double)]


# ----------------------------------------------------------------------------------------------------- clip arithmetic
def resize_shape(frame_size, height):
    """(rows, cols) of the resized gray frame for a (width, height) video: cv2.resize(gray, (height, int(w*height/h)))"""
    w, h = frame_size
    return int(w * height / h), int(height)


def kernel_size(context, step):
    """median filter length: the odd number around context / step, at least 3"""
    return max(3, int(np.ceil(context / step) // 2 * 2 + 1))


def medfilt(y, k):
    """scipy.signal.medfilt(y, k) for 1-D input: window median with zero padding at both ends"""
    y = np.asarray(y, dtype=np.float64)
    if y.size == 0:
        return y.copy()
    p = np.concatenate([np.zeros(k // 2), y, np.zeros(k // 2)])
    return np.median(np.lib.stride_tricks.sliding_window_view(p, k), axis=-1)


def segments(t, y, k, threshold, start, end):
    """shot segments from pair times t and DFDs y.  Index 0 is the pair of the first two frames; the run tracker
    starts at index 0, so an over-threshold index 1 is never a boundary (as in the reference).  0 / 0 gives NaN (never
    a boundary), x / 0 gives inf (always one).  Without any pair the whole video is one segment."""
    previous = start
    if len(y):
        y = np.asarray(y, dtype=np.float64)
        filtered = medfilt(y, k)
        with np.errstate(divide="ignore", invalid="ignore"):
            normalized = (y - filtered) / filtered
        last = 0
        for i in np.where(normalized > threshold)[0]:
            if i == last + 1:
                last = i
                continue
            yield Segment(previous, t[i])
            previous = t[i]
            last = i
    tail = Segment(previous, end)
    if tail:
        yield tail


# ----------------------------------------------------------------------------------------------------- geometry / tables
def _linear_taps(src, dst, zero_edges):
    """INTER_LINEAR source indices and float32 weights (half-pixel centres); along x a tap outside the image gets
    weight 0, along y rows are clamped"""
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


def gray_table(frame_size, rows, cols):
    """int32 [4*cols + 4*rows]: x0 x1 cx0 cx1 then y0 y1 cy0 cy1, weights in 11-bit fixed point (round to nearest)"""
    W, H = frame_size
    out = []
    for src, dst, zero in ((W, cols, True), (H, rows, False)):
        i0, i1, a0, a1 = _linear_taps(src, dst, zero)
        c0 = np.rint((a0 * f32(2048)).astype(f32)).astype(np.int32)
        c1 = np.rint((a1 * f32(2048)).astype(f32)).astype(np.int32)
        out += [i0.astype(np.int32), i1.astype(np.int32), c0, c1]
    return np.concatenate(out)


def _lin_table(src_rows, src_cols, rows, cols):
    x0, x1, ax0, ax1 = _linear_taps(src_cols, cols, True)
    y0, y1, ay0, ay1 = _linear_taps(src_rows, rows, False)
    return np.concatenate([x0.astype(f32), x1.astype(f32), ax0, ax1, y0.astype(f32), y1.astype(f32), ay0, ay1])


def pyramid_sizes(rows, cols):
    """[(rows, cols, scale)] of the Farneback levels used, coarsest first (levels below 32 pixels are skipped)"""
    scale, k = 1.0, 0
    while k < LEVELS:
        scale *= PYR_SCALE
        if cols * scale < MIN_SIZE or rows * scale < MIN_SIZE:
            break
        k += 1
    return [(int(np.rint(rows * PYR_SCALE ** lv)), int(np.rint(cols * PYR_SCALE ** lv)), PYR_SCALE ** lv)
            for lv in range(k, -1, -1)]


def _blur_taps(scale):
    sigma = (1.0 / scale - 1.0) * 0.5
    ksize = max(int(np.rint(sigma * 5)) | 1, 3)
    if sigma <= 0:
        return np.array([0.25, 0.5, 0.25], f32)             # OpenCV's fixed 3-tap kernel for sigma 0
    x = np.arange(ksize) - (ksize - 1) * 0.5
    k = np.exp(-x * x / (2 * sigma * sigma))
    return (k / k.sum()).astype(f32)


def _poly_constants(n=POLY_N, sigma=POLY_SIGMA):
    x = np.arange(-n, n + 1)
    g = np.exp(-(x * x) / (2 * sigma * sigma))
    g = (g / g.sum()).astype(f32)
    xg = (x.astype(f32) * g).astype(f32)
    xxg = ((x * x).astype(f32) * g).astype(f32)
    gg = (g[:, None] * g[None, :]).astype(f32)
    xf, yf = x.astype(f32)[None, :], x.astype(f32)[:, None]
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


def make_geometry(rows, cols):
    """(PvShotGeo, float32 table) of the Farneback pyramid of a rows x cols gray frame"""
    geo = PvShotGeo()
    geo.h, geo.w = rows, cols
    sizes = pyramid_sizes(rows, cols)
    geo.n_levels = len(sizes)
    tab, r_off = [], 0
    tab_len = 0
    prev = None
    for k, (lr, lc, s) in enumerate(sizes):
        L = geo.lv[k]
        L.rows, L.cols, L.r_off = lr, lc, r_off
        taps = _blur_taps(s)
        L.radius = len(taps) // 2
        for j, v in enumerate(taps):
            L.taps[j] = float(v)
        L.area2x = int(rows == 2 * lr and cols == 2 * lc)
        L.dn_off = L.up_off = -1
        if (lr, lc) != (rows, cols) and not L.area2x:
            t = _lin_table(rows, cols, lr, lc)
            L.dn_off, tab_len = tab_len, tab_len + t.size
            tab.append(t)
        if prev is not None:
            t = _lin_table(prev[0], prev[1], lr, lc)
            L.up_off, tab_len = tab_len, tab_len + t.size
            tab.append(t)
        prev = (lr, lc)
        r_off += 5 * lr * lc
    geo.r_stride = r_off
    g, xg, xxg, geo.ig11, geo.ig03, geo.ig33, geo.ig55 = _poly_constants()
    for j in range(2 * POLY_N + 1):
        geo.pg[j], geo.pxg[j], geo.pxxg[j] = float(g[j]), float(xg[j]), float(xxg[j])
    tab = np.concatenate(tab) if tab else np.zeros(1, f32)
    return geo, tab.astype(f32)


# ----------------------------------------------------------------------------------------------------- device level
class ShotDetector(object):
    """DFDs of consecutive frames already on the GPU.  `dfd_batch(frames)` takes uint8 [B,H,W,3] device frames (the
    tensors `Face` uploads) and returns the float64 DFDs of the pairs they complete: B of them, or B - 1 for the first
    batch.  The last frame of a batch (its gray image and its polynomial expansion) is carried into the next one, so
    the DFDs do not depend on how a clip is cut into batches.  Frames must be on the detector's device; every launch
    runs on that device's current stream, whatever the caller's current device is."""

    def __init__(self, frame_size, height=50, device=None, keep_flow=False):
        import torch
        if not torch.cuda.is_available():
            raise RuntimeError("pyannote_video_b200.Shot needs a CUDA device (B200); there is no CPU fallback")
        from . import _lib
        self._L = _lib
        dev = torch.device(device) if device is not None else torch.device("cuda")
        if dev.type != "cuda":
            raise RuntimeError("ShotDetector runs on a CUDA device, got %s" % dev)
        self.device = dev if dev.index is not None else torch.device("cuda", torch.cuda.current_device())
        self.frame_size = (int(frame_size[0]), int(frame_size[1]))
        self.rows, self.cols = resize_shape(self.frame_size, height)
        if self.rows < 1 or self.cols < 1:
            raise ValueError("resized frame would be empty: %r at height %d" % (self.frame_size, height))
        self.geo, tab = make_geometry(self.rows, self.cols)
        lib = _lib.lib()
        lib.pv_shot_polyexp_work_floats.restype = C.c_int64
        lib.pv_shot_flow_work_floats.restype = C.c_int64
        self._poly_wf = int(lib.pv_shot_polyexp_work_floats(C.byref(self.geo)))
        self._flow_wf = int(lib.pv_shot_flow_work_floats(C.byref(self.geo)))
        self._smem = 226 * 1024
        with torch.cuda.device(self.device):
            self.tab = torch.from_numpy(tab).to(self.device)
            self.gtab = torch.from_numpy(gray_table(self.frame_size, self.rows, self.cols)).to(self.device)
        self.keep_flow = keep_flow
        self.flow = None
        self._cap = 0
        self._has_prev = False

    def reset(self):
        self._has_prev = False

    def _ensure(self, B):
        import torch
        if B <= self._cap:
            return
        old = (self.gray, self.R) if self._cap else None
        n = B + 1
        self.gray = torch.empty((n, self.rows, self.cols), dtype=torch.uint8, device=self.device)
        self.R = torch.empty((n, self.geo.r_stride), dtype=torch.float32, device=self.device)
        self.dfd = torch.empty(B, dtype=torch.float64, device=self.device)
        self.poly_work = None if self._poly_wf * 4 <= self._smem else torch.empty(
            n * self.geo.n_levels * self._poly_wf, dtype=torch.float32, device=self.device)
        self.flow_work = None if self._flow_wf * 4 <= self._smem else torch.empty(
            B * self._flow_wf, dtype=torch.float32, device=self.device)
        if old is not None:
            self.gray[0].copy_(old[0][0])
            self.R[0].copy_(old[1][0])
        self._cap = B

    def gray_resize(self, frames):
        """uint8 [B,H,W,3] device frames -> uint8 [B, rows, cols] (a view of the detector's buffer)"""
        import torch
        B = self._check(frames)
        with torch.cuda.device(self.device):
            return self._gray_resize(frames, B)

    def _gray_resize(self, frames, B):
        self._ensure(B)
        L = self._L
        L.check(L.lib().pv_shot_gray_resize(L.ptr(frames), B, self.frame_size[1], self.frame_size[0], L.ptr(self.gtab),
                                            self.rows, self.cols, L.ptr(self.gray[1:]), L.stream_ptr()),
                "pv_shot_gray_resize")
        return self.gray[1:B + 1]

    def _check(self, frames):
        import torch
        if frames.device != self.device:
            raise RuntimeError("frames are on %s, the detector on %s" % (frames.device, self.device))
        if frames.dtype != torch.uint8 or frames.dim() != 4 or frames.shape[3] != 3:
            raise RuntimeError("frames must be uint8 [B,H,W,3]")
        if (int(frames.shape[2]), int(frames.shape[1])) != self.frame_size:
            raise RuntimeError("frame size %dx%d, detector built for %dx%d" % (frames.shape[2], frames.shape[1],
                                                                             *self.frame_size))
        if not frames.is_contiguous():
            raise RuntimeError("frames must be contiguous")
        return int(frames.shape[0])

    def dfd_batch(self, frames):
        """float64 device tensor of the DFDs of the pairs completed by these frames"""
        import torch
        B = self._check(frames)
        with torch.cuda.device(self.device):
            if B == 0:
                return torch.empty(0, dtype=torch.float64, device=self.device)
            return self._dfd_batch(frames, B)

    def _dfd_batch(self, frames, B):
        self._gray_resize(frames, B)
        L = self._L
        lib = L.lib()
        L.check(lib.pv_shot_polyexp(L.ptr(self.gray[1:]), B, C.byref(self.geo), L.ptr(self.tab), L.ptr(self.poly_work),
                                    L.ptr(self.R[1:]), L.stream_ptr()), "pv_shot_polyexp")
        first = 0 if self._has_prev else 1
        P = B - first
        out = self.dfd[:P]
        self.flow = None
        if P > 0:
            if self.keep_flow:
                import torch
                self.flow = torch.empty((P, self.rows, self.cols, 2), dtype=torch.float32, device=self.device)
            L.check(lib.pv_shot_flow_dfd(L.ptr(self.gray[first:]), L.ptr(self.R[first:]), P, C.byref(self.geo),
                                         L.ptr(self.tab), L.ptr(self.flow_work), L.ptr(out), L.ptr(self.flow),
                                         L.stream_ptr()), "pv_shot_flow_dfd")
        self.gray[0].copy_(self.gray[B])
        self.R[0].copy_(self.R[B])
        self._has_prev = True
        return out.clone()


# ----------------------------------------------------------------------------------------------------- public class
class Shot(object):
    """Shot boundary detection based on displaced frame difference (same constructor as the reference).

    video: `cli.ArrayVideo` or any object with the reference `Video` attributes (`_size` = (width, height), `step`,
    `start`, `end`, iteration over (t, rgb)); height: resized frame height (the reference's quirk: it becomes the
    number of columns); context: median filter context in seconds; threshold: on the normalised DFD;
    batch: frames per GPU launch.  Frames are staged in a pinned host buffer of `batch` frames (6.2 MB each at
    1080p: 400 MB at the default 64), allocated once per `Shot`; staging, upload and compute of a batch run one after
    the other."""

    def __init__(self, video, height=50, context=2.0, threshold=1.0, batch=64, device=None):
        import torch
        if not torch.cuda.is_available():
            raise RuntimeError("pyannote_video_b200.Shot needs a CUDA device (B200); there is no CPU fallback")
        self.video = video
        self.height = height
        self.context = context
        self.threshold = threshold
        self.batch = int(batch)
        if self.batch < 1:
            raise ValueError("batch must be >= 1")
        self._resize = (height, int(video._size[0] * height / video._size[1]))
        self._kernel_size = kernel_size(context, video.step)
        self._detector = ShotDetector(video._size, height=height, device=device)
        self._pinned = None

    def iter_dfd(self):
        """(t, dfd) of every consecutive pair, t = time of the pair's second frame"""
        import torch
        det = self._detector
        det.reset()
        times, n = [], 0
        pending = []

        def flush(k):
            with torch.cuda.device(det.device):
                frames = self._pinned[:k].to(det.device, non_blocking=True)
                d = det.dfd_batch(frames).cpu().numpy()
            ts = times[len(times) - len(d):] if len(d) else []
            return list(zip(ts, d.tolist()))

        for t, rgb in self.video:
            rgb = np.asarray(rgb)
            shape = (self.batch,) + rgb.shape
            if self._pinned is None or tuple(self._pinned.shape) != shape:
                self._pinned = torch.empty(shape, dtype=torch.uint8).pin_memory()
            self._pinned[n].numpy()[...] = rgb
            times.append(t)
            n += 1
            if n == self.batch:
                pending = flush(n)
                times = times[-1:]
                n = 0
                for item in pending:
                    yield item
        if n:
            for item in flush(n):
                yield item

    def __iter__(self):
        t, y = [], []
        for ti, yi in self.iter_dfd():
            t.append(ti)
            y.append(yi)
        return segments(t, y, self._kernel_size, self.threshold, self.video.start, self.video.end)
