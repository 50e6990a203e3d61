"""Shot threading on the GPU — a drop-in for pyannote.video.Thread (pyannote/video/structure/thread.py).

Shots n and n + k (0 < k <= lookahead) are linked when the frame 10 frames before the end of shot n and the frame
10 frames after the start of shot n + k share more than `min_match` ORB matches (cv2.ORB_create() features; a query
descriptor matches when its best Hamming distance is below 0.7 times the second best).  Threads are the connected
components of that graph, labelled A, B, ... by their first shot; `scenes` merges intertwined threads.

The frame work runs in csrc/orb.cu: resize + gray, then the whole ORB extraction of a frame in one CTA, many frames
per launch; every pair of a clip is matched in one more launch.  The matching is the exact brute-force 2-NN count,
which the reference's FLANN-LSH matcher approximates with random hash tables.  This module builds the geometry,
stages frames and does the (tiny) graph work on the host.
"""
import ctypes as C
import warnings

import numpy as np

from .annotation import Annotation, Segment, pairwise, string_generator
from .shot import gray_table

N_FEATURES = 500
SCALE_FACTOR = float(np.float32(1.2))       # cv2.ORB_create takes a float; the pyramid uses it as a double
N_LEVELS = 8
EDGE = 31
f32 = np.float32


class PvOrbGeo(C.Structure):
    _fields_ = [("n_levels", C.c_int32)] \
        + [(n, C.c_int32 * N_LEVELS) for n in ("rows", "cols", "off", "tab_off", "quota")] \
        + [("scale", C.c_float * N_LEVELS), ("gauss", C.c_float * 7), ("plane", C.c_int32), ("cand_cap", C.c_int32)]


# ----------------------------------------------------------------------------------------------------- geometry
def resize_shape(frame_size, height):
    """(rows, cols) of the resized frame for a (width, height) video: cv2.resize(rgb, (height, int(w*height/h)))"""
    w, h = frame_size
    return int(w * height / h), int(height)


def _round(v):
    return int(np.rint(v))                   # cvRound: half to even


def level_scales():
    """float32 scale of every level: (float)pow(1.2f, k), as cv2's getScale"""
    return [f32(SCALE_FACTOR ** k) for k in range(N_LEVELS)]


def level_sizes(rows, cols):
    """[(rows, cols)] of the ORB pyramid: cvRound(size / scale) with the division in float32 (int / float in cv2)"""
    return [(_round(f32(rows) / s), _round(f32(cols) / s)) for s in level_scales()]


def level_quotas(n=N_FEATURES):
    factor = f32(1.0 / SCALE_FACTOR)
    per = f32(n * (f32(1) - factor) / (f32(1) - f32(np.float64(factor) ** N_LEVELS)))
    out = []
    for _ in range(N_LEVELS - 1):
        out.append(_round(per))
        per = f32(per * factor)
    return out + [max(n - sum(out), 0)]


def gaussian7():
    """cv2.getGaussianKernel(7, 2, CV_32F): float32 samples, normalised by their double sum"""
    x = np.arange(7) - 3.0
    k = np.exp(-0.5 / 4.0 * x * x).astype(f32)
    return (k.astype(np.float64) * (1.0 / k.astype(np.float64).sum())).astype(f32)


def exact_taps(src, dst):
    """INTER_LINEAR_EXACT (offset, 8-bit weight of the second tap) per destination index; the ORB pyramid's 1.2x
    downscales never reach the replicated borders"""
    scale = 1.0 / (dst / src)
    ofs, c1 = np.empty(dst, np.int32), np.empty(dst, np.int32)
    for d in range(dst):
        f = scale * (d + 0.5) - 0.5
        i = int(np.floor(f))
        if i < 0 or i >= src - 1:
            raise ValueError("INTER_LINEAR_EXACT border taps (%d -> %d) are not supported" % (src, dst))
        ofs[d], c1[d] = i, _round((f - i) * 256)
    return ofs, c1


def make_geometry(rows, cols, n_features=N_FEATURES):
    """(PvOrbGeo, int32 table of the pyramid's resize taps)"""
    g = PvOrbGeo()
    sizes = level_sizes(rows, cols)
    g.n_levels = N_LEVELS
    tab, off, cap = [], 0, 0
    for k, ((r, c), q) in enumerate(zip(sizes, level_quotas(n_features))):
        g.rows[k], g.cols[k], g.off[k], g.quota[k] = r, c, off, q
        g.scale[k] = float(level_scales()[k])
        g.tab_off[k] = sum(t.size for t in tab)
        if k:
            pr, pc = sizes[k - 1]
            xo, xc = exact_taps(pc, c)
            yo, yc = exact_taps(pr, r)
            tab += [xo, xc, yo, yc]
        off += r * c
        # non-max suppression keeps no two 8-adjacent points: at most ceil(w/2) * ceil(h/2) inside the border
        cap += ((max(c - 2 * EDGE, 0) + 1) // 2) * ((max(r - 2 * EDGE, 0) + 1) // 2)
    for j, v in enumerate(gaussian7()):
        g.gauss[j] = float(v)
    g.plane = off
    g.cand_cap = max(cap, 1)
    tab = np.concatenate(tab) if tab else np.zeros(1, np.int32)
    return g, tab.astype(np.int32)


# ----------------------------------------------------------------------------------------------------- device level
class OrbExtractor(object):
    """cv2.ORB_create().detectAndCompute of `cv2.cvtColor(cv2.resize(rgb, (height, int(w*height/h))), RGB2GRAY)` for
    uint8 [B,H,W,3] frames already on the GPU.  `extract(frames)` returns (descriptors uint8 [N,32] on the device,
    int64 per-frame offsets [B+1] on the host); with keep_keypoints, `keypoints` then holds one float32 [n,5] array
    (x, y, octave, response, angle) per frame, in (octave, y, x) order.  Frames must be on the extractor's device;
    every launch runs on that device's current stream, whatever the caller's current device is."""

    def __init__(self, frame_size, height=200, device=None, keep_keypoints=False):
        import torch
        if not torch.cuda.is_available():
            raise RuntimeError("pyannote_video_b200.Thread needs a CUDA device (B200); there is no CPU fallback")
        from . import _lib
        self._L = _lib
        dev = torch.device(device) if device is not None else torch.device("cuda")
        if dev.type != "cuda":
            raise RuntimeError("OrbExtractor runs on a CUDA device, got %s" % dev)
        self.device = dev if dev.index is not None else torch.device("cuda", torch.cuda.current_device())
        self.frame_size = (int(frame_size[0]), int(frame_size[1]))
        self.rows, self.cols = resize_shape(self.frame_size, height)
        if self.rows < 1 or self.cols < 1:
            raise ValueError("resized frame would be empty: %r at height %d" % (self.frame_size, height))
        self.geo, tab = make_geometry(self.rows, self.cols)
        lib = _lib.lib()
        lib.pv_orb_work_bytes.restype = C.c_int64
        self._work_bytes = int(lib.pv_orb_work_bytes(C.byref(self.geo)))
        if self._work_bytes <= 0:
            raise RuntimeError("pv_orb_work_bytes: bad geometry for %dx%d" % (self.cols, self.rows))
        with torch.cuda.device(self.device):
            self.tab = torch.from_numpy(tab).to(self.device)
            self.gtab = torch.from_numpy(gray_table(self.frame_size, self.rows, self.cols)).to(self.device)
        self.keep_keypoints = keep_keypoints
        self.keypoints = None
        self._cap = 0

    def _ensure(self, B):
        import torch
        if B <= self._cap:
            return
        cap = self.geo.cand_cap
        self.gray = torch.empty((B, self.rows, self.cols), dtype=torch.uint8, device=self.device)
        self.work = torch.empty(B * self._work_bytes, dtype=torch.uint8, device=self.device)
        self.kp = torch.empty((B, cap, 5), dtype=torch.float32, device=self.device)
        self.desc = torch.empty((B, cap, 32), dtype=torch.uint8, device=self.device)
        self.count = torch.empty(B, dtype=torch.int32, device=self.device)
        self._cap = B

    def _check(self, frames):
        import torch
        if frames.device != self.device:
            raise RuntimeError("frames are on %s, the extractor on %s" % (frames.device, self.device))
        if frames.dtype != torch.uint8 or frames.dim() != 4 or frames.shape[3] != 3:
            raise RuntimeError("frames must be uint8 [B,H,W,3]")
        if (int(frames.shape[2]), int(frames.shape[1])) != self.frame_size:
            raise RuntimeError("frame size %dx%d, extractor built for %dx%d" % (frames.shape[2], frames.shape[1],
                                                                              *self.frame_size))
        if not frames.is_contiguous():
            raise RuntimeError("frames must be contiguous")
        return int(frames.shape[0])

    def gray_resize(self, frames):
        """uint8 [B,H,W,3] device frames -> uint8 [B, rows, cols] (a view of the extractor's buffer)"""
        import torch
        B = self._check(frames)
        with torch.cuda.device(self.device):
            return self._gray_resize(frames, B)

    def _gray_resize(self, frames, B):
        self._ensure(B)
        L = self._L
        L.check(L.lib().pv_orb_resize_gray(L.ptr(frames), B, self.frame_size[1], self.frame_size[0], L.ptr(self.gtab),
                                           self.rows, self.cols, L.ptr(self.gray), L.stream_ptr()),
                "pv_orb_resize_gray")
        return self.gray[:B]

    def extract(self, frames):
        import torch
        B = self._check(frames)
        with torch.cuda.device(self.device):
            if B == 0:
                self.keypoints = [] if self.keep_keypoints else None
                return torch.empty((0, 32), dtype=torch.uint8, device=self.device), np.zeros(1, np.int64)
            self._gray_resize(frames, B)
            L = self._L
            L.check(L.lib().pv_orb_detect(L.ptr(self.gray), B, C.byref(self.geo), L.ptr(self.tab), L.ptr(self.work),
                                          L.ptr(self.kp), L.ptr(self.desc), L.ptr(self.count), L.stream_ptr()),
                    "pv_orb_detect")
            counts = self.count[:B].cpu().numpy().astype(np.int64)
            if (counts < 0).any():
                raise RuntimeError("pv_orb_detect: keypoint candidates exceed %d slots" % self.geo.cand_cap)
            keep = torch.arange(self.geo.cand_cap, device=self.device)[None, :] < self.count[:B, None]
            desc = self.desc[:B][keep]
            if self.keep_keypoints:
                kp = self.kp[:B][keep].cpu().numpy()
                self.keypoints = np.split(kp, np.cumsum(counts)[:-1])
            return desc, np.concatenate([[0], np.cumsum(counts)])


def match_counts(desc, offsets, pairs, device):
    """int32 [P] exact 2-NN ratio counts of (query frame, train frame) pairs over packed descriptors"""
    import torch
    from . import _lib as L
    pairs = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
    if len(pairs) == 0:
        return np.zeros(0, np.int32)
    with torch.cuda.device(device):
        if desc.shape[0] == 0:
            desc = torch.zeros((1, 32), dtype=torch.uint8, device=device)
        off = torch.from_numpy(np.asarray(offsets, np.int32)).to(device)
        pr = torch.from_numpy(pairs).to(device)
        out = torch.empty(len(pairs), dtype=torch.int32, device=device)
        L.check(L.lib().pv_thread_match(L.ptr(desc.contiguous()), L.ptr(off), L.ptr(pr), len(pairs), L.ptr(out),
                                        L.stream_ptr()), "pv_thread_match")
        return out.cpu().numpy()


# ----------------------------------------------------------------------------------------------------- graph work
def lookahead_pairs(n, lookahead):
    """the pair set of the reference's product_lookahead: (i, j) with 0 < j - i <= lookahead"""
    return [(i, j) for i in range(n) for j in range(i + 1, min(n, i + lookahead + 1))]


def components(n, edges):
    """connected components of nodes 0..n-1 (union-find), each sorted, ordered by their first node"""
    parent = list(range(n))

    def find(a):
        while parent[a] != a:
            parent[a] = parent[parent[a]]
            a = parent[a]
        return a

    for a, b in edges:
        ra, rb = find(a), find(b)
        if ra != rb:
            parent[max(ra, rb)] = min(ra, rb)
    groups = {}
    for i in range(n):
        groups.setdefault(find(i), []).append(i)
    return sorted(groups.values(), key=lambda g: g[0])


def biconnected_components(edges):
    """node sets of the biconnected components of an undirected simple graph (iterative Tarjan)"""
    adj = {}
    for a, b in edges:
        if a != b:
            adj.setdefault(a, set()).add(b)
            adj.setdefault(b, set()).add(a)
    disc, low, out, clock = {}, {}, [], 0
    for root in adj:
        if root in disc:
            continue
        disc[root] = low[root] = clock
        clock += 1
        stack, estack = [(root, None, iter(sorted(adj[root])))], []
        while stack:
            u, parent, it = stack[-1]
            for v in it:
                if v == parent:
                    continue
                if v not in disc:
                    disc[v] = low[v] = clock
                    clock += 1
                    estack.append((u, v))
                    stack.append((v, u, iter(sorted(adj[v]))))
                    break
                if disc[v] < disc[u]:
                    low[u] = min(low[u], disc[v])
                    estack.append((u, v))
            else:
                stack.pop()
                if parent is not None:
                    low[parent] = min(low[parent], low[u])
                    if low[u] >= disc[parent]:
                        comp = set()
                        while True:
                            e = estack.pop()
                            comp.update(e)
                            if e == (parent, u):
                                break
                        out.append(comp)
    return out


def thread_annotation(shots, edges):
    """the reference's Thread.__call__ from its graph: components labelled A, B, ... by first shot, smoothed"""
    annotation = Annotation()
    labels = string_generator()
    for comp in components(len(shots), edges):
        label = next(labels)
        for i in comp:
            annotation[shots[i]] = label
    return annotation.smooth()


def scenes(threads):
    """the reference's Thread.scenes: tracks of every biconnected component (>= 3 tracks) of the graph of
    time-adjacent tracks and consecutive same-label tracks take the label of the component's first track"""
    edges = list(pairwise(threads.itertracks()))
    for label in threads.labels():
        edges += list(pairwise(threads.subset([label]).itertracks()))
    out = threads.copy()
    for shots in sorted(sorted(bc) for bc in biconnected_components(edges)):
        if len(shots) < 3:
            continue
        common = out[shots[0]]
        for shot in shots:
            out[shot] = common
    return out


# ----------------------------------------------------------------------------------------------------- public class
class Thread(object):
    """Shot threading based on ORB features (same constructor as the reference, plus `batch` and `device`).

    video: `cli.ArrayVideo` or any object with the reference `Video` interface (`_size`, `frame_rate`, `video(t)`);
    shot: iterable of segments (None: this package's GPU `Shot`); height: resized frame height (the reference's
    quirk: it becomes the number of columns); min_match: an edge needs more matches than this; lookahead: shots
    compared with each shot; batch: frames per ORB launch.  At most two frames per shot are read, staged in a pinned
    buffer of `batch` frames and uploaded batch by batch; all pairs are then matched in one launch."""

    def __init__(self, video, shot=None, height=200, min_match=20, lookahead=5, verbose=False, batch=64, device=None):
        import torch
        if not torch.cuda.is_available():
            raise RuntimeError("pyannote_video_b200.Thread needs a CUDA device (B200); there is no CPU fallback")
        self.video = video
        self.height = height
        w, h = video._size
        self._resize = (int(height), int(w * height / h))
        self.lookahead = lookahead
        if shot is None:
            from .shot import Shot
            shot = Shot(video, device=device)
        self.shot = shot
        self.verbose = verbose
        self.min_match = min_match
        self.batch = int(batch)
        if self.batch < 1:
            raise ValueError("batch must be >= 1")
        self._extractor = OrbExtractor(video._size, height=height, device=device)
        self._pinned = None
        self.counts = None

    def _descriptors(self, times):
        """(packed device descriptors, offsets [len(times)+1]) of the frames at `times`; a frame the video cannot
        reach warns and gets no descriptors, as in the reference"""
        import torch
        ext = self._extractor
        descs, sizes = [], np.zeros(len(times), np.int64)
        n, pending = 0, []

        def flush():
            with torch.cuda.device(ext.device):
                d, off = ext.extract(self._pinned[:n].to(ext.device, non_blocking=True))
            descs.append(d)
            sizes[pending] = np.diff(off)

        for i, t in enumerate(times):
            try:
                rgb = np.asarray(self.video(t))
            except IOError:
                warnings.warn("unable to reach t = {t:.3f}".format(t=t))
                continue
            shape = (self.batch,) + rgb.shape
            if self._pinned is None or tuple(self._pinned.shape) != shape:
                if n:
                    flush()
                    n, pending = 0, []
                self._pinned = torch.empty(shape, dtype=torch.uint8).pin_memory()
            self._pinned[n].numpy()[...] = rgb
            pending.append(i)
            n += 1
            if n == self.batch:
                flush()
                n, pending = 0, []
        if n:
            flush()
        packed = torch.cat(descs) if descs else torch.zeros((0, 32), dtype=torch.uint8, device=ext.device)
        return packed, np.concatenate([[0], np.cumsum(sizes)])

    def _graph(self):
        """(shots, edges); the count of every compared pair is kept in `self.counts`"""
        shots = [Segment(s.start, s.end) for s in self.shot]
        collar = 10. / self.video.frame_rate
        times, slot, ends, starts = [], {}, [], []
        for s in shots:
            for t, lst in ((s.end - collar, ends), (s.start + collar, starts)):
                if t not in slot:
                    slot[t] = len(times)
                    times.append(t)
                lst.append(slot[t])
        packed, offsets = self._descriptors(times)
        pairs = lookahead_pairs(len(shots), self.lookahead)
        qt = np.array([(ends[i], starts[j]) for i, j in pairs], np.int32).reshape(-1, 2)
        counts = match_counts(packed, offsets, qt, self._extractor.device)
        self.counts = dict(zip(pairs, counts.tolist()))
        return shots, [p for p, c in zip(pairs, counts) if c > self.min_match]

    def __call__(self):
        shots, edges = self._graph()
        return thread_annotation(shots, edges)

    def scenes(self, threads):
        return scenes(threads)
