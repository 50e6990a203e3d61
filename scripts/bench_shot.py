"""Shot boundary detection throughput: pairs/s of the CUDA path on 1080p frames, next to the CPU path of the
reference (cv2 Farneback plus the per-pixel DFD loop) and its cv2-only part, on the same frames.

    python scripts/bench_shot.py [--frames 2048] [--batch 512] [--passes 200] [--cpu-pairs 40] [--out result.json]

resident: 1080p RGB frames already in HBM (the tensors the face path uploads), cycled through `frames` distinct
frames (12.7 GB at 2048, far more than L2), timed with CUDA events.  e2e: the same from pinned host memory, upload
included.  Prints one JSON line; the card name and power limit are read in the same run.
"""
import argparse
import itertools
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (s.strip() for s in out.split(","))
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:                      # noqa: BLE001
        return dict(error=str(e))


def make_frames_gpu(n, H, W, device, seed=0):
    """smooth translating 1080p content with a hard cut every 97 frames"""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    out = torch.empty((n, H, W, 3), dtype=torch.uint8, device=device)
    for s in range(0, n, 97):
        m = min(97, n - s)
        base = torch.rand(1, 3, H // 24 + 16, W // 24 + 16, generator=g, device=device)
        tex = torch.nn.functional.interpolate(base, scale_factor=24, mode="bilinear", align_corners=False)[0]
        for i in range(m):
            out[s + i] = (tex[:, 2 * i:2 * i + H, 3 * i:3 * i + W].permute(1, 2, 0) * 255).to(torch.uint8)
    return out


def reference_loop_dfd(prev, cur, flow):
    """the per-pixel loop of the reference's DFD, as it runs there (Python, one pixel at a time)"""
    h, w = prev.shape
    rec = np.empty(prev.shape)
    for x, y in itertools.product(range(w), range(h)):
        dy, dx = flow[y, x]
        rx = int(max(0, min(x + dx, w - 1)))
        ry = int(max(0, min(y + dy, h - 1)))
        rec[y, x] = cur[ry, rx]
    return np.mean(np.abs(prev - rec))


def cpu_baseline(frames_np, height=50):
    import cv2
    h, w = frames_np.shape[1:3]
    size = (height, int(w * height / h))
    conv = lambda f: cv2.resize(cv2.cvtColor(f, cv2.COLOR_RGB2GRAY), size)   # noqa: E731
    flow = lambda a, b: cv2.calcOpticalFlowFarneback(a, b, None, 0.5, 3, 15, 3, 5, 1.1, 0)   # noqa: E731
    n = len(frames_np) - 1
    t0 = time.perf_counter()
    prev = conv(frames_np[0])
    for i in range(1, len(frames_np)):
        cur = conv(frames_np[i])
        reference_loop_dfd(prev, cur, flow(prev, cur))
        prev = cur
    t_ref = time.perf_counter() - t0
    t0 = time.perf_counter()
    prev = conv(frames_np[0])
    for i in range(1, len(frames_np)):
        cur = conv(frames_np[i])
        flow(prev, cur)
        prev = cur
    t_cv2 = time.perf_counter() - t0
    return dict(pairs=n, reference_pairs_per_s=n / t_ref, cv2_only_pairs_per_s=n / t_cv2, cv2_threads=cv2.getNumThreads())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=2048)
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--passes", type=int, default=200)
    ap.add_argument("--e2e-batches", type=int, default=8)
    ap.add_argument("--cpu-pairs", type=int, default=40)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_shot.py measures the CUDA path: no CUDA device")
    import __graft_entry__
    __graft_entry__.build()
    from pyannote_video_b200.shot import ShotDetector
    dev = torch.device("cuda:0")
    H, W = 1080, 1920
    frames = make_frames_gpu(a.frames, H, W, dev)
    det = ShotDetector((W, H), device=dev)
    B = a.batch
    det.dfd_batch(frames[:B].contiguous())          # warm-up (module load, workspaces)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pairs = 0
    e0.record()
    for _ in range(a.passes):
        for s in range(0, a.frames - B + 1, B):
            det.dfd_batch(frames[s:s + B])
            pairs += B
    e1.record()
    torch.cuda.synchronize()
    resident_s = e0.elapsed_time(e1) / 1e3

    host = frames[:B].cpu().pin_memory()
    host2 = frames[B:2 * B].cpu().pin_memory()
    det.reset()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e2e_pairs = 0
    for k in range(a.e2e_batches):
        d = det.dfd_batch((host if k % 2 == 0 else host2).to(dev, non_blocking=True))
        e2e_pairs += len(d)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0

    cpu = None
    try:
        cpu = cpu_baseline(frames[:a.cpu_pairs + 1].cpu().numpy())
    except ImportError:
        cpu = "not measured (cv2 missing)"
    res = dict(metric="shot_pairs_per_s", card=card(), frame="1080x1920 RGB", height=50, batch=B,
               resident=dict(frames=a.frames, bytes=int(frames.numel()), pairs=pairs, seconds=resident_s,
                             pairs_per_s=pairs / resident_s),
               e2e_pinned=dict(pairs=e2e_pairs, seconds=e2e_s, pairs_per_s=e2e_pairs / e2e_s,
                               upload_bytes_per_frame=H * W * 3),
               cpu_baseline=cpu)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
