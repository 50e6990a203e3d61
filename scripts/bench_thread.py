"""Shot-threading throughput on one GPU: ORB frames/s from 1080p sources (frames resident in device memory, and
uploaded from pinned host memory), matching pairs/s at lookahead 24, and the reference's CPU path (cv2 ORB and a
fresh FLANN-LSH matcher per pair) on the same frames.  Prints one JSON line and writes it to
profiles/thread_bench.json (or --out), with the card name and power limit.

    python scripts/bench_thread.py [--frames 256] [--batch 64] [--cpu-frames 16] [--out PATH]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _power_limit():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception:
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=256)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--cpu-frames", type=int, default=16)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "thread_bench.json"))
    a = ap.parse_args()
    import cv2
    import torch
    import thread_scenario as sc
    from pyannote_video_b200 import thread as T

    rng = np.random.default_rng(0)
    scenes = [sc._mosaic(np.random.default_rng(s), 1080 + 16, 1920 + 16) for s in range(8)]
    frames = np.stack([scenes[i % 8][o:o + 1080, o:o + 1920] for i, o in
                       enumerate(rng.integers(0, 16, a.frames))])
    ext = T.OrbExtractor((1920, 1080), height=200)
    dev = torch.from_numpy(frames).cuda()
    pinned = torch.from_numpy(frames).pin_memory()

    def run(src):
        descs, sizes = [], []
        for b in range(0, a.frames, a.batch):
            x = src[b:b + a.batch]
            x = x if x.is_cuda else x.cuda(non_blocking=True)
            d, off = ext.extract(x)
            descs.append(d)
            sizes.append(np.diff(off))
        return torch.cat(descs), np.concatenate([[0], np.cumsum(np.concatenate(sizes))])

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        best = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            out = fn()
            torch.cuda.synchronize()
            best.append(time.perf_counter() - t0)
        return float(np.median(best)), out

    t_res, (desc, off) = timed(lambda: run(dev))
    t_pin, _ = timed(lambda: run(pinned))
    pairs = np.array(T.lookahead_pairs(a.frames, 24), np.int32)
    t_match, _ = timed(lambda: T.match_counts(desc, off, pairs, ext.device))

    orb = cv2.ORB_create()
    flann = dict(algorithm=6, table_number=6, key_size=12, multi_probe_level=1)
    t0 = time.perf_counter()
    cd = [orb.detectAndCompute(cv2.cvtColor(cv2.resize(f, (200, 355)), cv2.COLOR_RGB2GRAY), None)[1]
          for f in frames[:a.cpu_frames]]
    t_cpu_orb = time.perf_counter() - t0
    cpairs = T.lookahead_pairs(a.cpu_frames, 24)
    t0 = time.perf_counter()
    for i, j in cpairs:
        cv2.FlannBasedMatcher(flann, dict(checks=50)).knnMatch(cd[i], cd[j], k=2)
    t_cpu_match = time.perf_counter() - t0

    res = {"gpu": torch.cuda.get_device_name(0), "power_limit": _power_limit(), "source": "1920x1080 -> 200x355",
           "frames": a.frames, "batch": a.batch, "keypoints_per_frame": float(np.diff(off).mean()),
           "orb_frames_per_s_resident": a.frames / t_res, "orb_frames_per_s_pinned": a.frames / t_pin,
           "match_pairs": len(pairs), "match_pairs_per_s": len(pairs) / t_match,
           "cpu_reference_orb_frames_per_s": a.cpu_frames / t_cpu_orb,
           "cpu_reference_flann_pairs_per_s": len(cpairs) / t_cpu_match}
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
