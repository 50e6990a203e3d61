#!/usr/bin/env python
"""bench.py — frames/sec of the face hot path (CNN detect -> correlation-tracker update -> 68-pt landmarks -> chip ->
ResNet embed) on synthetic 1080p, BASELINE.json configs[1], on N GPUs of one node.

    python bench.py --gpus 1 --steps 60 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the C++ CPU restatement of the reference's dlib path, all usable cores

A step = `--frames-per-step` (32) concurrent shot streams each advancing by ONE 1080p frame (tracking state is
independent per shot, pyannote/video/tracking.py:410-417, so shots are the unit that batches):
  * every frame detected with upsample 1 (reference semantics, pyannote/video/face/face.py:66),
  * K = 8 live tracks per stream, a forward and a backward correlation tracker each (tracking.py:199-206,331-337):
    16 `correlation_tracker.update` per frame, all streams in one bank launch,
  * F = 4 seeded face boxes per frame through landmarks + chip + embed (mirrors `extract`, where boxes come from the
    track file, scripts/pyannote-face.py:290-297).
Prints ONE JSON line (contract in the task statement).  Only the `cpu_baseline` leg and `--impl reference` execute
anything under oracle/ (the C++ restatement oracle/cpu, as the timed CPU baseline).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W = 1080, 1920
FACES_PER_FRAME = 4
TRACKS_PER_STREAM = 8          # live tracks per shot stream; x2 (forward + backward tracker) updates per frame
N_TIMES = 4                    # distinct time steps held per stream (ping-pong 0,1,2,3,2,1,...: motion stays continuous)
SHIFT = (1.0, 0.5)             # px / frame global translation (SURVEY.md §8d, C3)
METRIC = "frames/sec detect+track+embed on 1080p"
WORKLOAD = ("synthetic 1080p@25fps: batched CNN detect (upsample 1, every frame) + %d correlation-tracker updates/frame "
            "(%d live tracks x fwd+bwd) + %d faces/frame 68-pt landmarks + ResNet-v1 embed"
            % (2 * TRACKS_PER_STREAM, TRACKS_PER_STREAM, FACES_PER_FRAME))
TRACKER_BYTES_PER_UPDATE = 2.07e6      # SURVEY.md §8(d): A read + written (f32 complex 31x64x64), B, chip
DUMP_MAX_BYTES = 64 << 20


def time_index(s):
    seq = list(range(N_TIMES)) + list(range(N_TIMES - 2, 0, -1))
    return seq[s % len(seq)]


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm_gbs=d.get("hbm_gbs"), tf_sustained=d.get("bf16_tflops_sustained"), tf_burst=d.get("bf16_tflops"),
                    source="measured")
    return dict(hbm_gbs=6650.0, tf_sustained=1400.0, tf_burst=1590.0, source="fallback")


class ClockSampler(threading.Thread):
    """samples nvidia-smi clocks / throttle reasons during the timed region"""

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = False
        self.rows = []

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if r[1].isdigit()]
        reasons = []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for i, nme in enumerate(names):
            if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows):
                reasons.append(nme)
        return dict(sm_mhz=(sm[len(sm) // 2] if sm else None), sm_max_mhz=(max(mx) if mx else None), reasons=reasons,
                    samples=len(self.rows))


def dump_outputs(out_dir, arrays, seed=0):
    """--dump-outputs: `arrays` (name -> numpy array) as out_dir/<name>.npy, float64 kept, everything else as float32
    (integer outputs are small coordinates and counts, exact in float32).  Above DUMP_MAX_BYTES in all, every array keeps
    the same seeded sample of its leading-axis rows, so two runs with the same arguments write the same rows."""
    import numpy as np
    arrays = {k: np.ascontiguousarray(a, np.float64 if a.dtype == np.float64 else np.float32) for k, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if total > DUMP_MAX_BYTES and a.shape[0] > 1:
            keep = max(1, a.shape[0] * DUMP_MAX_BYTES // total)
            a = a[np.sort(np.random.default_rng(seed).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def make_models():
    from pyannote_video_b200 import weights as Wt
    return Wt.make_detector(seed=2), Wt.make_shape_predictor(seed=4), Wt.make_embedder(seed=3)


def track_rects(n_streams):
    """TRACKS_PER_STREAM 96x96 boxes on a 4x2 grid per stream: float32 [n*K,4] (l,t,r,b), stream index int32 [n*K]"""
    import torch
    rects, sidx = [], []
    for s in range(n_streams):
        for k in range(TRACKS_PER_STREAM):
            cx = 240.0 + 480.0 * (k % 4)
            cy = 300.0 + 480.0 * (k // 4)
            rects.append([cx - 48.0, cy - 48.0, cx + 48.0, cy + 48.0])
            sidx.append(s)
    return torch.tensor(rects, dtype=torch.float32), torch.tensor(sidx, dtype=torch.int32)


# ------------------------------------------------------------------------------------------------
# C++ CPU restatement of the reference path (oracle/cpu) — used by cpu_baseline and --impl reference
# ------------------------------------------------------------------------------------------------
class CpuPath(object):
    """the same per-frame work as one stream of the GPU step, on host cores: detect + 2K tracker updates + F faces"""

    def __init__(self, models, threads):
        from oracle import cpu_ref
        self.cpu_ref = cpu_ref
        self.threads = cpu_ref.set_threads(threads)
        det, sp, emb = models
        self.det = cpu_ref.Detector(det)
        self.sp = cpu_ref.ShapePredictor(sp)
        self.emb = cpu_ref.Embedder(emb)
        self.bank = None

    def start_tracks(self, frame):
        import numpy as np
        rects, _ = track_rects(1)
        rects = np.concatenate([rects.numpy(), rects.numpy()]).astype(np.float64)       # forward + backward trackers
        self.ids = np.arange(rects.shape[0], dtype=np.int32)
        self.bank = self.cpu_ref.TrackerBank(len(self.ids), use_scale=True)
        self.bank.start(frame, self.ids, rects)

    def frame(self, rgb, boxes):
        self.cpu_ref.set_threads(self.threads)
        self.det.detect(rgb, 1)
        self.bank.update(rgb, self.ids)
        parts = self.sp.predict(rgb, boxes)
        chips = self.cpu_ref.extract_chips(rgb, parts)
        return self.emb.forward(chips)


def cpu_sample(models, threads, n_frames, seed=0):
    """times n_frames frames through the C++ path; returns (seconds, threads used).  threads > 1 = frame-level
    parallelism (BASELINE.md §2 "B-cpu-N": `threads` independent streams, one host thread each, every stream doing the
    same per-frame work as one stream of the GPU step); threads == 1 = one stream on one thread ("B-cpu-1")."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import cpu_ref
    from pyannote_video_b200.synth import make_frames, make_boxes
    frames = make_frames(N_TIMES, H, W, seed=seed, shift_per_frame=SHIFT).numpy()
    boxes, fidx = make_boxes(N_TIMES, FACES_PER_FRAME, H, W, seed=1)
    boxes = boxes.numpy().reshape(N_TIMES, FACES_PER_FRAME, 4)
    threads = max(1, int(threads))
    per = max(1, n_frames // threads)
    cpu_ref.lib()                                   # (build and) load the library before the worker threads start

    def worker(k, timed):
        cpu_ref.set_threads(1)                      # OpenMP's thread count is per host thread: every worker runs serial code
        if k not in paths:
            paths[k] = CpuPath(models, 1)
            paths[k].start_tracks(frames[0])
            paths[k].frame(frames[1], boxes[1])     # warm-up (page faults, block pool)
        if timed:
            for i in range(per):
                t = time_index(i + 2)
                paths[k].frame(frames[t], boxes[t])

    paths = {}
    with ThreadPoolExecutor(max_workers=threads) as ex:
        list(ex.map(lambda k: worker(k, False), range(threads)))
        t0 = time.perf_counter()
        list(ex.map(lambda k: worker(k, True), range(threads)))
        el = time.perf_counter() - t0
    return el, threads, per * threads


def run_reference(args, rank, world):
    """--impl reference: the C++ restatement of the reference's dlib path with all usable host cores (rank 0 only):
    frame-level parallelism, one stream per core.  Each timed step = one frame per core."""
    if rank != 0:
        return
    from oracle import cpu_ref
    models = make_models()
    cores = cpu_ref.host_cores()
    steps = max(1, min(args.steps, 30))
    el, used, n = cpu_sample(models, cores, steps * cores)
    fps = n / el
    frames_per_step = cores
    sample = ("%d steps x %d 1080p frames (%d independent streams, one host thread each; same per-frame work as one stream "
              "of the GPU step)" % (steps, frames_per_step, used))
    line = dict(metric=METRIC, value=fps, unit="frames/s", n_gpus=args.gpus, steps=steps, warmup=1,
                ms_per_step=1000.0 * el / steps, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic", impl="reference",
                config=dict(workload=WORKLOAD, frames_per_step=frames_per_step, faces_per_frame=FACES_PER_FRAME,
                            tracker_updates_per_frame=2 * TRACKS_PER_STREAM, sample=sample,
                            implementation="restated dlib-style CPU baseline: C++ -O3 -march=native, fp32 blocked direct "
                                           "convolutions (oracle/cpu), frame-level parallelism over all usable cores; not dlib "
                                           "itself (absent here)"),
                cpu_baseline=dict(value=fps, unit="frames/s", cores=used, kind="port", sample=sample,
                                  host_threads_visible=os.cpu_count(),
                                  cores_note="usable cores = min(online CPUs, cgroup cpu.max quota)"),
                e2e=dict(value=fps, unit="frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames-per-step", type=int, default=32)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-tracker", action="store_true", help="leave the tracker updates out of the step (C2 without tracking)")
    ap.add_argument("--profile-convs", type=int, default=2, help="instrumented steps for the roofline leg")
    ap.add_argument("--ncu-step", action="store_true",
                    help="after the warm-up, run ONE serialised step between cudaProfilerStart/Stop and exit (for `ncu "
                         "--profile-from-start off`: the launch list / --set full capture of exactly one step)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (detections, landmarks, embeddings, "
                         "tracker state; rank 0) as DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    if world > 1:
        dist.barrier()
    from pyannote_video_b200 import _lib
    from pyannote_video_b200.face import Face
    from pyannote_video_b200.tracker import TrackerBank
    from pyannote_video_b200.synth import make_frames, make_boxes

    det_m, sp_m, emb_m = make_models()
    B = args.frames_per_step
    use_tracker = not args.no_tracker
    face = Face(landmarks=sp_m, embedding=emb_m, detector=det_m, upsample=1, device=dev, max_frames=B,
                max_faces=B * FACES_PER_FRAME)
    # B streams x N_TIMES consecutive frames each (a translating canvas per stream): 4 x B x 6.2 MB, larger than L2
    dev_sets = [torch.empty(B, H, W, 3, dtype=torch.uint8, device=dev) for _ in range(N_TIMES)]
    for b in range(B):
        seq = make_frames(N_TIMES, H, W, seed=1000 * rank + b, device=dev, shift_per_frame=SHIFT)
        for t in range(N_TIMES):
            dev_sets[t][b] = seq[t]
        del seq
    host_sets = [fr.cpu().pin_memory() for fr in dev_sets]
    box_sets = []
    for t in range(N_TIMES):
        bx, fi = make_boxes(B, FACES_PER_FRAME, H, W, seed=1 + t + 10 * rank)
        box_sets.append((bx.to(dev), fi.to(dev), bx.pin_memory(), fi.pin_memory()))

    # tracker bank: forward + backward tracker of K tracks in each of the B streams, started on time step 0
    n_tracks = 2 * TRACKS_PER_STREAM * B
    bank = None
    if use_tracker:
        bank = TrackerBank(capacity=n_tracks, device=dev)
        rects, sidx = track_rects(B)
        trk_rects = torch.cat([rects, rects]).to(dev)
        trk_frame = torch.cat([sidx, sidx]).to(dev)
        trk_ids = torch.arange(n_tracks, dtype=torch.int32, device=dev)
        bank.start_batch(dev_sets[0], trk_frame, trk_ids, trk_rects)
        torch.cuda.synchronize(dev)

    # landmarks + chips + embed of the seeded boxes and the tracker updates do not depend on this frame's detections
    # (in `extract` the boxes come from the track file; trackers are updated before association, tracking.py:202-206),
    # so they run on a side stream and fill the SM slots the pyramid kernels leave free.
    side = torch.cuda.Stream(device=dev)
    overlap = [True]
    det0 = face._detector_for(H, W)

    def step_device(fr, bx, fi, out=None):
        """one step on device-resident inputs; returns the dict of result tensors"""
        main = torch.cuda.current_stream()
        if overlap[0]:
            side.wait_stream(main)
            ctx = torch.cuda.stream(side)
        else:
            ctx = torch.cuda.stream(main)
        with ctx:
            res = face.extract_batch(fr, bx, fi, detect=False, out=out)
            if use_tracker:
                bank.update_batch(fr, trk_frame, trk_ids)
        boxes, scores, counts = det0.detect(fr)
        res["det_boxes"], res["det_scores"], res["det_counts"] = boxes, scores, counts
        if overlap[0]:
            main.wait_stream(side)
        return res

    res_buf = dict(landmarks=torch.empty(B * FACES_PER_FRAME, 68, 2, dtype=torch.int32, device=dev),
                   embeddings=torch.empty(B * FACES_PER_FRAME, 128, dtype=torch.float32, device=dev))

    def step_resident(s):
        t = time_index(s)
        bx, fi, _, _ = box_sets[t]
        return step_device(dev_sets[t], bx, fi, out=res_buf)

    # ---------------- end-to-end: pinned host frames -> Face.upload (public API, staging ring + copy stream) -> the same
    # step -> detections / tracker state / landmarks / embeddings copied back to pinned host memory, read one step behind
    out_host = [dict(boxes=torch.empty(B, det0.MAX_DET, 4, dtype=torch.int32).pin_memory(),
                     counts=torch.empty(B, dtype=torch.int32).pin_memory(),
                     parts=torch.empty(B * FACES_PER_FRAME, 68, 2, dtype=torch.int32).pin_memory(),
                     emb=torch.empty(B * FACES_PER_FRAME, 128, dtype=torch.float32).pin_memory(),
                     trk=torch.empty(n_tracks, 5, dtype=torch.float32).pin_memory(),
                     ev=torch.cuda.Event()) for _ in range(2)]
    staged = {}

    def upload(s):
        t = time_index(s)
        _, _, bx_h, fi_h = box_sets[t]
        staged[s] = face.upload(host_sets[t], bx_h, fi_h, slot=s % 3)

    def step_e2e(s, n_total):
        fr, bx, fi, ready = staged.pop(s)
        main = torch.cuda.current_stream()
        main.wait_event(ready)
        if s + 1 < n_total:
            upload(s + 1)                       # the next step's inputs travel while this step computes
        res = step_device(fr, bx, fi, out=res_buf)
        o = out_host[s % 2]
        o["boxes"].copy_(res["det_boxes"], non_blocking=True)
        o["counts"].copy_(res["det_counts"], non_blocking=True)
        o["parts"].copy_(res["landmarks"], non_blocking=True)
        o["emb"].copy_(res["embeddings"], non_blocking=True)
        if use_tracker:
            o["trk"].copy_(bank.read_state(trk_ids), non_blocking=True)
        o["ev"].record()
        face.release_upload(s % 3, o["ev"])

    def read_result(s):
        o = out_host[s % 2]
        o["ev"].synchronize()
        return int(o["counts"].sum()) + float(o["emb"][0, 0]) + float(o["trk"][0, 4])   # touch the data on the host

    def run_e2e(n_total):
        upload(0)
        for s in range(n_total):
            step_e2e(s, n_total)
            if s > 0:
                read_result(s - 1)                # results are consumed on the host one step behind
        read_result(n_total - 1)

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    # ---------------- device-resident timing (value) ----------------
    for s in range(args.warmup):
        step_resident(s)
    sync_all()
    if args.ncu_step:
        overlap[0] = False
        torch.cuda.profiler.start()
        step_resident(args.warmup)
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.stop()
        return
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    res = None
    t_host = time.perf_counter()
    host_ms = None
    n_host = min(4, args.steps)
    for s in range(args.steps):
        res = step_resident(args.warmup + s)
        if s + 1 == n_host:
            # time the host needs to enqueue one step, taken over the first steps only: later the launch queue is full and
            # the host simply waits for the GPU
            host_ms = 1000.0 * (time.perf_counter() - t_host) / n_host
    if world > 1:
        # the path's one exchange: all-gather of the per-rank embeddings before clustering
        embs = res["embeddings"].contiguous()
        gathered = [torch.empty_like(embs) for _ in range(world)]
        dist.all_gather(gathered, embs)
    e1.record()
    sync_all()
    ms = e0.elapsed_time(e1)
    launches = _lib.launch_count() - l0
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    det0.check()
    face.face_recognition_.check()
    if os.environ.get("PV_BENCH_DEBUG") and use_tracker:
        st_ = bank.read_state(trk_ids).float().cpu()
        wd_ = st_[:, 2] - st_[:, 0]
        sys.stderr.write("[bench debug] tracker state after the resident leg: |coord| max %.4g, width %.4g..%.4g, psr %.4g..%.4g, finite %s\n"
                         % (float(st_[:, :4].abs().max()), float(wd_.min()), float(wd_.max()), float(st_[:, 4].min()),
                            float(st_[:, 4].max()), bool(torch.isfinite(st_).all())))
    if args.dump_outputs and rank == 0:
        # the detector's boxes / scores are padded to MAX_DET per frame; slots past a frame's count hold stale data
        kept = torch.arange(det0.MAX_DET, device=dev)[None, :] < res["det_counts"].clamp(max=det0.MAX_DET)[:, None]
        outs = dict(det_boxes=torch.where(kept[..., None], res["det_boxes"], 0),
                    det_scores=torch.where(kept, res["det_scores"], 0.0),
                    det_counts=res["det_counts"], landmarks=res["landmarks"], embeddings=res["embeddings"])
        if use_tracker:
            outs["tracker_state"] = bank.read_state(trk_ids)
        dump_outputs(args.dump_outputs, {k: v.cpu().numpy() for k, v in outs.items()})

    # ---------------- end-to-end timing (host buffers, H2D + D2H inside) ----------------
    run_e2e(min(max(args.warmup, 1), 2))
    sync_all()
    e2e_steps = max(4, args.steps // 2)
    torch.cuda.synchronize(dev)
    e0.record()
    run_e2e(e2e_steps)
    e1.record()
    sync_all()
    ms_e2e = e0.elapsed_time(e1)
    t = torch.tensor([ms_e2e], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_e2e = float(t.item())
    if rank == 0:
        sampler.stop_flag = True
        sampler.join(timeout=3)

    # ---------------- roofline leg: CUDA events around every tensor-core conv launch and every stage ----------------
    # Dominant kernel family = rsconv_kernel (detector convs 2..7, csrc/rsconv.cu): achieved = algorithmic FLOPs of those
    # six layers / their summed launch time.  conv1_fused, the embedder's srgemm launches and the tracker bank are reported
    # beside it.  One un-timed instrumented step runs first (the first instrumented call after a sync absorbs host latency).
    roof = None
    if rank == 0 and args.profile_convs > 0:
        net = face.face_recognition_
        det_names = list(det0.layer_names)           # "conv1+2" = conv1 and conv2 in one launch (csrc/c12.cu)
        conv_ops = [(n, op) for n, (op, _) in zip(det_names, det0.convs)] + [("embed", op) for op, _ in net.conv_ops()]
        evs = []
        orig = {}
        for name, op in conv_ops:
            orig[id(op)] = op.run

            def timed_run(q_rows=None, _name=name, _run=op.run):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                _run(q_rows)
                b.record()
                evs.append((_name, a, b))
            op.run = timed_run
        stage_ev = {}

        def timed_stage(name, fn):
            def wrapped(*a, **k):
                e_a, e_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e_a.record()
                r = fn(*a, **k)
                e_b.record()
                stage_ev.setdefault(name, []).append((e_a, e_b))
                return r
            return wrapped

        patched = [(det0, "build_plane", "pyramid"), (det0, "forward_scores", "convs+shift_sum"), (det0, "decode", "decode+nms"),
                   (face.shape_predictor_, "predict", "landmarks"), (face._chipper, "extract", "chips"),
                   (net, "forward_chips", "embed")]
        if use_tracker:
            patched.append((bank, "update_batch", "tracker"))
        saved = [(o, n, getattr(o, n)) for o, n, _ in patched]
        for o, n, label in patched:
            setattr(o, n, timed_stage(label, getattr(o, n)))
        overlap[0] = False
        ev_a, ev_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        step_resident(0)                                     # un-timed instrumented step (warms the patched path)
        torch.cuda.synchronize(dev)
        evs.clear()
        stage_ev.clear()
        ev_a.record()
        for s in range(args.profile_convs):
            step_resident(1 + s)
        ev_b.record()
        torch.cuda.synchronize(dev)
        serial_ms = ev_a.elapsed_time(ev_b) / args.profile_convs
        overlap[0] = True
        for o, n, f in saved:
            setattr(o, n, f)
        for name, op in conv_ops:
            op.run = orig[id(op)]
        P = args.profile_convs
        stage_ms = {k: sum(a.elapsed_time(b) for a, b in v) / max(1, P) for k, v in stage_ev.items()}
        layer_ms = {}
        for name, a, b in evs:
            layer_ms[name] = layer_ms.get(name, 0.0) + a.elapsed_time(b) / P
        layer_flops = {n: B * f for n, f in zip(det_names, det0.algorithmic_flops_per_op)}   # per pyramid pixel, padding excluded
        layer_flops["embed"] = B * FACES_PER_FRAME * net.flops_per_face
        peaks = load_peaks()
        peak = peaks["tf_sustained"]
        layers = {n: dict(ms=round(layer_ms[n], 4), tflops=round(layer_flops[n] / (layer_ms[n] * 1e-3) / 1e12, 1),
                          frac=round(layer_flops[n] / (layer_ms[n] * 1e-3) / 1e12 / peak, 4)) for n in layer_ms}
        dom = [n for n in det_names if n not in ("conv1", "conv1+2")]      # the rsconv_kernel launches
        dom_ms = sum(layer_ms[n] for n in dom)
        dom_fl = sum(layer_flops[n] for n in dom)
        all_ms = sum(layer_ms.values())
        all_fl = sum(layer_flops.values())
        traffic, traffic_source = None, None
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as f:
                tj = json.load(f)
            tj_layers = tj.get("layers", ["conv%d" % i for i in range(2, 8)])
            if (tj.get("plane") == [det0.geo.plane_h, det0.geo.plane_w] and tj.get("impl", "detconv") == det0.conv_impl
                    and tj_layers == dom):
                traffic = tj["detconv_dram_bytes_per_frame"] * B
                traffic_source = ("static: dram__bytes_read+write of the six rsconv launches from the committed ncu --set full "
                                  "capture (profiles/ncu_traffic.json: %s), x frames per step; not measured in this run"
                                  % tj.get("source", "r01"))
        achieved = dom_fl / (dom_ms * 1e-3) / 1e12
        roof = dict(bound="tensor", achieved=achieved, peak=peak, unit="TFLOP/s", frac=achieved / peak, traffic=traffic,
                    traffic_source=traffic_source, peak_source=peaks["source"],
                    kernel="rsconv_kernel (detector %s, %d launches/step)" % ("convs " + dom[0][4:] + "..7", len(dom)),
                    kernel_ms_per_step=round(dom_ms, 4), algorithmic_flops_per_step=dom_fl,
                    all_convs=dict(ms_per_step=round(all_ms, 4), tflops=round(all_fl / (all_ms * 1e-3) / 1e12, 1),
                                   frac=round(all_fl / (all_ms * 1e-3) / 1e12 / peak, 4), launches_per_step=len(evs) // P),
                    layers=layers, stage_ms_per_step={k: round(v, 3) for k, v in stage_ms.items()},
                    serial_step_ms=round(serial_ms, 3))
        if use_tracker and "tracker" in stage_ms:
            ups = n_tracks / (stage_ms["tracker"] * 1e-3)
            roof["tracker"] = dict(bound="hbm", updates_per_step=n_tracks, ms=round(stage_ms["tracker"], 3),
                                   updates_per_s=round(ups), achieved=round(ups * TRACKER_BYTES_PER_UPDATE / 1e9, 1),
                                   peak=peaks["hbm_gbs"], unit="GB/s",
                                   frac=round(ups * TRACKER_BYTES_PER_UPDATE / 1e9 / peaks["hbm_gbs"], 4),
                                   algorithmic_bytes_per_update=TRACKER_BYTES_PER_UPDATE)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    frames_total = args.steps * B * world
    value = frames_total / (ms_max * 1e-3)
    e2e_value = e2e_steps * B * world / (ms_e2e * 1e-3)
    h2d = B * H * W * 3 + B * FACES_PER_FRAME * (16 + 4)
    d2h = B * det0.MAX_DET * 16 + B * 4 + B * FACES_PER_FRAME * (68 * 2 * 4 + 128 * 4) + (n_tracks * 20 if use_tracker else 0)

    cpu = None
    if not args.no_cpu_baseline:
        from oracle import cpu_ref
        models = (det_m, sp_m, emb_m)
        cores = cpu_ref.host_cores()
        el1, _, n1 = cpu_sample(models, 1, 2)
        el_n, used, n_all = cpu_sample(models, cores, 4 * cores)
        cpu = dict(value=n_all / el_n, unit="frames/s", cores=used, kind="port",
                   sample="%d x 1080p frames (%d independent streams, one host thread each: detect + %d tracker updates + %d "
                          "faces per frame) through the C++ restatement oracle/cpu (-O3 -march=native), %.1f s"
                          % (n_all, used, 2 * TRACKS_PER_STREAM, FACES_PER_FRAME, el_n),
                   single_thread=dict(value=n1 / el1, cores=1, sample="%d frames, %.1f s" % (n1, el1)),
                   core_scaling=round((n_all / el_n) / (n1 / el1), 2), host_threads_visible=os.cpu_count(),
                   cores_note="usable cores = min(online CPUs, cgroup cpu.max quota)")

    line = dict(metric=METRIC, value=value, unit="frames/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
                ms_per_step=ms_max / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="bf16",
                data="synthetic",
                config=dict(workload=WORKLOAD, frames_per_step=B, faces_per_frame=FACES_PER_FRAME,
                            tracker_updates_per_frame=(2 * TRACKS_PER_STREAM if use_tracker else 0),
                            streams="%d concurrent shot streams per GPU, one frame each per step" % B,
                            parallelism="frame-shard x%d" % world,
                            l2="%d distinct input batches (%d MB) + ~1.4 GB/frame of plane and activation traffic per step: "
                               "inputs larger than L2" % (N_TIMES, N_TIMES * B * H * W * 3 // 1000000)),
                clocks=sampler.summary(),
                e2e=dict(value=e2e_value, unit="frames/s", h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h, steps=e2e_steps,
                         api="Face.upload (pinned host -> staging ring) + Face.extract_batch + DetectorNet.detect + "
                             "TrackerBank.update_batch, results to pinned host memory"),
                gpu_launches=int(launches), host_enqueue_ms_per_step=round(host_ms, 3),
                roofline=roof, cpu_baseline=cpu)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main_guarded():
    """Single-GPU runs execute the measurement in a child process and repeat it (at most twice) if the child dies:
    one of seven otherwise identical runs of this round aborted with a CUDA illegal-address error in the e2e leg
    (profiles/README.md, gpurun #84; not reproduced since, root cause open — the chip / tracker samplers were hardened
    against non-finite coordinates afterwards).  A repeat is reported in the JSON line as "retries".  Multi-rank
    (torchrun) runs, --impl reference and PV_BENCH_NO_RETRY=1 run in-process."""
    if (int(os.environ.get("WORLD_SIZE", "1")) > 1 or "--impl" in sys.argv or os.environ.get("PV_BENCH_NO_RETRY")
            or os.environ.get("PV_BENCH_CHILD")):
        return main()
    env = dict(os.environ, PV_BENCH_CHILD="1")
    try:                                     # build once here (the child finds the library up to date) and map it in this process too
        import __graft_entry__ as ge
        ge.build()
    except Exception as e:  # noqa: BLE001
        sys.stderr.write("bench.py: build failed in the parent process: %r\n" % (e, ))
    for attempt in range(3):
        r = subprocess.run([sys.executable, os.path.abspath(__file__)] + sys.argv[1:], env=env, stdout=subprocess.PIPE, text=True)
        lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
        if r.returncode == 0 and lines:
            line = json.loads(lines[-1])
            line["retries"] = attempt
            print(json.dumps(line), flush=True)
            return
        if r.returncode >= 0 and r.returncode != 134:
            sys.stdout.write(r.stdout)                     # an ordinary failure (no device, bad arguments): not repeated
            raise SystemExit(r.returncode)
        sys.stderr.write("bench.py: attempt %d died (exit code %d); repeating\n" % (attempt + 1, r.returncode))
    raise SystemExit("bench.py: the measurement died three times")


if __name__ == "__main__":
    main_guarded()
