"""GPU: shot boundary detection (csrc/shot.cu behind pyannote_video_b200.shot) against the reference golden
(tests/golden/shot_golden.npz) and the numpy oracle (oracle/shot.py), stage by stage, then end to end."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import shot as O
import shot_scenario as sc

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "shot_golden.npz")

# R: the kernel follows the oracle's float32 / float64 operation order with explicitly rounded, unfused operations
# (pre-blur, level resize or 2x2 mean, both passes of the expansion): bit-exact
# flow: the oracle sums the 15 x 15 window as OpenCV does (running float64 sums fed float32 differences), the
# kernel sums each window directly (float32 columns, float64 rows)
FLOW_MEAN_TOL = 5e-3
FLOW_P99_TOL = 5e-2
# DFD vs the reference (cv2 flow): the flows differ in their last bits inside the image and by more near the
# border, so a few int() truncations of x + flow flip; measured with the oracle flow: <= 4.5 % on one pair, median 2 %
DFD_RTOL = 0.08
DFD_MEDIAN_RTOL = 0.02


@pytest.fixture(scope="module")
def golden():
    return np.load(GOLDEN)


def _detector(cuda, name, **kw):
    from pyannote_video_b200.shot import ShotDetector
    H, W = sc.CLIPS[name][:2]
    return ShotDetector((W, H), height=sc.height_of(name), device=cuda, **kw)


def _dfds(cuda, name, batch, **kw):
    det = _detector(cuda, name, **kw)
    frames = torch.from_numpy(sc.make_clip(name)).to(cuda)
    out = [det.dfd_batch(frames[i:i + batch].contiguous()) for i in range(0, len(frames), batch)]
    return torch.cat(out).cpu().numpy(), det


@pytest.mark.parametrize("name", sorted(sc.CLIPS))
def test_gray_resize_bit_exact(cuda, golden, name):
    frames = sc.make_clip(name)
    assert sc.sha256(frames) == str(golden[name + "/sha256"])
    ref = golden[name + "/gray"]
    det = _detector(cuda, name)
    got = det.gray_resize(torch.from_numpy(frames[:len(ref)]).to(cuda)).cpu().numpy()
    assert np.array_equal(got, ref)


# (frames, height): three golden clips (one level; 77 x 50; 177 x 100 = two levels, the coarse one by linear resize)
# and 400 x 704 at height 100 = 176 x 100, whose coarse level 88 x 50 is the exact 2x2 mean
FLOW_CASES = {
    "hd": lambda: (sc.make_clip("hd")[:2], 50),
    "odd": lambda: (sc.make_clip("odd")[:2], 50),
    "h100": lambda: (sc.make_clip("h100")[:2], 100),
    "area2x": lambda: (sc.translating(400, 704, 2, seed=9), 100),
}


@pytest.mark.parametrize("case", sorted(FLOW_CASES))
def test_polyexp_and_flow_against_oracle(cuda, case):
    from pyannote_video_b200.shot import ShotDetector
    frames_np, height = FLOW_CASES[case]()
    H, W = frames_np.shape[1:3]
    det = ShotDetector((W, H), height=height, device=cuda, keep_flow=True)
    if case == "area2x":
        assert det.geo.n_levels == 2 and det.geo.lv[0].area2x == 1 and (det.rows, det.cols) == (176, 100)
    d = det.dfd_batch(torch.from_numpy(frames_np).to(cuda))
    g = det.gray[1:3].cpu().numpy()      # slot 0 holds the carried last frame, slots 1..2 the batch
    R = det.R[1:3].cpu().numpy()
    trace = []
    flow = O.farneback(g[0], g[1], trace=trace)
    assert len(trace) == det.geo.n_levels
    for k, lv in enumerate(trace):
        L = det.geo.lv[k]
        n = 5 * L.rows * L.cols
        for slot, key in ((0, "R0"), (1, "R1")):
            got = R[slot, L.r_off:L.r_off + n].reshape(5, L.rows, L.cols)
            assert np.array_equal(got, lv[key]), (k, key, np.abs(got - lv[key]).max())
    fg = det.flow[0].cpu().numpy()
    e = np.abs(fg - flow)
    assert e.mean() < FLOW_MEAN_TOL and np.quantile(e, 0.99) < FLOW_P99_TOL, (e.mean(), np.quantile(e, 0.99), e.max())
    assert np.isfinite(d.cpu().numpy()).all()


@pytest.mark.parametrize("name", sorted(sc.CLIPS))
def test_dfd_and_segments_match_reference(cuda, golden, name):
    from pyannote_video_b200 import Shot
    from pyannote_video_b200.cli import ArrayVideo
    frames = sc.make_clip(name)
    video = ArrayVideo(frames, 25.0)
    shot = Shot(video, height=sc.height_of(name), device=cuda)
    tds = list(shot.iter_dfd())
    t = np.array([a for a, _ in tds])
    d = np.array([b for _, b in tds])
    ref = golden[name + "/dfd"]
    assert np.array_equal(t, golden[name + "/t"])
    rel = np.abs(d - ref) / np.maximum(ref, 1e-12)
    rel[(ref == 0) & (d == 0)] = 0.0
    assert rel.max() <= DFD_RTOL and np.median(rel) <= DFD_MEDIAN_RTOL, (rel.max(), np.median(rel))
    segs = np.array([(s.start, s.end) for s in shot], np.float64).reshape(-1, 2)
    assert np.array_equal(segs, golden[name + "/segments"])


@pytest.mark.parametrize("name", ["sd", "h100", "static_cut"])
def test_dfds_do_not_depend_on_batching(cuda, name):
    T = sc.CLIPS[name][2]
    whole, _ = _dfds(cuda, name, T)
    assert len(whole) == T - 1
    for b in (1, 7):
        got, _ = _dfds(cuda, name, b)
        assert np.array_equal(got, whole), b


def _clip_with_cuts():
    return sc.make_clip("sd")                 # 360 x 640, cuts at frames 50 and 110 (2.0 s and 4.4 s)


def _detector_model(frames, n_keep=30):
    """seeded CNN detector whose threshold keeps the n_keep best-scoring cells of the first frame (scores from the
    CPU oracle), so the texture clip gives detections and therefore tracks"""
    from oracle import cpu_ref
    from pyannote_video_b200 import weights as W
    det = W.make_detector(seed=2, score_bias=0.0)
    cpu_ref.set_threads(0)
    o = cpu_ref.Detector(det, bf16=True)
    plane, _ = o.build_plane(frames[0], 1)
    sc_ = o.scores(plane)
    det["adjust_threshold"] = float(np.quantile(sc_, 1 - float(n_keep) / sc_.size))
    return det


def _inside_one_shot(ts, shots):
    return any(s.start <= min(ts) and max(ts) <= s.end for s in shots)


def test_shot_then_face_tracking(cuda):
    from pyannote_video_b200 import Shot, FaceTracking
    from pyannote_video_b200.cli import ArrayVideo
    from pyannote_video_b200.face import Face
    frames = _clip_with_cuts()
    video = ArrayVideo(frames, 25.0)
    shots = list(Shot(video, device=cuda, batch=16))
    assert [round(s.start, 3) for s in shots] == [0.0, 2.0, 4.4]
    assert shots[-1].end == pytest.approx(video.end)
    face = Face(detector=_detector_model(frames), device=cuda)
    tracks = list(FaceTracking(face=face, track_min_confidence=3.0, track_max_gap=0.0)(video, shots))
    assert len(tracks) >= 2
    for trk in tracks:                        # no track crosses a shot boundary
        assert _inside_one_shot([t for t, _, _ in trk], shots)


def test_cli_shot_then_track(cuda, tmp_path):
    from pyannote_video_b200 import cli
    npy = str(tmp_path / "clip.npy")
    np.save(npy, _clip_with_cuts())
    shots = str(tmp_path / "shots.json")
    assert cli.main(["shot", npy, shots]) == 0
    data = json.load(open(shots))
    assert data["pyannote"] == "Timeline" and [round(s["start"], 3) for s in data["content"]] == [0.0, 2.0, 4.4]
    from pyannote_video_b200 import weights as W
    model = str(tmp_path / "det.npz")
    W.save_model(model, _detector_model(np.load(npy)))
    out = str(tmp_path / "out.track.txt")
    assert cli.main(["--detector", model, "track", "--min-confidence", "3", "--max-gap", "0", npy, shots, out]) == 0
    rows = cli.read_track_file(out)
    assert len(rows) > 10
    segs = cli.load_shots(shots)
    for ident in {r[1] for r in rows}:
        assert _inside_one_shot([r[0] for r in rows if r[1] == ident], segs)


def test_detector_runs_on_its_own_device_and_rejects_others(cuda):
    """launches happen on the detector's device whatever the current device is; frames elsewhere are refused"""
    from pyannote_video_b200.shot import ShotDetector
    frames = torch.from_numpy(sc.make_clip("odd")[:6]).to(cuda)
    H, W = frames.shape[1:3]
    ref = ShotDetector((W, H), device=cuda).dfd_batch(frames).cpu().numpy()
    det = ShotDetector((W, H), device="cuda")
    assert det.device == torch.device("cuda", torch.cuda.current_device())
    with pytest.raises(RuntimeError, match="frames are on cpu"):
        det.dfd_batch(frames.cpu())
    if torch.cuda.device_count() > 1:
        other = torch.device("cuda", 1)
        with pytest.raises(RuntimeError, match="frames are on"):
            det.dfd_batch(frames.to(other))
        det1 = ShotDetector((W, H), device=other)
        with torch.cuda.device(0):
            got = det1.dfd_batch(frames.to(other)).cpu().numpy()
        assert np.array_equal(got, ref)
