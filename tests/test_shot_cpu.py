"""Shot boundary detection on the CPU: the oracle against the reference golden (tests/golden/shot_golden.npz, made by
tests/golden/make_shot_golden.py from the reference's own Shot), the numpy Farneback against cv2, the median filter
against scipy, the gray + resize tables against cv2, the segmentation rules and the CLI plumbing."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import shot as O
from pyannote_video_b200 import shot as S
from pyannote_video_b200.annotation import Segment
import shot_scenario as sc

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "shot_golden.npz")

# numpy Farneback vs cv2 on the stored first flow of a clip: the interior agrees to float rounding, the five
# outermost pixels of the update-matrix weighting and the box window around them differ more
FLOW_MEAN_TOL = 0.02
FLOW_P99_TOL = 0.25


@pytest.fixture(scope="module")
def golden():
    return np.load(GOLDEN)


def test_scenario_generator_is_deterministic(golden):
    for name in sc.CLIPS:
        assert sc.sha256(sc.make_clip(name)) == str(golden[name + "/sha256"]), name


@pytest.mark.parametrize("name", sorted(sc.CLIPS))
def test_oracle_reproduces_reference_dfds_and_segments(golden, name):
    pytest.importorskip("cv2")
    frames = sc.make_clip(name)
    gray, dfd = O.reference_dfds(frames, sc.height_of(name))
    assert np.array_equal(gray[:len(golden[name + "/gray"])], golden[name + "/gray"])
    assert np.array_equal(dfd, golden[name + "/dfd"])
    T = len(frames)
    segs = list(S.segments(golden[name + "/t"], dfd, S.kernel_size(2.0, 1 / 25.0), 1.0, 0.0, T / 25.0))
    assert np.array_equal(np.array(segs, np.float64).reshape(-1, 2), golden[name + "/segments"])


@pytest.mark.parametrize("name", ["hd", "odd", "h100"])
def test_numpy_farneback_against_cv2(golden, name):
    g = golden[name + "/gray"]
    flow = O.farneback(g[0], g[1])
    d = np.abs(flow - golden[name + "/flow"][0])
    assert d.mean() < FLOW_MEAN_TOL and np.quantile(d, 0.99) < FLOW_P99_TOL, (d.mean(), np.quantile(d, 0.99), d.max())


def test_gray_table_formula_matches_cv2():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(0)
    for (H, W), height in [((1080, 1920), 50), ((333, 517), 50), ((101, 203), 100), ((360, 640), 100), ((64, 40), 50)]:
        rgb = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        rows, cols = S.resize_shape((W, H), height)
        tab = S.gray_table((W, H), rows, cols).astype(np.int64)
        x0, x1, cx0, cx1 = tab[:4 * cols].reshape(4, cols)
        y0, y1, cy0, cy1 = tab[4 * cols:].reshape(4, rows)
        r, g, b = (rgb[..., c].astype(np.int64) for c in range(3))
        gray = (r * 9798 + g * 19235 + b * 3735 + (1 << 14)) >> 15
        hs = gray[:, x0] * cx0 + gray[:, x1] * cx1
        s0, s1 = hs[y0], hs[y1]
        ours = ((((s0 >> 4) * cy0[:, None]) >> 16) + (((s1 >> 4) * cy1[:, None]) >> 16) + 2) >> 2
        assert np.array_equal(ours, O.cv2_convert(rgb, height)), (H, W, height)


def test_medfilt_equals_scipy():
    signal = pytest.importorskip("scipy.signal")
    rng = np.random.default_rng(1)
    for n, k in [(1, 3), (5, 51), (60, 51), (200, 3), (37, 9)]:
        y = rng.random(n) * 10
        y[rng.random(n) < 0.2] = 0.0
        assert np.array_equal(S.medfilt(y, k), signal.medfilt(y, kernel_size=k))


def test_kernel_size_and_resize_rules():
    assert S.kernel_size(2.0, 1 / 25.0) == 51
    assert S.kernel_size(2.0, 1 / 30.0) == 61
    assert S.kernel_size(0.01, 1 / 25.0) == 3
    assert S.kernel_size(2.0, 1 / 24.0) == 49
    assert S.resize_shape((1920, 1080), 50) == (88, 50)
    assert S.resize_shape((1920, 1080), 100) == (177, 100)
    assert S.resize_shape((517, 333), 50) == (77, 50)
    assert [s[:2] for s in S.pyramid_sizes(88, 50)] == [(88, 50)]
    assert [s[:2] for s in S.pyramid_sizes(176, 100)] == [(88, 50), (176, 100)]
    assert [s[:2] for s in S.pyramid_sizes(88, 50)] == [s[:2] for s in O.pyramid_sizes(88, 50)]
    geo, tab = S.make_geometry(177, 100)
    assert geo.n_levels == 2 and geo.lv[1].rows == 177 and geo.lv[0].rows == 88 and geo.lv[0].area2x == 0


def _segs(y, threshold=1.0, k=3, end=None):
    t = [0.04 * (i + 1) for i in range(len(y))]
    end = 0.04 * (len(y) + 1) if end is None else end
    return [(round(s.start, 6), round(s.end, 6)) for s in S.segments(t, np.asarray(y, float), k, threshold, 0.0, end)]


def test_segmentation_edge_cases():
    base = [1.0] * 12
    # a single spike at index 5 -> one boundary at t[5]
    y = list(base); y[5] = 5.0
    assert _segs(y) == [(0.0, 0.24), (0.24, 0.52)]
    # a run 5, 6, 7 keeps only its first element
    y = list(base); y[5] = y[6] = y[7] = 9.0
    assert _segs(y, k=9) == [(0.0, 0.24), (0.24, 0.52)]
    # index 1 directly follows the tracker's initial 0: never a boundary, even when index 0 is not over threshold
    y = list(base); y[1] = 9.0
    assert _segs(y) == [(0.0, 0.52)]
    # index 0 is a boundary
    y = list(base); y[0] = 9.0
    assert _segs(y)[0] == (0.0, 0.04)
    # all zeros: 0 / 0 = NaN, no boundary; one non-zero among zeros: x / 0 = inf, a boundary
    assert _segs([0.0] * 10) == [(0.0, 0.44)]
    y = [0.0] * 10; y[4] = 3.0
    assert _segs(y) == [(0.0, 0.2), (0.2, 0.44)]
    # a boundary on the last pair whose time equals the video end: the empty tail is not yielded
    y = list(base); y[-1] = 9.0
    assert _segs(y, end=0.48) == [(0.0, 0.48)]
    # fewer than two frames: one segment over the video (the reference raises on the empty zip)
    assert _segs([], end=0.04) == [(0.0, 0.04)]
    assert _segs([], end=0.0) == []


def test_segments_are_pyannote_segments():
    out = list(S.segments([0.04, 0.08], np.array([1.0, 1.0]), 3, 1.0, 0.0, 0.12))
    assert out == [Segment(0.0, 0.12)] and isinstance(out[0], Segment)


def test_array_video_has_reference_video_attributes():
    from pyannote_video_b200.cli import ArrayVideo
    v = ArrayVideo(np.zeros((10, 6, 8, 3), np.uint8), 25.0)
    assert v._size == (8, 6) and v.step == pytest.approx(0.04) and v.start == 0.0 and v.end == pytest.approx(0.4)


def test_cli_shot_parsing_and_timeline_roundtrip(tmp_path, monkeypatch):
    from pyannote_video_b200 import cli
    seen = {}

    def fake(video, output, height=50, window=2.0, threshold=1.0):
        seen.update(video=video, output=output, height=height, window=window, threshold=threshold)
        return cli.write_timeline([Segment(0.0, 1.2), Segment(1.2, 3.0)], output)

    monkeypatch.setattr(cli, "shot_cmd", fake)
    monkeypatch.setattr(cli, "open_video", lambda spec, fr: (spec, fr))
    out = str(tmp_path / "shots.json")
    assert cli.main(["shot", "--height", "100", "--window", "3.5", "--threshold", "0.5", "v.npy", out]) == 0
    assert seen == dict(video=("v.npy", 25.0), output=out, height=100, window=3.5, threshold=0.5)
    assert json.load(open(out)) == {"pyannote": "Timeline", "content": [{"start": 0.0, "end": 1.2}, {"start": 1.2, "end": 3.0}]}
    assert [(s.start, s.end) for s in cli.load_shots(out)] == [(0.0, 1.2), (1.2, 3.0)]
    assert cli.main(["shot", "v.npy", out]) == 0
    assert (seen["height"], seen["window"], seen["threshold"]) == (50, 2.0, 1.0)


def test_shot_raises_without_device():
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from pyannote_video_b200 import Shot
    from pyannote_video_b200.cli import ArrayVideo
    with pytest.raises(RuntimeError):
        Shot(ArrayVideo(np.zeros((3, 36, 64, 3), np.uint8)))


def test_detector_refuses_frames_on_another_device():
    """the device check runs before anything touches a GPU: frames must live on the detector's device"""
    from pyannote_video_b200.shot import ShotDetector
    det = ShotDetector.__new__(ShotDetector)
    det.device = torch.device("cuda", 1)
    det.frame_size = (64, 36)
    frames = torch.zeros((2, 36, 64, 3), dtype=torch.uint8)
    with pytest.raises(RuntimeError, match=r"frames are on cpu, the detector on cuda:1"):
        det.dfd_batch(frames)
    with pytest.raises(RuntimeError, match=r"frames are on cpu, the detector on cuda:1"):
        det.gray_resize(frames)
