"""CPU: the shot-threading oracle pinned against cv2 (FAST, Harris, angles, rBRIEF with the recovered pattern, the
pyramid and blur restatements, the match count), host geometry, the graph work against the reference's golden
output, the Annotation additions, ArrayVideo.__call__ and the thread / scene CLI."""
import json
import os
import re
import sys

import cv2
import numpy as np
import pytest
import torch

from oracle import thread as O
from pyannote_video_b200 import thread as T
from pyannote_video_b200.annotation import Annotation, Segment, string_generator
from pyannote_video_b200.cli import ArrayVideo, main, load_annotation, write_annotation

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import thread_scenario as sc  # noqa: E402

GOLDEN = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "thread_golden.json")))


def _frames():
    rng = np.random.default_rng(7)
    out = [rng.integers(0, 256, (200, 355), dtype=np.uint8), rng.integers(0, 256, (131, 97), dtype=np.uint8)]
    for name in ("abab", "overseg"):
        frames, _ = sc.make_clip(name)
        out.append(O.cv2_gray(frames[30], O.resize_dsize((frames.shape[2], frames.shape[1]), 200)))
    tile = np.random.default_rng(0).integers(0, 256, (10, 10, 3), dtype=np.uint8)
    out.append(O.cv2_gray(np.tile(tile, (20, 24, 1)), O.resize_dsize((240, 200), 200)))
    return out


def test_tie_frame_keeps_more_than_the_quota():
    kc, _ = O.cv2_orb(_frames()[4])
    assert np.sum(kc[:, 2] == 0) > O.level_quotas()[0]


@pytest.mark.parametrize("k", range(5))
def test_orb_restatement_matches_cv2(k):
    gray = _frames()[k]
    kp, d = O.orb(gray)
    kc, dc = O.cv2_orb(gray)
    assert len(kp) == len(kc)
    assert O.as_set(kp, d) == O.as_set(kc, dc)


@pytest.mark.parametrize("shape", [(333, 200), (200, 333), (345, 200), (369, 200), (414, 200)])
def test_orb_restatement_at_float32_rounding_sizes(shape):
    """row / column counts whose level sizes round differently with a float64 division (cv2 divides in float32)"""
    gray = np.random.default_rng(shape[0] * 1000 + shape[1]).integers(0, 256, shape, dtype=np.uint8)
    kp, d = O.orb(gray)
    kc, dc = O.cv2_orb(gray)
    assert O.as_set(kp, d) == O.as_set(kc, dc)
    assert T.level_sizes(*shape) == O.level_sizes(*shape)


def test_level_sizes_divide_in_float32():
    # 369 / 1.2^k: the float32 and float64 quotients round to different integers at some level
    f64 = [int(np.rint(369 / O.SCALE_FACTOR ** k)) for k in range(O.N_LEVELS)]
    assert [r for r, _ in O.level_sizes(369, 200)] != f64
    assert all(isinstance(s, np.float32) for s in O.level_scales())


def test_kernel_patch_table_equals_oracle_umax():
    src = open(os.path.join(os.path.dirname(O.PATTERN_H), "orb.cu")).read()
    body = re.search(r"c_umax\[[^]]*\]\s*=\s*\{([^}]*)\}", src).group(1)
    assert [int(v) for v in body.split(",")] == O.umax()


def test_fast_keypoints_match_cv2():
    for gray in _frames():
        x, y, s = O.fast_keypoints(gray)
        det = cv2.FastFeatureDetector_create(20, True, cv2.FAST_FEATURE_DETECTOR_TYPE_9_16).detect(gray)
        assert set(zip(x.tolist(), y.tolist(), s.astype(float).tolist())) == \
            {(int(p.pt[0]), int(p.pt[1]), p.response) for p in det}


def test_fast_atan2_matches_cv2():
    rng = np.random.default_rng(0)
    vals = np.concatenate([rng.integers(-400000, 400000, (5000, 2)), rng.integers(-50, 50, (5000, 2)),
                           [[0, 0], [0, 5], [5, 0], [-5, 0], [0, -5], [3, 3], [-3, -3]]])
    for y, x in vals.astype(np.float32):
        assert O.fast_atan2(y, x) == np.float32(cv2.fastAtan2(float(y), float(x)))


def test_pyramid_and_blur_restatements():
    rng = np.random.default_rng(3)
    for r, c in [(355, 200), (200, 355), (57, 99), (333, 517)]:
        img = rng.integers(0, 256, (r, c), dtype=np.uint8)
        assert np.array_equal(O.orb_blur_restated(img), O.orb_blur(img))
        prev = img
        for rr, cc in O.level_sizes(r, c)[1:]:
            want = cv2.resize(prev, (cc, rr), interpolation=cv2.INTER_LINEAR_EXACT)
            assert np.array_equal(O.resize_exact(prev, rr, cc), want)
            prev = want


def test_descriptors_at_random_rotated_keypoints():
    """proves the recovered pattern table: cv2.ORB.compute keeps the given angles"""
    rng = np.random.default_rng(5)
    img = O.orb_blur(rng.integers(0, 256, (240, 320), dtype=np.uint8))
    img = (img.astype(np.int32) * 3 % 256).astype(np.uint8)
    pts = [cv2.KeyPoint(float(rng.integers(40, 280)), float(rng.integers(40, 200)), 31,
                        float(np.float32(rng.uniform(0, 360))), 0, 0) for _ in range(400)]
    pts.append(cv2.KeyPoint(100.0, 100.0, 31, 0.0, 0, 0))
    kps, desc = cv2.ORB_create().compute(img, pts)
    blurred = O.orb_blur(img)
    pat = O.pattern()
    assert kps[-1].angle == 0
    for k, d in zip(kps, desc):
        got = O.brief(blurred, int(k.pt[0]), int(k.pt[1]), np.float32(k.angle), pat)
        assert np.array_equal(got, d)


def test_harris_and_angle_at_cv2_keypoints():
    gray = _frames()[0]
    levels = O.pyramid(gray)
    kc, _ = O.cv2_orb(gray)
    for x, y, lv, resp, ang in kc:
        lv = int(lv)
        s = np.float32(O.SCALE_FACTOR ** lv)
        inv = np.float32(1) / s
        cx, cy = int(np.rint(np.float32(x) * inv)), int(np.rint(np.float32(y) * inv))
        assert O.harris(levels[lv], [cx], [cy])[0] == np.float32(resp)
        assert O.ic_angle(levels[lv], cx, cy) == np.float32(ang)


def test_match_count_equals_bf_ratio_test():
    rng = np.random.default_rng(9)
    for trial in range(30):
        nq, nt = rng.integers(2, 60, 2)
        base = rng.integers(0, 256, (4, 32), dtype=np.uint8)
        q = base[rng.integers(0, 4, nq)] ^ (rng.random((nq, 32)) < 0.1).astype(np.uint8) * rng.integers(0, 256, (nq, 32), dtype=np.uint8)
        t = base[rng.integers(0, 4, nt)] ^ (rng.random((nt, 32)) < 0.1).astype(np.uint8) * rng.integers(0, 256, (nt, 32), dtype=np.uint8)
        t[:2] = q[0]                                            # equal best and second distances
        assert O.match_count(q, t) == O.cv2_bf_count(q, t)
    # second distances that are multiples of 10: d1 = 7, d2 = 10 is not a match (0.7 * 10 rounds to 7.0)
    q = np.zeros((2, 32), np.uint8)
    t = np.zeros((2, 32), np.uint8)
    t[0, 0] = 0x7F
    t[1, :2] = (0xFF, 0x03)
    assert O.match_count(q, t) == O.cv2_bf_count(q, t)
    assert O.match_count(q[:1], t) == 0


def test_host_geometry_matches_oracle():
    for rows, cols in [(355, 200), (200, 355), (113, 200)]:
        g, tab = T.make_geometry(rows, cols)
        sizes = O.level_sizes(rows, cols)
        assert [(g.rows[k], g.cols[k]) for k in range(8)] == sizes
        assert list(g.quota) == O.level_quotas() == [109, 90, 75, 63, 52, 44, 36, 31]
        assert np.array_equal(np.array(g.gauss, np.float32), cv2.getGaussianKernel(7, 2, cv2.CV_32F).ravel())
        assert [g.scale[k] for k in range(8)] == [float(np.float32(O.SCALE_FACTOR ** k)) for k in range(8)]
        for k in range(1, 8):
            xo, xc = O.linear_exact_taps(sizes[k - 1][1], sizes[k][1])
            o = g.tab_off[k]
            assert np.array_equal(tab[o:o + len(xo)], xo) and np.array_equal(tab[o + len(xo):o + 2 * len(xo)], xc)


def test_resize_shape_matches_reference_quirk():
    assert T.resize_shape((1920, 1080), 200) == (355, 200)
    assert O.resize_dsize((1920, 1080), 200) == (200, 355)


# ---------------------------------------------------------------------------------------------------- graph work
def test_lookahead_pairs_equal_reference_product_lookahead():
    for item in GOLDEN["product_lookahead"]:
        got = T.lookahead_pairs(item["n"], item["lookahead"])
        assert sorted(got) == sorted(map(tuple, item["pairs"]))
        assert len(got) == len(item["pairs"])


@pytest.mark.parametrize("name", sorted(GOLDEN["clips"]))
def test_threads_and_scenes_from_golden_edges(name):
    g = GOLDEN["clips"][name]
    shots = [Segment(*s) for s in g["shots"]]
    threads = T.thread_annotation(shots, [tuple(e) for e in g["edges"]])
    assert [[s.start, s.end, l] for s, _, l in threads.itertracks(yield_label=True)] == g["threads"]
    scenes = T.scenes(threads)
    assert [[s.start, s.end, l] for s, _, l in scenes.itertracks(yield_label=True)] == g["scenes"]


def test_scenario_clips_are_the_golden_ones():
    for name, g in GOLDEN["clips"].items():
        frames, segs = sc.make_clip(name)
        assert sc.sha256(frames) == g["sha256"]
        assert [list(s) for s in segs] == g["shots"]


def test_biconnected_components_match_networkx():
    nx = pytest.importorskip("networkx")
    rng = np.random.default_rng(2)
    for _ in range(40):
        n = int(rng.integers(2, 14))
        edges = {tuple(sorted(e)) for e in rng.integers(0, n, (int(rng.integers(1, 2 * n)), 2)).tolist() if e[0] != e[1]}
        g = nx.Graph(list(edges))
        want = sorted(sorted(c) for c in nx.biconnected_components(g))
        assert sorted(sorted(c) for c in T.biconnected_components(edges)) == want


def test_components_ordered_by_first_node():
    assert T.components(6, [(4, 5), (0, 2), (2, 4)]) == [[0, 2, 4, 5], [1], [3]]


# ---------------------------------------------------------------------------------------------------- annotation
def test_annotation_segment_key_and_tuple_key():
    a = Annotation()
    a[Segment(0, 1)] = "A"
    assert a[Segment(0, 1)] == "A"
    assert a[Segment(0, 1), "_"] == "A"
    a[(0, 2), "t"] = "B"                                        # tuple keys as before
    assert a[Segment(0, 2), "t"] == "B"
    assert len(a) == 2


def test_annotation_smooth_and_subset():
    a = Annotation()
    a[Segment(0, 1)] = "A"
    a[Segment(1, 2)] = "A"
    a[Segment(2, 3)] = "B"
    a[Segment(3, 4)] = "A"
    s = a.smooth()
    assert [(x.start, x.end, l) for x, _, l in s.itertracks(yield_label=True)] == [(0, 2, "A"), (2, 3, "B"), (3, 4, "A")]
    assert [l for _, _, l in a.subset(["B"]).itertracks(yield_label=True)] == ["B"]


def test_string_generator():
    g = string_generator()
    labels = [next(g) for _ in range(28)]
    assert labels[:3] == ["A", "B", "C"] and labels[25:] == ["Z", "AA", "AB"]


# ---------------------------------------------------------------------------------------------------- video / CLI
def test_array_video_call_index_rule():
    frames = np.arange(10, dtype=np.uint8)[:, None, None, None] * np.ones((1, 4, 6, 3), np.uint8)
    v = ArrayVideo(frames, 25.0)
    assert v(0.0)[0, 0, 0] == 0
    assert v(0.04)[0, 0, 0] == 1                                # int(25 * 0.04 + 1e-5) = 1
    assert v(0.0799)[0, 0, 0] == 1
    assert v(9 / 25.)[0, 0, 0] == 9
    assert v(-0.01)[0, 0, 0] == 0                              # int(-0.25 + 1e-5) truncates to 0
    for t in (-0.2, 10 / 25.):
        with pytest.raises(IOError):
            v(t)
    v.frame_size = (3, 2)
    assert v(0.0).shape == (2, 3, 3)


def test_annotation_json_round_trip(tmp_path):
    a = Annotation()
    a[Segment(0, 1), "A"] = "A"
    a[Segment(1, 3), "B"] = "B"
    p = str(tmp_path / "a.json")
    write_annotation(a, p)
    data = json.load(open(p))
    assert data["pyannote"] == "Annotation"
    assert data["content"][0] == {"segment": {"start": 0.0, "end": 1.0}, "track": "A", "label": "A"}
    assert load_annotation(p) == a


def test_scene_verb_runs_on_cpu(tmp_path):
    g = GOLDEN["clips"]["abab"]
    threads = Annotation()
    for i, (s, e, l) in enumerate(g["threads"]):
        threads[Segment(s, e), str(i)] = l
    src, dst = str(tmp_path / "threads.json"), str(tmp_path / "scenes.json")
    write_annotation(threads, src)
    assert main(["scene", "unused.npy", src, dst]) == 0
    got = [[c["segment"]["start"], c["segment"]["end"], c["label"]] for c in json.load(open(dst))["content"]]
    assert got == g["scenes"]


def test_thread_needs_cuda():
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    frames, segs = sc.make_clip("abab")
    with pytest.raises(RuntimeError):
        T.Thread(ArrayVideo(frames), shot=[Segment(*s) for s in segs])
