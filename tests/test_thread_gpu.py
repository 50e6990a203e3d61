"""GPU: resize + gray and ORB bit-exact against cv2, exact match counts against cv2's BFMatcher, Thread / scenes
against the reference's golden output, batch-size independence, the Shot -> Thread and CLI chains."""
import json
import os
import sys

import numpy as np
import pytest
import torch

from oracle import thread as O
from pyannote_video_b200 import thread as T
from pyannote_video_b200.annotation import Segment
from pyannote_video_b200.cli import ArrayVideo, main

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import thread_scenario as sc  # noqa: E402

pytestmark = pytest.mark.gpu
GOLDEN = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "thread_golden.json")))


def _golden_frames(name):
    frames, segs = sc.make_clip(name)
    collar = 10. / sc.FPS
    v = ArrayVideo(frames, sc.FPS)
    picks = []
    for s, e in segs:
        for t in (e - collar, s + collar):
            try:
                picks.append(v(t))
            except IOError:
                pass
    return frames, np.stack(picks)


def _tie_frame():
    """a 10 px tiled patch, 240 x 200 (resized to itself): exact Harris ties, levels 0 and 1 exceed their quotas"""
    tile = np.random.default_rng(0).integers(0, 256, (10, 10, 3), dtype=np.uint8)
    return np.tile(tile, (20, 24, 1))


# source sizes whose resized row count (369, 333) has pyramid levels where float32 and float64 division of the row
# count by the level scale round differently: 1920 x 1038 (1.85:1) and 333 x 200
ROUNDING_SIZES = {"rows369": (1038, 1920), "rows333": (200, 333)}


@pytest.mark.parametrize("name", sorted(GOLDEN["clips"]) + ["tie", "flat"] + sorted(ROUNDING_SIZES))
def test_orb_bit_exact_vs_cv2(name):
    if name == "tie":
        frames = _tie_frame()[None]
    elif name in ROUNDING_SIZES:
        H, W = ROUNDING_SIZES[name]
        frames = np.stack([sc._mosaic(np.random.default_rng(s), H, W) for s in (1, 2)])
    elif name == "flat":
        frames = np.full((1, 120, 200, 3), 77, np.uint8)
    else:
        frames = _golden_frames(name)[1]
    size = (frames.shape[2], frames.shape[1])
    ext = T.OrbExtractor(size, height=200, keep_keypoints=True)
    dev = torch.from_numpy(frames).cuda()
    gray = ext.gray_resize(dev).cpu().numpy()
    want_gray = np.stack([O.cv2_gray(f, O.resize_dsize(size, 200)) for f in frames])
    assert np.array_equal(gray, want_gray)
    desc, off = ext.extract(dev)
    desc = desc.cpu().numpy()
    for i, g in enumerate(want_gray):
        kc, dc = O.cv2_orb(g)
        kp = ext.keypoints[i].astype(np.float64)
        d = desc[off[i]:off[i + 1]]
        assert len(kp) == len(kc), (i, len(kp), len(kc))
        assert O.as_set(kp, d) == O.as_set(kc, dc), i
        if name == "tie":
            assert max(np.sum(kc[:, 2] == lv) - q for lv, q in enumerate(O.level_quotas())) > 0
        if name == "flat":
            assert len(kc) == 0


def test_match_counts_equal_bf_on_cv2_descriptors():
    _, picks = _golden_frames("abab")
    size = (picks.shape[2], picks.shape[1])
    descs = [O.cv2_orb(O.cv2_gray(f, O.resize_dsize(size, 200)))[1] for f in picks]
    off = np.concatenate([[0], np.cumsum([len(d) for d in descs])])
    packed = torch.from_numpy(np.concatenate(descs)).cuda()
    pairs = [(i, j) for i in range(len(descs)) for j in range(len(descs))]
    got = T.match_counts(packed, off, np.array(pairs), torch.device("cuda", 0))
    assert got.tolist() == [O.cv2_bf_count(descs[i], descs[j]) for i, j in pairs]


def _tracks(a):
    return [[s.start, s.end, l] for s, _, l in a.itertracks(yield_label=True)]


@pytest.mark.parametrize("name", sorted(GOLDEN["clips"]))
def test_thread_equals_reference(name):
    g = GOLDEN["clips"][name]
    frames, segs = sc.make_clip(name)
    shots = [Segment(*s) for s in segs]
    per_batch = []
    for batch in (1, 7, 64):
        th = T.Thread(ArrayVideo(frames, sc.FPS), shot=shots, lookahead=sc.lookahead_of(name), batch=batch)
        threads = th()
        assert _tracks(threads) == g["threads"]
        assert _tracks(th.scenes(threads)) == g["scenes"]
        per_batch.append(th.counts)
    assert per_batch[0] == per_batch[1] == per_batch[2]
    assert {(i, j): bf for i, j, _, bf in g["pairs"]} == per_batch[0]


def test_frames_on_another_device_are_refused():
    ext = T.OrbExtractor((320, 180))
    with pytest.raises(RuntimeError):
        ext.extract(torch.zeros((1, 180, 320, 3), dtype=torch.uint8))


def test_extractors_on_two_devices_agree():
    """the pattern and patch tables are static __constant__ data, present on every device"""
    if torch.cuda.device_count() < 2:
        pytest.skip("one CUDA device")
    frames = _golden_frames("abab")[1]
    size = (frames.shape[2], frames.shape[1])
    out = []
    for dev in (torch.device("cuda", 0), torch.device("cuda", torch.cuda.device_count() - 1)):
        ext = T.OrbExtractor(size, height=200, device=dev)
        desc, off = ext.extract(torch.from_numpy(frames).to(dev))
        out.append((desc.cpu().numpy(), off))
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])
    want = O.cv2_orb(O.cv2_gray(frames[0], O.resize_dsize(size, 200)))[1]
    assert sorted(map(bytes, out[1][0][:out[1][1][1]])) == sorted(map(bytes, want))


def _assert_same_tracks(got, want):
    assert len(got) == len(want)
    for (s, e, l), (ws, we, wl) in zip(got, want):
        assert (l, round(s, 9), round(e, 9)) == (wl, round(ws, 9), round(we, 9))


def test_shot_then_thread_chain():
    """GPU Shot finds the golden boundaries of the clip, so Thread(shot=None) gives the reference's threads"""
    g = GOLDEN["clips"]["abab"]
    frames, _ = sc.make_clip("abab")
    th = T.Thread(ArrayVideo(frames, sc.FPS), lookahead=sc.lookahead_of("abab"))
    threads = th()
    _assert_same_tracks(_tracks(threads), g["threads"])
    _assert_same_tracks(_tracks(th.scenes(threads)), g["scenes"])


def test_cli_shot_thread_scene(tmp_path):
    frames, _ = sc.make_clip("abab")
    vid = str(tmp_path / "v.npy")
    np.save(vid, frames)
    shot, thr, scn = (str(tmp_path / n) for n in ("shot.json", "thread.json", "scene.json"))
    assert main(["shot", vid, shot]) == 0
    assert main(["thread", "--lookahead", "5", vid, shot, thr]) == 0
    assert main(["scene", vid, thr, scn]) == 0
    g = GOLDEN["clips"]["abab"]
    for path, want in ((thr, g["threads"]), (scn, g["scenes"])):
        data = json.load(open(path))
        assert data["pyannote"] == "Annotation"
        got = [[c["segment"]["start"], c["segment"]["end"], c["label"]] for c in data["content"]]
        _assert_same_tracks(got, want)
