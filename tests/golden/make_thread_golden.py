"""Generates tests/golden/thread_golden.json by running the REFERENCE's own Thread
(/root/reference/pyannote/video/structure/thread.py, imported unmodified from where it lies, with cv2 and networkx)
on the deterministic clips of tests/thread_scenario.py.

pyannote.core is not installed: Annotation, Segment and the generators are this package's.  The module's ORB branch
is chosen by `OPENCV = int(cv2.__version__[0])`, which assigns no ORB under OpenCV 4; it is set to 3 so that
`cv2.ORB_create()` is used.  FLANN-LSH counts are random (its hash tables are rebuilt on every match); the generator
asserts that the FLANN count and the exact brute-force count fall on the same side of min_match for every pair, so
the reference's own output is the expected output of the exact matcher.  Run in the build container only:

    python tests/golden/make_thread_golden.py
"""
import importlib.util
import json
import os
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from pyannote_video_b200 import annotation as A          # noqa: E402
from pyannote_video_b200.cli import ArrayVideo           # noqa: E402
from oracle import thread as O                           # noqa: E402
import thread_scenario as sc                             # noqa: E402

for name in ("pyannote", "pyannote.core", "pyannote.core.utils", "pyannote.core.utils.generators", "pyannote.video",
             "pyannote.video.structure", "pyannote.video.structure.shot", "tqdm"):
    sys.modules[name] = types.ModuleType(name)
    sys.modules[name].__path__ = []
sys.modules["pyannote.core"].Annotation = A.Annotation
sys.modules["pyannote.core.utils.generators"].pairwise = A.pairwise
sys.modules["pyannote.core.utils.generators"].string_generator = A.string_generator
sys.modules["pyannote.video.structure.shot"].Shot = object
sys.modules["tqdm"].tqdm = None

spec = importlib.util.spec_from_file_location("pyannote.video.structure.thread",
                                              "/root/reference/pyannote/video/structure/thread.py")
ref = importlib.util.module_from_spec(spec)
sys.modules[spec.name] = ref
spec.loader.exec_module(ref)
ref.OPENCV = 3
MIN_MATCH = 20


def tracks(annotation):
    return [[s.start, s.end, label] for s, _, label in annotation.itertracks(yield_label=True)]


out = {"min_match": MIN_MATCH, "clips": {}, "product_lookahead": []}
for n in range(0, 9):
    for la in range(1, 7):
        out["product_lookahead"].append({"n": n, "lookahead": la,
                                         "pairs": [list(p) for p in ref.product_lookahead(range(n), la)]})
for name in sc.CLIPS:
    frames, segs = sc.make_clip(name)
    video = ArrayVideo(frames, sc.FPS)
    shots = [A.Segment(*s) for s in segs]
    th = ref.Thread(video, shot=shots, min_match=MIN_MATCH, lookahead=sc.lookahead_of(name))
    collar = 10. / video.frame_rate
    index = {s: i for i, s in enumerate(shots)}
    pairs = []
    for a, b in ref.product_lookahead(shots, th.lookahead):
        q, t = th._compute_orb(a.end - collar), th._compute_orb(b.start + collar)
        flann = int(th._match(q, t))
        bf = O.cv2_bf_count(q, t)
        assert (flann > MIN_MATCH) == (bf > MIN_MATCH), (name, a, b, flann, bf)
        pairs.append([index[a], index[b], flann, bf])
    threads = th()
    scenes = th.scenes(threads)
    out["clips"][name] = {"sha256": sc.sha256(frames), "shots": [list(s) for s in segs], "pairs": pairs,
                          "edges": [[i, j] for i, j, _, bf in pairs if bf > MIN_MATCH],
                          "threads": tracks(threads), "scenes": tracks(scenes)}
    print(name, frames.shape, "pairs", len(pairs), "bf", [p[3] for p in pairs], "threads", tracks(threads),
          "scenes", [s[2] for s in tracks(scenes)])

with open(os.path.join(HERE, "thread_golden.json"), "w") as f:
    json.dump(out, f, indent=1)
