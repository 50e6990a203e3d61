"""Generates tests/golden/shot_golden.npz by running the REFERENCE's own Shot
(/root/reference/pyannote/video/structure/shot.py, imported unmodified from where it lies, with cv2 and scipy) on the
deterministic clips of tests/shot_scenario.py.

The module imports `pyannote.core.Segment` and `..video.Video`; pyannote.core is not installed, so Segment is this
package's namedtuple duck type and the Video import is a stub (the clips are passed as cli.ArrayVideo).  Run in the
build container only:

    python tests/golden/make_shot_golden.py
"""
import importlib.util
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from pyannote_video_b200.annotation import Segment      # noqa: E402
from pyannote_video_b200.cli import ArrayVideo          # noqa: E402
from oracle import shot as O                            # noqa: E402
import shot_scenario as sc                              # noqa: E402

for name in ("pyannote", "pyannote.core", "pyannote.video", "pyannote.video.video", "pyannote.video.structure"):
    sys.modules[name] = types.ModuleType(name)
    sys.modules[name].__path__ = []
sys.modules["pyannote.core"].Segment = Segment
sys.modules["pyannote.video.video"].Video = object

spec = importlib.util.spec_from_file_location("pyannote.video.structure.shot",
                                              "/root/reference/pyannote/video/structure/shot.py")
ref = importlib.util.module_from_spec(spec)
sys.modules[spec.name] = ref
spec.loader.exec_module(ref)

GRAY_KEPT = 8                          # gray frames stored per clip (the rest is checked through the DFDs)
FLOW_CLIPS = ("hd", "odd", "h100")    # clips whose first cv2 flow is stored
out = {}
for name in sc.CLIPS:
    frames = sc.make_clip(name)
    height = sc.height_of(name)
    video = ArrayVideo(frames)
    shot = ref.Shot(video, height=height)
    gray = np.stack([shot._convert(f) for f in frames])
    tds = list(shot.iter_dfd())
    segs = [(s.start, s.end) for s in ref.Shot(video, height=height)]
    out[name + "/sha256"] = np.array(sc.sha256(frames))
    out[name + "/gray"] = gray[:GRAY_KEPT]
    out[name + "/t"] = np.array([t for t, _ in tds])
    out[name + "/dfd"] = np.array([d for _, d in tds])
    out[name + "/segments"] = np.array(segs, np.float64).reshape(-1, 2)
    if name in FLOW_CLIPS:
        out[name + "/flow"] = O.cv2_flow(gray[0], gray[1])[None]
    print(name, frames.shape, "gray", gray.shape, "segments", len(segs), "boundaries at",
          [round(s[0], 3) for s in segs[1:]])

np.savez_compressed(os.path.join(HERE, "shot_golden.npz"), **out)
print("written", os.path.getsize(os.path.join(HERE, "shot_golden.npz")), "bytes")
