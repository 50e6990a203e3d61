"""Face detection, tracking, feature extraction and clustering — command line.

Mirrors `scripts/pyannote-face.py` of the reference (usage string at :29-89; `track` :239-269,
`extract` :271-314) with the same verbs, flags, defaults and on-disk formats (SURVEY.md App. B):

  pyannote-face-b200 track   [options] <video> <shot.json> <tracking>
  pyannote-face-b200 extract [options] <video> <tracking> <landmark_model> <embedding_model> <landmarks> <embeddings>
  pyannote-face-b200 detect  [options] <video> <detections>        (new: raw per-frame detections)
  pyannote-face-b200 embed   ...                                     (alias of extract)
  pyannote-face-b200 cluster [--threshold=0.6] <embeddings> <labels> (notebook cells 18-22 as a verb)
  pyannote-face-b200 shot    [--height=50] [--window=2.0] [--threshold=1.0] <video> <output.json>
                             (pyannote-structure.py shot: the <shot.json> that `track` reads)
  pyannote-face-b200 thread  [--height=200] [--min-match=20] [--lookahead=24] <video> <shot.json> <output.json>
  pyannote-face-b200 scene   <video> <thread.json> <output.json>
                             (pyannote-structure.py thread / scene: Annotation JSON of threads, then of scenes)

`docopt`, `ffmpeg` and `pyannote.core` do not exist in the build environment, hence argparse and a
frame source that reads `.npy` arrays ([T,H,W,3] uint8) or `synthetic:<W>x<H>:<frames>[:<seed>]`;
`<shot.json>` is a JSON list of {"start":..,"end":..} segments (the timeline pyannote.core.json
would hold).  The `demo` verb (moviepy visualisation) is out of scope.
"""
import argparse
import json
import sys

import numpy as np

MIN_OVERLAP_RATIO = 0.5
MIN_CONFIDENCE = 10.
MAX_GAP = 1.

FACE_TEMPLATE = ('{t:.3f} {identifier:d} '
                 '{left:.3f} {top:.3f} {right:.3f} {bottom:.3f} '
                 '{status:s}\n')


class Segment(object):
    def __init__(self, start, end):
        self.start, self.end = float(start), float(end)


class ArrayVideo(object):
    """Minimal stand-in for pyannote.video.Video (pyannote/video/video.py:94-187,408-467): iteration
    yields (t, HxWx3 uint8 RGB); `frame_size` setter rescales frames (bilinear, like cv2.resize there)."""

    def __init__(self, frames, frame_rate=25.0):
        self.frames = frames
        self.frame_rate = float(frame_rate)
        self.size = (int(frames.shape[2]), int(frames.shape[1]))
        self._frame_size = self.size
        self.duration = frames.shape[0] / self.frame_rate

    @property
    def frame_size(self):
        return self._frame_size

    # the attributes pyannote.video.Video exposes to Shot: frame size (width, height), frame step, time range
    @property
    def _size(self):
        return self._frame_size

    @property
    def step(self):
        return 1.0 / self.frame_rate

    @property
    def start(self):
        return 0.0

    @property
    def end(self):
        return self.duration

    @frame_size.setter
    def frame_size(self, value):
        self._frame_size = (int(value[0]), int(value[1]))

    def __iter__(self):
        step = 1.0 / self.frame_rate
        for i in range(self.frames.shape[0]):
            rgb = np.asarray(self.frames[i])
            if self._frame_size != self.size:
                import cv2
                rgb = cv2.resize(rgb, self._frame_size)
            yield (i * step, rgb)

    def __call__(self, t):
        """the frame at time t: index int(frame_rate * t + 1e-5), as the reference Video; IOError outside the clip"""
        i = int(self.frame_rate * t + 1e-5)
        if i < 0 or i >= self.frames.shape[0]:
            raise IOError("no frame at t = %.3f" % t)
        rgb = np.asarray(self.frames[i])
        if self._frame_size != self.size:
            import cv2
            rgb = cv2.resize(rgb, self._frame_size)
        return rgb


def open_video(spec, frame_rate=25.0):
    if spec.startswith("synthetic:"):
        parts = spec.split(":")
        w, h = (int(v) for v in parts[1].lower().split("x"))
        n = int(parts[2])
        seed = int(parts[3]) if len(parts) > 3 else 0
        from .synth import make_frames
        return ArrayVideo(make_frames(n, h, w, seed=seed).numpy(), frame_rate)
    frames = np.load(spec, mmap_mode="r")
    if frames.ndim != 4 or frames.shape[-1] != 3 or frames.dtype != np.uint8:
        raise IOError("video array must be uint8 [T,H,W,3]: " + spec)
    return ArrayVideo(frames, frame_rate)


def load_shots(path):
    with open(path) as fp:
        data = json.load(fp)
    if isinstance(data, dict):
        data = data.get("content", data.get("segments", []))
    segs = []
    for s in data:
        if isinstance(s, dict) and "segment" in s:
            s = s["segment"]
        segs.append(Segment(s["start"], s["end"]))
    return segs


def read_track_file(path):
    """rows (t, track, left, top, right, bottom, status) sorted by t (stable), coordinates as float32
    (the reference parses them with dtype float32, scripts/pyannote-face.py:126-130)."""
    rows = []
    with open(path) as f:
        for line in f:
            p = line.split()
            if not p:
                continue
            rows.append((float(p[0]), int(p[1]), np.float32(p[2]), np.float32(p[3]), np.float32(p[4]),
                         np.float32(p[5]), p[6]))
    rows.sort(key=lambda r: r[0])
    return rows


def face_generator(tracking, frame_width, frame_height, reference_quirks=False):
    """Coroutine re-synchronising the track file with frame times (reference getFaceGenerator,
    scripts/pyannote-face.py:121-175): send(t) returns (T, faces) where faces are released on the first
    frame whose time >= the group time.  The reference never yields the last group (App. E.3); that
    is reproduced only with `reference_quirks`."""
    from .geometry import Rect
    rows = read_track_file(tracking)
    t = yield
    groups = []
    for (T, identifier, left, top, right, bottom, status) in rows:
        face = Rect(int(left * frame_width), int(top * frame_height), int(right * frame_width), int(bottom * frame_height))
        if groups and groups[-1][0] == T:
            groups[-1][1].append((identifier, face, status))
        else:
            groups.append((T, [(identifier, face, status)]))
    if reference_quirks and groups:
        groups = groups[:-1]
    for T, faces in groups:
        while T > t:
            t = yield t, []
        t = yield T, faces
    while True:
        t = yield t, []


def track(video, shot, output, detect_min_size=0.0, detect_every=0.0, track_min_overlap_ratio=MIN_OVERLAP_RATIO,
          track_min_confidence=MIN_CONFIDENCE, track_max_gap=MAX_GAP, face=None, tracker_bank=None, detector=None,
          control=None):
    """Tracking by detection"""
    from .tracking import FaceTracking
    if face is None:
        from .face import Face
        face = Face(detector=detector)
    tracking = FaceTracking(detect_min_size=detect_min_size, detect_every=detect_every,
                            track_min_overlap_ratio=track_min_overlap_ratio,
                            track_min_confidence=track_min_confidence, track_max_gap=track_max_gap, face=face,
                            tracker_bank=tracker_bank, control=control)
    shots = load_shots(shot) if isinstance(shot, str) else shot
    with open(output, 'w') as foutput:
        for identifier, trk in enumerate(tracking(video, shots)):
            for t, (left, top, right, bottom), status in trk:
                foutput.write(FACE_TEMPLATE.format(t=t, identifier=identifier, status=status, left=left, right=right,
                                                   top=top, bottom=bottom))
            foutput.flush()


def extract(video, landmark_model, embedding_model, tracking, landmark_output, embedding_output, face=None,
            reference_quirks=False):
    """Facial features detection: landmarks + embedding of every tracked face, all faces of a frame
    in one batched pass."""
    from .face import Face
    frame_width, frame_height = video.frame_size
    gen = face_generator(tracking, frame_width, frame_height, reference_quirks=reference_quirks)
    gen.send(None)
    face = face if face is not None else Face(landmarks=landmark_model, embedding=embedding_model)
    with open(landmark_output, 'w') as flandmark, open(embedding_output, 'w') as fembedding:
        for timestamp, rgb in video:
            T, faces = gen.send(timestamp)
            if faces:
                boxes = [[f.left(), f.top(), f.right(), f.bottom()] for _, f, _ in faces]
                fidx = [0] * len(faces)
                frames = face._to_device_frames(rgb)
                parts_dev = face.landmarks_batch(frames, boxes, fidx)
                emb = face.embed_batch(frames, parts_dev, fidx).cpu().numpy()
                parts = parts_dev.cpu().numpy()
                for k, (identifier, _, _) in enumerate(faces):
                    flandmark.write('{t:.3f} {identifier:d}'.format(t=T, identifier=identifier))
                    for x, y in parts[k]:
                        flandmark.write(' {x:.5f} {y:.5f}'.format(x=x / frame_width, y=y / frame_height))
                    flandmark.write('\n')
                    fembedding.write('{t:.3f} {identifier:d}'.format(t=T, identifier=identifier))
                    for x in emb[k]:
                        fembedding.write(' {x:.5f}'.format(x=x))
                    fembedding.write('\n')
            flandmark.flush()
            fembedding.flush()


def detect(video, output, face=None, detector=None):
    from .face import Face
    face = face if face is not None else Face(detector=detector)
    w, h = video.frame_size
    with open(output, 'w') as f:
        for t, rgb in video:
            for r in face.iterfaces(rgb):
                f.write('{t:.3f} {l:.3f} {tp:.3f} {r:.3f} {b:.3f}\n'.format(t=t, l=r.left() / w, tp=r.top() / h,
                                                                          r=r.right() / w, b=r.bottom() / h))


def shot_cmd(video, output, height=50, window=2.0, threshold=1.0):
    """Shot boundaries as a pyannote.core Timeline JSON, the file `track` reads"""
    from .shot import Shot
    return write_timeline(Shot(video, height=height, context=window, threshold=threshold), output)


def write_timeline(segments, output):
    """segments -> {"pyannote": "Timeline", "content": [{"start", "end"}, ...]} (pyannote.core's JSON)"""
    content = [{"start": float(s.start), "end": float(s.end)} for s in segments]
    with open(output, "w") as f:
        json.dump({"pyannote": "Timeline", "content": content}, f)
    return content


def write_annotation(annotation, output):
    """-> {"pyannote": "Annotation", "content": [{"segment": {"start", "end"}, "track", "label"}, ...]}"""
    content = [{"segment": {"start": float(s.start), "end": float(s.end)}, "track": t, "label": l}
               for s, t, l in annotation.itertracks(yield_label=True)]
    with open(output, "w") as f:
        json.dump({"pyannote": "Annotation", "content": content}, f)
    return content


def load_annotation(path):
    from .annotation import Annotation, Segment
    with open(path) as f:
        data = json.load(f)
    out = Annotation()
    for item in data["content"] if isinstance(data, dict) else data:
        out[Segment(float(item["segment"]["start"]), float(item["segment"]["end"])), item["track"]] = item["label"]
    return out


def thread_cmd(video, shot, output, height=200, min_match=20, lookahead=24):
    """Shot threads (pyannote-structure.py thread) as pyannote.core Annotation JSON"""
    from .annotation import Segment
    from .thread import Thread
    shots = [Segment(s.start, s.end) for s in load_shots(shot)] if isinstance(shot, str) else shot
    threads = Thread(video, shot=shots, height=height, min_match=min_match, lookahead=lookahead)()
    write_annotation(threads, output)
    return threads


def scene_cmd(threads, output):
    """Scenes from threads (Thread.scenes) as pyannote.core Annotation JSON"""
    from .thread import scenes
    out = scenes(load_annotation(threads) if isinstance(threads, str) else threads)
    write_annotation(out, output)
    return out


def cluster_cmd(embeddings, output, threshold=0.6, metric="euclidean"):
    from .clustering import FaceClustering
    clustering = FaceClustering(threshold=threshold, metric=metric)
    starting_point, features = clustering.model.preprocess(embeddings)
    result = clustering(starting_point, features=features)
    labels = result.to_dict()
    with open(output, 'w') as f:
        for trk in sorted(labels):
            f.write('{0:d} {1:d}\n'.format(trk, labels[trk]))
    return result


def main(argv=None):
    ap = argparse.ArgumentParser(prog="pyannote-face-b200", description=__doc__,
                                 formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--verbose", action="store_true")
    ap.add_argument("--frame-rate", type=float, default=25.0)
    ap.add_argument("--control", default=None, choices=["python", "native"],
                    help="tracking control loop (association, link graph, _fix, _fill_gaps): this package's Python or the C++ "
                         "of csrc/control.cu — identical tracks (default: $PV_TRACK_CONTROL or python)")
    ap.add_argument("--detector", default=None,
                    help="detector model: CNN (MMOD) — mmod_human_face_detector.dat or an .npz container — or a HOG model "
                         "(.npz of kind 'hog_detector', the reference's detector family); 'synthetic' / 'synthetic-hog' "
                         "select the seeded random-weight detectors of the tests (default: $PYANNOTE_FACE_DETECTOR)")
    sub = ap.add_subparsers(dest="verb", required=True)
    p = sub.add_parser("track")
    p.add_argument("video")
    p.add_argument("shot")
    p.add_argument("tracking")
    p.add_argument("--min-size", type=float, default=0.0)
    p.add_argument("--every", type=float, default=0.0)
    p.add_argument("--min-overlap", type=float, default=MIN_OVERLAP_RATIO)
    p.add_argument("--min-confidence", type=float, default=MIN_CONFIDENCE)
    p.add_argument("--max-gap", type=float, default=MAX_GAP)
    for name in ("extract", "embed"):
        p = sub.add_parser(name)
        p.add_argument("video")
        p.add_argument("tracking")
        p.add_argument("landmark_model")
        p.add_argument("embedding_model")
        p.add_argument("landmarks")
        p.add_argument("embeddings")
        p.add_argument("--reference-quirks", action="store_true")
    p = sub.add_parser("detect")
    p.add_argument("video")
    p.add_argument("detections")
    p = sub.add_parser("cluster")
    p.add_argument("embeddings")
    p.add_argument("labels")
    p.add_argument("--threshold", type=float, default=0.6)
    p.add_argument("--metric", default="euclidean", choices=["euclidean", "cosine"])
    p = sub.add_parser("shot")
    p.add_argument("video")
    p.add_argument("output")
    p.add_argument("--height", type=int, default=50)
    p.add_argument("--window", type=float, default=2.0)
    p.add_argument("--threshold", type=float, default=1.0)
    p = sub.add_parser("thread")
    p.add_argument("video")
    p.add_argument("shot")
    p.add_argument("output")
    p.add_argument("--height", type=int, default=200)
    p.add_argument("--min-match", type=int, default=20)
    p.add_argument("--lookahead", type=int, default=24)
    p = sub.add_parser("scene")
    p.add_argument("video")
    p.add_argument("threads")
    p.add_argument("output")
    a = ap.parse_args(argv)
    if a.verb == "track":
        track(open_video(a.video, a.frame_rate), a.shot, a.tracking, detect_min_size=a.min_size, detect_every=a.every,
              track_min_overlap_ratio=a.min_overlap, track_min_confidence=a.min_confidence, track_max_gap=a.max_gap,
              detector=a.detector, control=a.control)
    elif a.verb in ("extract", "embed"):
        extract(open_video(a.video, a.frame_rate), a.landmark_model, a.embedding_model, a.tracking, a.landmarks,
                a.embeddings, reference_quirks=a.reference_quirks)
    elif a.verb == "detect":
        detect(open_video(a.video, a.frame_rate), a.detections, detector=a.detector)
    elif a.verb == "shot":
        shot_cmd(open_video(a.video, a.frame_rate), a.output, height=a.height, window=a.window, threshold=a.threshold)
    elif a.verb == "thread":
        thread_cmd(open_video(a.video, a.frame_rate), a.shot, a.output, min_match=a.min_match, lookahead=a.lookahead,
                   height=a.height)
    elif a.verb == "scene":
        scene_cmd(a.threads, a.output)
    elif a.verb == "cluster":
        cluster_cmd(a.embeddings, a.labels, threshold=a.threshold, metric=a.metric)
    return 0


if __name__ == "__main__":
    sys.exit(main())
