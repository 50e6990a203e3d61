"""Minimal `pyannote.core.Segment` / `Annotation` duck types.

`pyannote.core` is absent from the build environment; the reference's `FaceClustering` takes and returns
`Annotation` objects (pyannote/video/face/clustering.py:59-82,138-148; notebook cells 18-22 iterate them with
`itertracks(yield_label=True)`).  Only the part of the interface that path uses is provided.
"""
import itertools
import string
from collections import namedtuple

DEFAULT_TRACK = "_"


def string_generator():
    """A, B, ..., Z, AA, AB, ... (pyannote.core.utils.generators.string_generator)"""
    for n in itertools.count(1):
        for letters in itertools.product(string.ascii_uppercase, repeat=n):
            yield "".join(letters)


def pairwise(iterable):
    """(s0, s1), (s1, s2), ..."""
    a, b = itertools.tee(iterable)
    next(b, None)
    return zip(a, b)


class Segment(namedtuple("Segment", ["start", "end"])):
    __slots__ = ()

    @property
    def duration(self):
        return max(0.0, self.end - self.start)

    @property
    def middle(self):
        return 0.5 * (self.start + self.end)

    def __bool__(self):
        return bool((self.end - self.start) > 0.0)          # empty segments are falsy, as in pyannote.core

    def __str__(self):
        return "[%.3f --> %.3f]" % (self.start, self.end)


class Annotation(object):
    """(segment, track) -> label, iterated in (segment, track) order"""

    def __init__(self, uri=None, modality=None):
        self.uri, self.modality = uri, modality
        self._tracks = {}

    @staticmethod
    def _key(key):
        """(segment, track) from a (segment, track) tuple or a bare Segment (track "_", as pyannote.core)"""
        if isinstance(key, Segment):
            return key, DEFAULT_TRACK
        return key

    def __setitem__(self, key, label):
        segment, track = self._key(key)
        if not isinstance(segment, Segment):
            segment = Segment(*segment)
        if not segment:
            return                                           # pyannote.core ignores empty segments
        self._tracks[(segment, track)] = label

    def __getitem__(self, key):
        segment, track = self._key(key)
        if not isinstance(segment, Segment):
            segment = Segment(*segment)
        return self._tracks[(segment, track)]

    def __len__(self):
        return len(self._tracks)

    def __bool__(self):
        return len(self._tracks) > 0

    def itertracks(self, yield_label=False):
        for (segment, track) in sorted(self._tracks, key=lambda k: (k[0].start, k[0].end, str(k[1]))):
            if yield_label:
                yield segment, track, self._tracks[(segment, track)]
            else:
                yield segment, track

    def itersegments(self):
        for segment, _ in self.itertracks():
            yield segment

    def labels(self):
        return sorted(set(self._tracks.values()), key=str)

    def rename_labels(self, mapping):
        out = Annotation(self.uri, self.modality)
        for k, v in self._tracks.items():
            out._tracks[k] = mapping.get(v, v)
        return out

    def copy(self):
        out = Annotation(self.uri, self.modality)
        out._tracks = dict(self._tracks)
        return out

    def label_tracks(self, label):
        return [(s, t) for s, t, l in self.itertracks(yield_label=True) if l == label]

    def subset(self, labels):
        """the tracks whose label is in `labels`"""
        labels = set(labels)
        out = Annotation(self.uri, self.modality)
        out._tracks = {k: v for k, v in self._tracks.items() if v in labels}
        return out

    def smooth(self):
        """per label, touching or overlapping segments merged into one; tracks renamed A, B, ... label by label"""
        names = string_generator()
        out = Annotation(self.uri, self.modality)
        for label in self.labels():
            merged = []
            for segment in sorted(s for (s, _), v in self._tracks.items() if v == label):
                if merged and segment.start <= merged[-1].end:
                    merged[-1] = Segment(merged[-1].start, max(merged[-1].end, segment.end))
                else:
                    merged.append(segment)
            for segment in merged:
                out[segment, next(names)] = label
        return out

    def to_dict(self):
        """{track: label} (track names are unique on this path: one segment per face track)"""
        return {t: l for _, t, l in self.itertracks(yield_label=True)}

    def __eq__(self, other):
        return isinstance(other, Annotation) and self._tracks == other._tracks

    def __repr__(self):
        return "Annotation(%d tracks, %d labels)" % (len(self), len(self.labels()))
