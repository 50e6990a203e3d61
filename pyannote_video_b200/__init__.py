"""pyannote_video_b200 — B200-native (sm_100a) face detect -> track -> embed -> cluster, a drop-in
for the hot path of pyannote-video (pyannote/video/__init__.py:40-44 exports Face, FaceTracking,
FaceClustering).  Kernels live in csrc/ behind the C ABI of include/pv_b200.h; this package is
the Python host side.  Imports are lazy so that planning code and tests work without a GPU."""

__version__ = "0.1.0"

_EXPORTS = {
    "Face": ("face", "Face"),
    "DLIB_SMALLEST_FACE": ("face", "DLIB_SMALLEST_FACE"),
    "FaceTracking": ("tracking", "FaceTracking"),
    "TrackingByDetection": ("tracking", "TrackingByDetection"),
    "FaceClustering": ("clustering", "FaceClustering"),
    "cluster": ("clustering", "cluster"),
    "Rect": ("geometry", "Rect"),
    "DRect": ("geometry", "DRect"),
    "Point": ("geometry", "Point"),
    "FullObjectDetection": ("geometry", "FullObjectDetection"),
    "Shot": ("shot", "Shot"),
    "Thread": ("thread", "Thread"),
}

__all__ = sorted(_EXPORTS)


def __getattr__(name):
    if name in _EXPORTS:
        import importlib
        mod, attr = _EXPORTS[name]
        return getattr(importlib.import_module("." + mod, __name__), attr)
    raise AttributeError(name)
