"""analyze_track's tempo, key, scale and energy (tasks/analysis.py:344-365) on the B200.

    feats = track_features([pcm_16k, ...])       # per track {"tempo", "key", "scale", "energy"} or None

The reference computes these with librosa on the CPU, one track at a time (beat_track, rms, chroma_stft and a
key / scale correlation block).  Here every track of a call is packed into one buffer and all of it runs on the
device (csrc/track_features.cu).  Parity with librosa itself is unpinned; oracle/track_features.py is the restatement
the device path is tested against.  Allocation failures raise `B200OutOfMemory`.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import numpy as np

from . import _lib

KEYS = ("C", "C#", "D", "D#", "E", "F", "F#", "G", "G#", "A", "A#", "B")
N_LAGS = 250
# samples per am_features_run call (2^26 = 70 minutes at 16 kHz: about 0.9 GB of workspace); a longer track goes alone
MAX_SAMPLES_PER_CALL = 1 << 26


class FeatureSession:
    """Owns the device tables and the workspace of the track-feature kernels."""

    def __init__(self):
        lib = _lib.load()
        _lib.check(lib.am_init(-1))
        h = C.c_void_p()
        _lib.check(lib.am_features_create(C.byref(h)))
        self._h = h

    def run(self, waveforms_16k: Sequence[np.ndarray], tempogram: bool = False):
        """One call over all the tracks: (am_track_feat array, f32[n, 250] tempogram means or None)."""
        lens = np.array([np.asarray(w).size for w in waveforms_16k], dtype=np.int64)
        offsets = np.zeros(len(lens) + 1, dtype=np.int64)
        np.cumsum(lens, out=offsets[1:])
        pcm = np.empty(max(int(offsets[-1]), 1), dtype=np.float32)
        for w, a in zip(waveforms_16k, offsets[:-1]):
            pcm[a:a + np.asarray(w).size] = np.asarray(w, dtype=np.float32).reshape(-1)
        n = len(lens)
        out = (_lib.TrackFeat * max(n, 1))()
        tg = np.zeros((n, N_LAGS), dtype=np.float32) if tempogram else None
        if n:
            _lib.check(_lib.load().am_features_run(self._h, _lib.ptr(pcm), _lib.ptr(offsets), n, out,
                                                   _lib.ptr(tg) if tg is not None else None))
        return out[:n], tg

    def run_dev(self, pcm_dev_ptr: int, offsets: np.ndarray, tempogram: bool = False, stream: int = 0):
        """As run(), with the PCM already on the device (offsets on the host, in samples)."""
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        n = len(offsets) - 1
        out = (_lib.TrackFeat * max(n, 1))()
        tg = np.zeros((n, N_LAGS), dtype=np.float32) if tempogram else None
        if n:
            _lib.check(_lib.load().am_features_run_dev(self._h, C.c_void_p(pcm_dev_ptr), _lib.ptr(offsets), n, out,
                                                       _lib.ptr(tg) if tg is not None else None, C.c_void_p(stream)))
        return out[:n], tg

    def release_workspace(self) -> None:
        _lib.check(_lib.load().am_features_release_workspace(self._h))

    def close(self) -> None:
        if getattr(self, "_h", None):
            _lib.load().am_features_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def as_result(f) -> dict:
    """The values analyze_track stores (tasks/analysis.py:544-550) from one am_track_feat."""
    return {"tempo": float(f.tempo), "key": KEYS[f.key], "scale": "major" if f.is_major else "minor",
            "energy": float(f.energy)}


def track_features(waveforms_16k: Sequence[np.ndarray], max_samples: int = MAX_SAMPLES_PER_CALL,
                   session: Optional[FeatureSession] = None) -> List[Optional[dict]]:
    """Per 16 kHz mono track: {"tempo", "key", "scale", "energy"}, or None for an empty or all-zero track (the
    reference skips those, tasks/analysis.py:340-342).  Tracks go to the device in calls of at most `max_samples`."""
    sess = session if session is not None else FeatureSession()
    waves = [np.asarray(w, dtype=np.float32).reshape(-1) for w in waveforms_16k]
    res: List[Optional[dict]] = [None] * len(waves)
    live = [i for i, w in enumerate(waves) if w.size and np.any(w)]
    group, size = [], 0

    def flush():
        feats, _ = sess.run([waves[i] for i in group])
        for i, f in zip(group, feats):
            res[i] = as_result(f)

    for i in live:
        if group and size + waves[i].size > max_samples:
            flush()
            group, size = [], 0
        group.append(i)
        size += waves[i].size
    if group:
        flush()
    return res
