"""MusiCNN embedding / mood tower on the B200 behind the reference's own call surface (tasks/analysis.py:324-573).

    sess = MusicnnSession("musicnn_embedding.onnx")        # onnxruntime.InferenceSession duck type
    emb = sess.run(None, {"model/Placeholder:0": patches})[0]     # [n, 187, 96] -> [n, 200]
    analyze_tracks([pcm_16k, ...], emb_sess, pred_sess)            # bulk: per-track 200-d means + 50 moods

`run_inference` (analysis.py:129-170) resolves tensor names through `get_inputs()` / `get_outputs()` and calls
`run([output_name], feeds)`; both graphs keep the exported names.  Allocation failures raise `B200OutOfMemory`
(its message contains "out of memory").  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Sequence

import numpy as np

from . import _lib


class _Arg:
    """onnxruntime.NodeArg look-alike: what run_inference reads (.name, .shape, .type)."""

    def __init__(self, name: str, shape, type_: str = "tensor(float)"):
        self.name, self.shape, self.type = name, shape, type_

    def __repr__(self):
        return f"NodeArg(name={self.name!r}, shape={self.shape})"


class MusicnnSession:
    """Stands in for onnxruntime.InferenceSession(musicnn_embedding.onnx | musicnn_prediction.onnx)."""

    def __init__(self, path_or_bytes, providers=None, **_ignored):
        lib = _lib.load()
        _lib.check(lib.am_init(-1))
        h = C.c_void_p()
        if isinstance(path_or_bytes, (bytes, bytearray)):
            blob = bytes(path_or_bytes)
            buf = C.create_string_buffer(blob, len(blob))
            _lib.check(lib.am_musicnn_load_mem(buf, len(blob), C.byref(h)))
        else:
            _lib.check(lib.am_musicnn_load(os.fsencode(path_or_bytes), C.byref(h)))
        self._h = h
        emb, ind, outd = C.c_int(), C.c_int(), C.c_int()
        _lib.check(lib.am_musicnn_dims(h, C.byref(emb), C.byref(ind), C.byref(outd)))
        self.is_embedding, self.in_dim, self.out_dim = bool(emb.value), ind.value, outd.value
        cap = lib.am_musicnn_io_names(h, None, None, 0)
        bi, bo = C.create_string_buffer(cap), C.create_string_buffer(cap)
        lib.am_musicnn_io_names(h, bi, bo, cap)
        shape_in = ["batch", 187, 96] if self.is_embedding else ["batch", self.in_dim]
        self._inputs = [_Arg(bi.value.decode(), shape_in)]
        self._outputs = [_Arg(bo.value.decode(), ["batch", self.out_dim])]

    def get_inputs(self) -> List[_Arg]:
        return list(self._inputs)

    def get_outputs(self) -> List[_Arg]:
        return list(self._outputs)

    def get_providers(self) -> List[str]:
        return ["B200ExecutionProvider"]

    def run(self, output_names, input_feed, run_options=None):
        if len(input_feed) != 1:
            raise ValueError(f"expected one input, got {sorted(input_feed)}")
        name, x = next(iter(input_feed.items()))
        if name not in {a.name for a in self._inputs}:
            raise ValueError(f"unknown input {name!r}; the graph takes {[a.name for a in self._inputs]}")
        for o in output_names or []:
            if o not in {a.name for a in self._outputs}:
                raise ValueError(f"unknown output {o!r}")
        x = np.ascontiguousarray(x, dtype=np.float32)
        if self.is_embedding:
            if x.ndim != 3:
                raise ValueError(f"patches must be [n, frames, mels], got {x.shape}")
            n, T, F = x.shape
        else:
            if x.ndim != 2 or x.shape[1] != self.in_dim:
                raise ValueError(f"rows must be [n, {self.in_dim}], got {x.shape}")
            n, T, F = x.shape[0], self.in_dim, 1
        out = np.empty((n, self.out_dim), dtype=np.float32)
        if n:
            _lib.check(_lib.load().am_musicnn_run(self._h, _lib.ptr(x), n, T, F, _lib.ptr(out)))
        return [out for _ in (output_names or [None])]

    def flops_per_patch(self, T: int = 187, F: int = 96):
        """(all flops, front-end flops) of one patch, from the graph's shapes."""
        fr = C.c_double()
        tot = _lib.load().am_musicnn_flops_per_patch(self._h, T, F, C.byref(fr))
        return float(tot), float(fr.value)

    def run_dev(self, x_dev_ptr: int, n: int, T: int, F: int, out_dev_ptr: int, stream: int = 0) -> None:
        _lib.check(_lib.load().am_musicnn_run_dev(self._h, C.c_void_p(x_dev_ptr), n, T, F, C.c_void_p(out_dev_ptr),
                                                  C.c_void_p(stream)))

    def release_workspace(self) -> None:
        _lib.check(_lib.load().am_musicnn_release_workspace(self._h))

    def close(self) -> None:
        if getattr(self, "_h", None):
            _lib.load().am_musicnn_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# samples staged on the device per am_musicnn_analyze_tracks call (2^26 = 70 minutes at 16 kHz: 256 MB of PCM and
# about 1.6 GB of patches); a longer track is sent alone
MAX_SAMPLES_PER_CALL = 1 << 26


def analyze_tracks(waveforms_16k: Sequence[np.ndarray], embedding: MusicnnSession,
                   prediction: Optional[MusicnnSession] = None, max_samples: int = MAX_SAMPLES_PER_CALL):
    """Bulk MusiCNN analysis of 16 kHz mono tracks, all on the device, in calls of at most `max_samples` samples.
    Returns a list with, per track, (embedding f32[200], moods f32[50] or None, n_patches), or None for a track too
    short for one patch (analysis.py:378-381)."""
    if not embedding.is_embedding or (prediction is not None and prediction.is_embedding):
        raise ValueError("analyze_tracks takes the embedding session first and the prediction session second")
    out, group, size = [], [], 0
    for w in waveforms_16k:
        if group and size + len(w) > max_samples:
            out += _analyze_group(group, embedding, prediction)
            group, size = [], 0
        group.append(w)
        size += len(w)
    if group:
        out += _analyze_group(group, embedding, prediction)
    return out


def _analyze_group(waveforms_16k, embedding, prediction):
    lens = np.array([len(w) for w in waveforms_16k], dtype=np.int64)
    offsets = np.zeros(len(lens) + 1, dtype=np.int64)
    np.cumsum(lens, out=offsets[1:])
    pcm = np.empty(int(offsets[-1]), dtype=np.float32)
    for w, a in zip(waveforms_16k, offsets[:-1]):
        pcm[a:a + len(w)] = np.asarray(w, dtype=np.float32).reshape(-1)
    n = len(lens)
    emb = np.zeros((n, embedding.out_dim), dtype=np.float32)
    moods = np.zeros((n, prediction.out_dim), dtype=np.float32) if prediction is not None else None
    npatch = np.zeros(n, dtype=np.int32)
    if n:
        _lib.check(_lib.load().am_musicnn_analyze_tracks(
            embedding._h, prediction._h if prediction is not None else None, _lib.ptr(pcm), _lib.ptr(offsets), n,
            _lib.ptr(emb), _lib.ptr(moods) if moods is not None else None, _lib.ptr(npatch)))
    return [None if npatch[i] == 0 else (emb[i], moods[i] if moods is not None else None, int(npatch[i]))
            for i in range(n)]


def describe_file(path: str) -> str:
    """The lowered program of an ONNX file, computed on the CPU (no GPU needed)."""
    lib = _lib.load()
    need = lib.am_musicnn_describe_file(os.fsencode(path), None, 0)
    if need < 0:
        _lib.check(need)
    buf = C.create_string_buffer(need + 1)
    _lib.check(min(0, lib.am_musicnn_describe_file(os.fsencode(path), buf, need + 1)))
    return buf.value.decode()
