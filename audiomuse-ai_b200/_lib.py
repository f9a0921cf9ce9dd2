"""ctypes binding of libaudiomuse_b200.so (include/audiomuse_b200.h).

The library is loaded lazily and never at import time of the package (RQ workers fork per
job, rq_worker.py:48-55; CUDA must be initialised in the child).  There is NO CPU fallback:
if the shared library or a CUDA device is missing the calls raise ``B200Error``.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "libaudiomuse_b200.so")

AM_OK, AM_ERR_INVALID, AM_ERR_CUDA, AM_ERR_OOM, AM_ERR_NO_DEVICE, AM_ERR_IO, AM_ERR_RECALL = 0, -1, -2, -3, -4, -5, -6


class B200Error(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"libaudiomuse_b200 error {code}: {message}")
        self.code = code


class B200OutOfMemory(B200Error, MemoryError):
    """Message contains 'out of memory' so tasks/memory_utils.py's string match retries."""


class MelCfg(C.Structure):
    _fields_ = [("sr", C.c_int), ("n_fft", C.c_int), ("hop", C.c_int), ("n_mels", C.c_int),
                ("fmin", C.c_float), ("fmax", C.c_float), ("transpose", C.c_int)]


class TrackFeat(C.Structure):
    """am_track_feat"""
    _fields_ = [("tempo", C.c_double), ("tuning", C.c_double), ("energy", C.c_float), ("chroma_mean", C.c_float * 12),
                ("period", C.c_int), ("key", C.c_int), ("is_major", C.c_int), ("n_frames", C.c_int),
                ("n_pitches", C.c_int), ("tuning_counts", C.c_int * 100)]


_vp, _i, _i64, _f, _u64, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_uint64, C.c_size_t
_P = C.POINTER

# name -> (restype, argtypes); mirrors include/audiomuse_b200.h one to one
SIGNATURES = {
    "am_init": (_i, [_i]),
    "am_shutdown": (None, []),
    "am_last_error": (C.c_char_p, []),
    "am_version": (_i, []),
    "am_launch_count": (_u64, []),
    "am_profile_enable": (None, [_i]),
    "am_profile_report": (_i, [C.c_char_p, _i]),
    "am_mel_plan_create": (_i, [_P(MelCfg), _P(_vp)]),
    "am_mel_plan_free": (None, [_vp]),
    "am_mel_filterbank": (_i, [_P(MelCfg), _vp]),
    "am_mel_num_frames": (_i, [_P(MelCfg), _i]),
    "am_mel_batch": (_i, [_vp, _i, _i, _P(MelCfg), _vp]),
    "am_mel_batch_i16": (_i, [_vp, _i, _i, _P(MelCfg), _vp]),
    "am_mel_batch_dev": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    "am_mel_plan_create_ex": (_i, [_P(MelCfg), _i, _i, _P(_vp)]),
    "am_mel_num_frames_ex": (_i, [_P(MelCfg), _i, _i]),
    "am_mel_batch_ex": (_i, [_vp, _i, _i, _P(MelCfg), _i, _i, _vp]),
    "am_pcm_to_segments": (_i, [_vp, _i64, _vp, _i, _P(_i)]),
    "am_wav_info": (_i, [C.c_char_p, _P(_i), _P(_i), _P(_i64), _P(_i)]),
    "am_wav_decode_mono": (_i, [C.c_char_p, _i64, _vp, _i64, _P(_i64), _P(_i)]),
    "am_wav_to_segments": (_i, [C.c_char_p, C.c_double, _vp, _i, _P(_i), _P(C.c_double)]),
    "am_resample_plan_create": (_i, [_i, _i, _P(_vp)]),
    "am_resample_plan_free": (None, [_vp]),
    "am_resample_out_len": (_i64, [_vp, _i64]),
    "am_resample_dev": (_i, [_vp, _vp, _i64, _vp, _vp]),
    "am_resample_filter": (_i, [_i, _i, _vp, _i, _P(_i), _P(_i), _P(_i), _P(_i64)]),
    "am_resample": (_i, [_vp, _i64, _i, _i, _vp, _i64, _P(_i64)]),
    "am_num_segments": (_i, [_i64]),
    "am_audio_to_segments_dev": (_i, [_vp, _i64, _vp, _i, _P(_i), _vp]),
    "am_clap_load": (_i, [C.c_char_p, _P(_vp)]),
    "am_clap_load_mem": (_i, [_vp, _sz, _P(_vp)]),
    "am_clap_describe_file": (_i, [C.c_char_p, C.c_char_p, _i]),
    "am_clap_release_workspace": (_i, [_vp]),
    "am_clap_free": (None, [_vp]),
    "am_clap_embedding_dim": (_i, [_vp]),
    "am_clap_n_mels": (_i, [_vp]),
    "am_clap_flops_per_segment": (C.c_double, [_vp, _i]),
    "am_clap_flops_split": (_i, [_vp, _i, _P(C.c_double), _P(C.c_double), _P(C.c_double)]),
    "am_clap_embed": (_i, [_vp, _vp, _i, _i, _vp]),
    "am_clap_embed_dev": (_i, [_vp, _vp, _i, _i, _vp, _vp]),
    "am_clap_embed_tracks": (_i, [_vp, _P(MelCfg), _vp, _i, _vp, _i, _vp]),
    "am_clap_embed_tracks_submit": (_i, [_vp, _P(MelCfg), _vp, _i, _vp, _i, _vp]),
    "am_clap_embed_tracks_collect": (_i, [_vp]),
    "am_clap_embed_tracks_dev": (_i, [_vp, _vp, _vp, _i, _vp, _i, _i, _vp, _vp]),
    "am_musicnn_load": (_i, [C.c_char_p, _P(_vp)]),
    "am_musicnn_load_mem": (_i, [_vp, _sz, _P(_vp)]),
    "am_musicnn_describe_file": (_i, [C.c_char_p, C.c_char_p, _i]),
    "am_musicnn_free": (None, [_vp]),
    "am_musicnn_release_workspace": (_i, [_vp]),
    "am_musicnn_dims": (_i, [_vp, _P(_i), _P(_i), _P(_i)]),
    "am_musicnn_io_names": (_i, [_vp, C.c_char_p, C.c_char_p, _i]),
    "am_musicnn_flops_per_patch": (C.c_double, [_vp, _i, _i, _P(C.c_double)]),
    "am_musicnn_run": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "am_musicnn_run_dev": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    "am_musicnn_analyze_tracks": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "am_features_create": (_i, [_P(_vp)]),
    "am_features_free": (None, [_vp]),
    "am_features_release_workspace": (_i, [_vp]),
    "am_features_run": (_i, [_vp, _vp, _vp, _i, _vp, _vp]),
    "am_features_run_dev": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "am_knn_build": (_i, [_vp, _i64, _i, _i, _P(_vp)]),
    "am_knn_build_dev": (_i, [_vp, _i64, _i, _i, _vp, _P(_vp)]),
    "am_knn_free": (None, [_vp]),
    "am_knn_size": (_i64, [_vp]),
    "am_knn_dim": (_i, [_vp]),
    "am_knn_get_vector": (_i, [_vp, _i64, _vp]),
    "am_knn_query": (_i, [_vp, _vp, _i, _i, _vp, _vp]),
    "am_knn_query_ex": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    "am_knn_filter_by_distance": (_i, [_vp, _vp, _i, _i, C.c_float, _i, _i, _vp]),
    "am_knn_pairwise": (_i, [_vp, _vp, _i, _vp]),
    "am_knn_get_vectors": (_i, [_vp, _vp, _i, _vp]),
    "am_knn_query_dev": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "am_kmeans_fit": (_i, [_vp, _i64, _i, _i, _i, _i, _f, _u64, _vp, _vp, _vp, _P(_f), _P(_i)]),
    "am_pca_moments": (_i, [_vp, _i64, _i, _vp, _vp]),
    "am_pca_project": (_i, [_vp, _i64, _i, _vp, _vp, _i, _vp]),
    "am_dbscan": (_i, [_vp, _i64, _i, _f, _i, _vp, _P(_i)]),
    "am_kmeans_assign_dev": (_i, [_vp, _i64, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "am_kmeans_plan_create": (_i, [_vp, _i64, _i, _i, _vp, _P(_vp)]),
    "am_kmeans_plan_step": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "am_kmeans_plan_uses_tensor_cores": (_i, [_vp]),
    "am_kmeans_plan_last_recheck": (_i, [_vp, _vp, _P(_i)]),
    "am_kmeans_plan_free": (None, [_vp]),
}

# include/audiomuse_b200_debug.h: probes and self tests, in libaudiomuse_b200_debug.so only
DEBUG_LIB_PATH = os.path.join(_PKG_DIR, "libaudiomuse_b200_debug.so")
DEBUG_SIGNATURES = {
    "am_selftest_gemm": (_i, [_i, _i, _i, _i, _P(C.c_double)]),
    "am_bench_gemm": (_i, [_i, _i, _i, _i, _P(C.c_double)]),
    "am_probe_mma": (_i, [_i, _i, _i, _i, _P(C.c_double), _P(C.c_double)]),
    "am_probe_tmem_ld": (_i, [_i, _i, _i, _i, _i, _P(C.c_double), _P(C.c_double)]),
    "am_probe_pipe": (_i, [_i, _i, _i, _P(C.c_double)]),
    "am_probe_mn_major": (_i, [C.c_void_p, C.c_void_p, _i, _i, _i, _i, _i, _i, C.c_void_p]),
}

_lib = None
_debug_lib = None
_lock = threading.Lock()


def load_debug():
    """dlopen the debug library (the product library's objects + the probes / self tests); tests and tools only."""
    global _debug_lib
    if _debug_lib is None:
        with _lock:
            if _debug_lib is None:
                if not os.path.exists(DEBUG_LIB_PATH):
                    raise B200Error(AM_ERR_NO_DEVICE, f"{DEBUG_LIB_PATH} is missing: run `python __graft_entry__.py`")
                lib = C.CDLL(DEBUG_LIB_PATH)
                for name, (res, args) in {**DEBUG_SIGNATURES, "am_last_error": (C.c_char_p, [])}.items():
                    fn = getattr(lib, name)
                    fn.restype = res
                    fn.argtypes = args
                _debug_lib = lib
    return _debug_lib


def load():
    """dlopen the library (no CUDA work happens here)."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise B200Error(AM_ERR_NO_DEVICE,
                                f"{LIB_PATH} is missing: run `python __graft_entry__.py` (build()) first; "
                                "there is no CPU fallback")
            lib = C.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(lib, name)
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


def last_error() -> str:
    return load().am_last_error().decode("utf-8", "replace")


def check(status: int):
    if status == AM_OK:
        return
    msg = last_error()
    if status == AM_ERR_OOM:
        raise B200OutOfMemory(status, msg)
    raise B200Error(status, msg)


def check_debug(status: int):
    """like check(), for calls into the debug library (it carries its own copy of the error state)"""
    if status != AM_OK:
        raise B200Error(status, load_debug().am_last_error().decode("utf-8", "replace"))


def ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def as_f32(a, shape=None) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.float32)
    if shape is not None:
        a = a.reshape(shape)
    return a


def launch_count() -> int:
    return int(load().am_launch_count())


def profile_enable(on: bool) -> None:
    load().am_profile_enable(1 if on else 0)


def profile_report() -> dict:
    """Per-kernel device time (ms) and launch count since the last report."""
    import json
    lib = load()
    n = lib.am_profile_report(None, 0)
    buf = C.create_string_buffer(n + 16)
    lib.am_profile_report(buf, n + 16)
    return json.loads(buf.value.decode() or "{}")
