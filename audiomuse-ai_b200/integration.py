"""The patch a maintainer applies to AudioMuse-AI (INTEGRATION.md section 3), as code.

    from audiomuse_ai_b200 import integration
    integration.install_voyager_shim()      # BEFORE `import tasks.voyager_manager` / `tasks.clap_text_search`
    import tasks.clap_analyzer, tasks.voyager_manager, tasks.clustering_gpu
    integration.apply(clap=tasks.clap_analyzer, voyager_manager=tasks.voyager_manager, clustering=tasks.clustering_gpu)

Nothing in the reference tree is modified; every assignment below replaces a module attribute that the reference's
own callers look up at call time (tasks/analysis.py:883 imports analyze_audio_file as clap_analyze from the module,
tasks/voyager_manager.py:1594 calls the module-level _filter_by_distance, clustering_helper.py:21 calls
get_clustering_model).  tests/test_reference_shims.py applies exactly this to the stub-imported reference modules.
"""
from __future__ import annotations

import os
import sys

CLAP_NAMES = ("compute_mel_spectrogram", "analyze_audio_file", "initialize_clap_audio_model", "get_clap_audio_model",
              "unload_clap_audio_only", "unload_clap_model", "is_clap_model_loaded", "is_clap_audio_loaded")


def install_voyager_shim() -> None:
    """`import voyager` in tasks/voyager_manager.py:12 and tasks/clap_text_search.py resolves to the flat exact index:
    Index(space, num_dimensions, M, ef_construction), add_items, query, get_vector, len, .ef, save / load,
    Space.Cosine, RecallError."""
    from . import voyager_compat

    sys.modules["voyager"] = voyager_compat


def make_filter_by_distance(vm):
    """voyager_manager._filter_by_distance (tasks/voyager_manager.py:526-617) on the vectors already in HBM: one
    device walk instead of O(k) get_vector calls + Python distance loops.  Keeps exactly the items upstream keeps
    (tests/golden/filter_golden.npz)."""

    def _filter_by_distance_b200(song_results, db_conn):
        if vm.DUPLICATE_DISTANCE_CHECK_LOOKBACK <= 0 or not song_results:
            return song_results
        ids = [vm.reverse_id_map.get(s["item_id"], -1) for s in song_results]   # unknown item -> dropped, as upstream
        thr = (vm.DUPLICATE_DISTANCE_THRESHOLD_COSINE if vm.VOYAGER_METRIC == "angular"
               else vm.DUPLICATE_DISTANCE_THRESHOLD_EUCLIDEAN)
        keep = vm.voyager_index.filter_by_distance([-1 if i is None else i for i in ids], thr,
                                                   lookback=vm.DUPLICATE_DISTANCE_CHECK_LOOKBACK,
                                                   batch=vm.BATCH_SIZE_VECTOR_OPS)
        return [s for s, k in zip(song_results, keep) if k]

    return _filter_by_distance_b200


MUSICNN_MODEL_FILES = ("musicnn_embedding.onnx", "musicnn_prediction.onnx")


class OrtProxy:
    """Stands in for the `ort` (onnxruntime) module that tasks/analysis.py uses only for MusiCNN (:405-509, :763-841):
    InferenceSession returns a B200 MusicnnSession for the two MusiCNN model files (config EMBEDDING_MODEL_PATH /
    PREDICTION_MODEL_PATH) and the real session for anything else; every other attribute (get_available_providers,
    capi.onnxruntime_pybind11_state.RuntimeException named by the reference's except clauses, ...) is the real
    module's."""

    def __init__(self, real):
        self._real = real

    def InferenceSession(self, path_or_bytes, *args, **kwargs):
        if isinstance(path_or_bytes, (str, os.PathLike)) and os.path.basename(os.fspath(path_or_bytes)) in MUSICNN_MODEL_FILES:
            from .musicnn import MusicnnSession

            return MusicnnSession(os.fspath(path_or_bytes))
        return self._real.InferenceSession(path_or_bytes, *args, **kwargs)

    def __getattr__(self, name):
        return getattr(self._real, name)


def make_analyze_track(analysis):
    """analyze_track (tasks/analysis.py:324-573) with everything after decoding on the B200: the tempo / energy /
    key / scale features (track_features) and the MusiCNN embedding + moods (musicnn.analyze_tracks).  Same signature
    and the same 2- or 4-tuples; an empty, silent, too-short or failed track gives the None tuple, as upstream.
    Decoding stays the reference's own: analysis.robust_load_audio_with_fallback, looked up at call time.
    MusiCNN sessions come from onnx_sessions when they are B200 MusicnnSessions, else from model_paths (loaded once
    per path).  On B200OutOfMemory the workspaces are released and the track is retried once."""
    import logging

    import numpy as np

    from . import _lib, musicnn, track_features as tfm

    log = logging.getLogger(__name__)
    state = {"features": None, "sessions": {}}

    def _sessions(model_paths, onnx_sessions):
        if onnx_sessions is not None and all(isinstance(onnx_sessions.get(k), musicnn.MusicnnSession)
                                             for k in ("embedding", "prediction")):
            return onnx_sessions["embedding"], onnx_sessions["prediction"]
        out = []
        for k in ("embedding", "prediction"):
            path = os.fspath(model_paths[k])
            if path not in state["sessions"]:
                state["sessions"][path] = musicnn.MusicnnSession(path)
            out.append(state["sessions"][path])
        return tuple(out)

    def _run(audio, emb, pred):
        if state["features"] is None:
            state["features"] = tfm.FeatureSession()
        feats = tfm.track_features([audio], session=state["features"])[0]
        tower = musicnn.analyze_tracks([audio], emb, pred)[0]
        return feats, tower

    def analyze_track(file_path, mood_labels_list, model_paths, onnx_sessions=None, return_audio=False):
        none = (None, None, None, None) if return_audio else (None, None)
        audio, sr = analysis.robust_load_audio_with_fallback(file_path, target_sr=16000)
        if audio is None or audio.size == 0 or not np.any(audio):
            log.warning("Could not load a valid audio signal for %s. Skipping track.", os.path.basename(file_path))
            return none
        audio = np.ascontiguousarray(audio, dtype=np.float32).reshape(-1)
        try:
            emb, pred = _sessions(model_paths, onnx_sessions)
            try:
                feats, tower = _run(audio, emb, pred)
            except _lib.B200OutOfMemory:
                log.warning("B200 out of memory for %s: releasing workspaces and retrying once",
                            os.path.basename(file_path))
                for s in (state["features"], emb, pred):
                    if s is not None:
                        s.release_workspace()
                feats, tower = _run(audio, emb, pred)
        except _lib.B200Error as e:
            log.error("B200 analysis failed for %s: %s", os.path.basename(file_path), e)
            return none
        if tower is None or feats is None:
            log.warning("Track too short to create spectrogram patches: %s", os.path.basename(file_path))
            return none
        embedding, moods, _ = tower
        result = {"tempo": feats["tempo"], "key": feats["key"], "scale": feats["scale"],
                  "moods": {label: float(v) for label, v in zip(mood_labels_list, moods)},
                  "energy": feats["energy"]}
        embedding = np.asarray(embedding, dtype=np.float32)
        return (result, embedding, audio, sr) if return_audio else (result, embedding)

    analyze_track._b200 = True
    return analyze_track


def apply(clap=None, voyager_manager=None, clustering=None, allow_sklearn_fallback: bool = True, analysis=None,
          analyze_track: bool = False) -> None:
    """clap / voyager_manager / clustering / analysis: the reference's already imported tasks.* modules (pass only the
    ones to patch).  analysis (tasks.analysis): its `ort` becomes an OrtProxy, so analyze_track's MusiCNN sessions run
    on the B200.  With analyze_track=True, analysis.analyze_track itself is replaced by make_analyze_track(analysis)
    (analyze_album_task resolves that module global at call time), so its librosa tempo / energy / chroma code runs
    on the B200 too; with the default False that code stays as it is.  allow_sklearn_fallback keeps the
    reference's contract that a failing GPU k-means silently falls back to scikit-learn (tasks/clustering_gpu.py:130-148); this repository's own tests run with it off so a missing CUDA
    library can never pass as the GPU path."""
    if analyze_track and analysis is None:
        raise ValueError("apply(analyze_track=True) needs the analysis module")
    if clap is not None:
        from . import clap_analyzer as b200_clap

        for name in CLAP_NAMES:
            setattr(clap, name, getattr(b200_clap, name))
    if voyager_manager is not None:
        voyager_manager._filter_by_distance = make_filter_by_distance(voyager_manager)
    if clustering is not None:
        from . import clustering_gpu as b200_cg

        clustering.GPUKMeans = b200_cg.GPUKMeans
        clustering.GPUDBSCAN = b200_cg.GPUDBSCAN   # get_clustering_model / get_pca_model look the classes up at call time
        clustering.GPUPCA = b200_cg.GPUPCA
        clustering.check_gpu_available = b200_cg.check_gpu_available
        if allow_sklearn_fallback:
            os.environ.setdefault("B200_ALLOW_SKLEARN_FALLBACK", "1")
    if analysis is not None and not isinstance(analysis.ort, OrtProxy):
        analysis.ort = OrtProxy(analysis.ort)
    if analyze_track and not getattr(analysis.analyze_track, "_b200", False):
        analysis.analyze_track = make_analyze_track(analysis)
