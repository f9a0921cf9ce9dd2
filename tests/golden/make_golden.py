#!/usr/bin/env python
"""Generate golden vectors by RUNNING THE REFERENCE'S OWN PYTHON CODE in the build container.

    AUDIOMUSE_AI_SRC=<AudioMuse-AI checkout> python tests/golden/make_golden.py

The reference tree is imported read-only.  Third-party modules that are not installed here
(librosa, onnxruntime, voyager, psycopg2, pydub, ...) are replaced by inert stubs so
that the reference's *own* logic runs unmodified:

  * tasks/clap_analyzer.py::analyze_audio_file (:467-574) -- int16 round trip,
    segmentation, per-segment loop, mean + L2 pooling -- with
      - tasks.analysis.robust_load_audio_with_fallback -> returns a seeded waveform,
      - compute_mel_spectrogram -> deterministic stand-in (the segment itself),
      - the ORT session -> deterministic stand-in "encoder" (strided partial sums);
  * student_clap/preprocessing/audio_segmentation.py::segment_audio /
    compute_segment_positions;
  * tasks/voyager_manager.py::_get_direct_cosine_distance / _get_direct_euclidean_distance
  * tasks/voyager_manager.py::_filter_by_distance (both the <= 50 and the batched branch)
    (:99-135);
  * tests/unit/test_clap_text_search.py::DummyVoyagerIndex.query (:11-24).

Outputs (committed): tests/golden/segments_golden.npz, knn_distance_golden.json,
dummy_index_golden.npz.  The tests recompute the same quantities with oracle/ and with
the CUDA path and compare.
"""
import importlib.util
import json
import os
import sys
import types

import numpy as np

REF = os.environ.get("AUDIOMUSE_AI_SRC", "")
HERE = os.path.dirname(os.path.abspath(__file__))


def _stub(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


def _load(mod_name, rel):
    spec = importlib.util.spec_from_file_location(mod_name, os.path.join(REF, rel))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[mod_name] = mod
    spec.loader.exec_module(mod)
    return mod


# ---- shared deterministic stand-ins (also used by tests/test_oracle_golden.py) -------------
def golden_waveform(case_seed, length):
    rng = np.random.default_rng(case_seed)
    x = rng.standard_normal(length).astype(np.float32) * np.float32(0.4)
    x[::997] *= 4.0  # some samples exceed +-1: exercises the clip
    return x


def standin_mel(segment):
    return np.asarray(segment, dtype=np.float32)[np.newaxis, np.newaxis, np.newaxis, :]


def standin_encoder(mel):
    """Deterministic 512-d function of a segment: strided partial sums in float64."""
    seg = np.asarray(mel, dtype=np.float64).reshape(-1)
    n = (len(seg) // 512) * 512
    emb = seg[:n].reshape(-1, 512).sum(axis=0) + np.arange(512) * 1e-3
    return emb.astype(np.float32)[np.newaxis, :]


SEGMENT_CASE_LENGTHS = [1, 1000, 479_999, 480_000, 480_001, 700_000, 720_000, 720_001,
                        960_000, 1_199_999, 1_200_000, 1_440_000]


def main():
    if not os.path.isdir(os.path.join(REF, "tasks")):
        raise SystemExit("set AUDIOMUSE_AI_SRC to an AudioMuse-AI checkout")
    sys.path.insert(0, REF)
    os.environ.setdefault("TRANSFORMERS_NO_ADVISORY_WARNINGS", "1")
    import config  # the reference's config.py (pure env-var defaults)

    # --- stubs for absent third-party / heavy modules ------------------------------------
    _stub("psycopg2", extras=None, OperationalError=Exception)
    _stub("psycopg2.extras", DictCursor=object)
    tasks_pkg = _stub("tasks")
    tasks_pkg.__path__ = [os.path.join(REF, "tasks")]
    waveforms = {}
    _stub("tasks.analysis",
          robust_load_audio_with_fallback=lambda path, target_sr=48000: (waveforms[path], target_sr))
    _stub("tasks.mediaserver", create_instant_playlist=lambda *a, **k: None)
    _load("tasks.memory_utils", "tasks/memory_utils.py")
    clap = _load("tasks.clap_analyzer", "tasks/clap_analyzer.py")

    # --- analyze_audio_file with stand-in mel/encoder --------------------------------------
    seen = []

    class FakeSession:
        def run(self, _outs, feeds):
            mel = feeds["mel_spectrogram"]
            seen[-1].append(mel.reshape(-1))
            return [standin_encoder(mel)]

    clap.get_clap_audio_model = lambda: FakeSession()
    clap.compute_mel_spectrogram = lambda seg, sr=48000: standin_mel(seg)
    clap.comprehensive_memory_cleanup = lambda **k: None

    out = {"lengths": np.array(SEGMENT_CASE_LENGTHS, dtype=np.int64)}
    for ci, L in enumerate(SEGMENT_CASE_LENGTHS):
        path = f"case{ci}"
        waveforms[path] = golden_waveform(100 + ci, L)
        seen.append([])
        emb, dur, nseg = clap.analyze_audio_file(path)
        segs = seen[-1]
        assert emb is not None and nseg == len(segs)
        out[f"emb_{ci}"] = np.asarray(emb, dtype=np.float32)
        out[f"dur_{ci}"] = np.float64(dur)
        out[f"nseg_{ci}"] = np.int64(nseg)
        # fingerprints of each window the reference fed to the model
        out[f"seg_sum_{ci}"] = np.array([s.astype(np.float64).sum() for s in segs])
        out[f"seg_head_{ci}"] = np.stack([s[:8] for s in segs]).astype(np.float32)
        out[f"seg_tail_{ci}"] = np.stack([s[-8:] for s in segs]).astype(np.float32)

    # --- student_clap segment_audio / compute_segment_positions ----------------------------
    seg_mod = _load("ref_audio_segmentation", "student_clap/preprocessing/audio_segmentation.py")
    for ci, L in enumerate(SEGMENT_CASE_LENGTHS):
        pos = seg_mod.compute_segment_positions(L)
        out[f"positions_{ci}"] = np.array(pos, dtype=np.int64).reshape(-1, 2)
        out[f"nseg_student_{ci}"] = np.int64(len(seg_mod.segment_audio(np.zeros(L, np.float32))))
    np.savez_compressed(os.path.join(HERE, "segments_golden.npz"), **out)

    # --- voyager_manager distance helpers ------------------------------------------------
    vm = _load("tasks.voyager_manager", "tasks/voyager_manager.py")
    rng = np.random.default_rng(5)
    pairs = []
    fixed = [([1, 2, 3], [1, 2, 3]), ([1, 0], [0, 1]), ([1, 0], [-1, 0]), ([0, 0], [1, 1]),
             ([1, 1], [10, 10]), ([0, 0, 0], [3, 4, 0])]
    for a, b in fixed:
        pairs.append((np.array(a, np.float32), np.array(b, np.float32)))
    for d in (2, 200, 512):
        for _ in range(6):
            pairs.append((rng.standard_normal(d).astype(np.float32),
                          rng.standard_normal(d).astype(np.float32)))
    gold = []
    for a, b in pairs:
        gold.append({"a": a.tolist(), "b": b.tolist(),
                     "cosine": vm._get_direct_cosine_distance(a, b),
                     "euclidean": vm._get_direct_euclidean_distance(a, b)})
    gold.append({"a": None, "b": [1.0, 2.0], "cosine": vm._get_direct_cosine_distance(None, np.ones(2)),
                 "euclidean": vm._get_direct_euclidean_distance(None, np.ones(2))})
    with open(os.path.join(HERE, "knn_distance_golden.json"), "w") as f:
        json.dump({"metric": config.VOYAGER_METRIC, "cases": gold}, f,
                  default=lambda o: "inf" if o == float("inf") else o)

    # --- _filter_by_distance (voyager_manager.py:526-617): the greedy duplicate filter, both branches --------
    rng = np.random.default_rng(23)
    F = rng.standard_normal((400, 32)).astype(np.float32)
    F[200:] = F[:200] + 2e-3 * rng.standard_normal((200, 32)).astype(np.float32)   # near-duplicates of rows 0..199
    F[50:60] = F[40:50]                                                            # exact duplicates
    F /= np.linalg.norm(F, axis=1, keepdims=True)

    class _FakeIndex:
        def get_vector(self, i):
            return F[int(i)]

    class _Cur:
        def __enter__(self):
            return self

        def __exit__(self, *a):
            return False

        def execute(self, *a, **k):
            pass

        def fetchall(self):
            return []

    class _Conn:
        def cursor(self, *a, **k):
            return _Cur()

    vm.voyager_index = _FakeIndex()
    vm.reverse_id_map = {str(i): i for i in range(len(F))}
    vm.reverse_id_map["missing"] = None            # an item whose vector is unavailable: dropped by the filter
    fcases = {}
    for ci, (n_items, seed) in enumerate([(40, 1), (50, 2), (51, 3), (130, 4), (237, 5)]):
        q = np.random.default_rng(100 + seed).standard_normal(32).astype(np.float32)
        order = np.argsort(-(F @ q), kind="stable")[:n_items]      # a result list: closest first
        items = [str(int(i)) for i in order]
        if ci == 3:
            items[7] = "missing"
        for lb in (1, 3):
            vm.DUPLICATE_DISTANCE_CHECK_LOOKBACK = lb
            if hasattr(vm._get_cached_vector, "cache_clear"):
                vm._get_cached_vector.cache_clear()
            kept = vm._filter_by_distance([{"item_id": it} for it in items], _Conn())
            fcases[f"order_{ci}"] = np.array([-1 if it == "missing" else int(it) for it in items], dtype=np.int64)
            fcases[f"kept_{ci}_lb{lb}"] = np.array([int(s["item_id"]) for s in kept], dtype=np.int64)
    np.savez_compressed(os.path.join(HERE, "filter_golden.npz"), vectors=F,
                        threshold=np.float64(config.DUPLICATE_DISTANCE_THRESHOLD_COSINE),
                        batch=np.int64(vm.BATCH_SIZE_VECTOR_OPS), n_cases=np.int64(5), **fcases)

    # --- DummyVoyagerIndex (the reference tests' brute-force spec of query) ----------------
    tmod = _load("ref_test_clap_text_search", "tests/unit/test_clap_text_search.py")
    rng = np.random.default_rng(11)
    E = rng.standard_normal((500, 512)).astype(np.float32)
    E /= np.linalg.norm(E, axis=1, keepdims=True)
    Q = rng.standard_normal((8, 512)).astype(np.float32)
    Q /= np.linalg.norm(Q, axis=1, keepdims=True)
    idx = tmod.DummyVoyagerIndex(E)
    ids, dists = [], []
    for q in Q:
        i, d = idx.query(q, 50)
        ids.append(np.array(i, dtype=np.int64))
        dists.append(np.asarray(d, dtype=np.float32))
    np.savez_compressed(os.path.join(HERE, "dummy_index_golden.npz"), seed=np.int64(11),
                        ids=np.stack(ids), dists=np.stack(dists), n=np.int64(len(idx)))
    print("golden vectors written to", HERE)


if __name__ == "__main__":
    main()
