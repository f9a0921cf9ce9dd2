#!/usr/bin/env python
"""Golden "call traces" of the reference's own query functions, so that the tests need no reference tree.

    AUDIOMUSE_AI_SRC=<AudioMuse-AI checkout> python tests/golden/make_ref_trace.py   # writes tests/golden/ref_trace.npz

Runs, UNMODIFIED and over a recording brute-force index (tests/ref_harness.RecordingIndex = the reference tests'
DummyVoyagerIndex contract with float64 ranking and lower-id ties),

    tasks.voyager_manager.find_nearest_neighbors_by_vector   (:1547-1657; k = n + 4n and n + 0.2n expansions,
                                                              _filter_by_distance, title/artist de-dup, artist cap)
    tasks.voyager_manager.find_nearest_neighbors_by_id        (:1372-1545; get_vector + k = n + max(20, 3n) + 1, both the
                                                              standard branch and the radius walk :842-1367)
    tasks.voyager_manager.get_max_distance_for_id             (:1660-1702; k = len(index))
    tasks.clap_text_search.search_by_text                     (:448-532; text tower stubbed with a seeded vector)

on seeded libraries (3000 x 200 "music_library", 2000 x 512 CLAP) with an in-memory metadata table, and stores every
index call they made (query vector, k -> ids, distances; get_vector id -> vector) together with each function's final
answer.  tests/test_gpu_ref_trace.py replays the calls against audiomuse_ai_b200.voyager_compat.Index on the B200: if
every call returns what the recording index returned, the reference functions -- deterministic given those returns --
produce the recorded answers over the shim as well.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from tests import ref_harness as rh  # noqa: E402

N_MUSIC, D_MUSIC, N_CLAP, D_CLAP = 3000, 200, 2000, 512


def music_library():
    rng = np.random.default_rng(41)
    base = rng.standard_normal((60, D_MUSIC)).astype(np.float32)
    x = base[rng.integers(0, 60, N_MUSIC)] + 0.35 * rng.standard_normal((N_MUSIC, D_MUSIC)).astype(np.float32)
    x[1500:1560] = x[100:160] + 1e-3 * rng.standard_normal((60, D_MUSIC)).astype(np.float32)   # near-duplicate tracks
    return x.astype(np.float32)


def clap_library():
    rng = np.random.default_rng(43)
    x = rng.standard_normal((N_CLAP, D_CLAP)).astype(np.float32)
    return (x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32)


def main():
    db = rh.FakeDB()
    db.score = rh.make_score_table(N_MUSIC, 7)
    ref = rh.load_reference(types_voyager(), db)
    vm, cts = ref.vm, ref.cts
    X = music_library()
    rec = rh.RecordingIndex(X)
    vm.voyager_index = rec
    vm.id_map = {i: f"item{i}" for i in range(N_MUSIC)}
    vm.reverse_id_map = {v: k for k, v in vm.id_map.items()}
    calls, answers = [], {}

    def run(tag, fn):
        start = len(rec.trace)
        if hasattr(vm._get_cached_vector, "cache_clear"):
            vm._get_cached_vector.cache_clear()
        out = fn()
        answers[tag] = out
        for c in rec.trace[start:]:
            calls.append(dict(c, scenario=tag, index="music"))

    rng = np.random.default_rng(5)
    q1 = X[77] + 0.2 * rng.standard_normal(D_MUSIC).astype(np.float32)
    q2 = rng.standard_normal(D_MUSIC).astype(np.float32)
    run("by_vector_n100_dedupe", lambda: vm.find_nearest_neighbors_by_vector(q1, n=100, eliminate_duplicates=True))
    run("by_vector_n100_plain", lambda: vm.find_nearest_neighbors_by_vector(q2, n=100, eliminate_duplicates=False))
    run("by_vector_n25_default", lambda: vm.find_nearest_neighbors_by_vector(q1 * 3.0, n=25))
    run("by_id_n25_standard", lambda: vm.find_nearest_neighbors_by_id("item120", n=25, eliminate_duplicates=True,
                                                                     mood_similarity=False, radius_similarity=False))
    run("by_id_n10_plain", lambda: vm.find_nearest_neighbors_by_id("item9", n=10, eliminate_duplicates=False,
                                                                   mood_similarity=False, radius_similarity=False))
    run("by_id_n25_radius_walk", lambda: vm.find_nearest_neighbors_by_id("item300", n=25, eliminate_duplicates=True,
                                                                        mood_similarity=False, radius_similarity=True))
    run("max_distance", lambda: vm.get_max_distance_for_id("item42"))

    # ---- CLAP text search over its own index cache (clap_text_search.py:30-35)
    C = clap_library()
    crec = rh.RecordingIndex(C)
    if not isinstance(cts, Exception):
        cts._CLAP_INDEX_CACHE.update(index=crec, id_map={i: f"item{i}" for i in range(N_CLAP)},
                                     reverse_id_map={f"item{i}": i for i in range(N_CLAP)}, loaded=True)
        import types as _t
        text_vec = np.random.default_rng(99).standard_normal(D_CLAP).astype(np.float32)
        text_vec /= np.linalg.norm(text_vec)
        clap_stub = _t.ModuleType("tasks.clap_analyzer")
        clap_stub.get_text_embedding = lambda text: text_vec
        sys.modules["tasks.clap_analyzer"] = clap_stub
        cts.warmup_text_search_model = lambda *a, **k: None
        cts._fetch_clap_metadata = lambda ids: {i: {"title": db.score[i]["title"], "author": db.score[i]["author"]}
                                                for i in ids if i in db.score}
        start = len(crec.trace)
        answers["search_by_text_limit50"] = cts.search_by_text("upbeat summer songs", limit=50)
        for c in crec.trace[start:]:
            calls.append(dict(c, scenario="search_by_text_limit50", index="clap"))

    assert all(answers[k] for k in answers), {k: bool(v) for k, v in answers.items()}
    out = {"n_calls": np.int64(len(calls))}
    meta = []
    for i, c in enumerate(calls):
        meta.append({"op": c["op"], "scenario": c["scenario"], "index": c["index"], "k": c.get("k", 0), "id": c.get("id", -1)})
        out[f"vec_{i}"] = c["vector"]
        if c["op"] == "query":
            out[f"ids_{i}"] = c["ids"]
            out[f"dist_{i}"] = c["dist"]
    np.savez_compressed(os.path.join(HERE, "ref_trace.npz"), **out)
    with open(os.path.join(HERE, "ref_trace.json"), "w") as f:
        json.dump({"calls": meta, "answers": answers,
                   "libraries": {"music": [N_MUSIC, D_MUSIC, "make_ref_trace.music_library()"],
                                 "clap": [N_CLAP, D_CLAP, "make_ref_trace.clap_library()"]}}, f, indent=1)
    print(f"{len(calls)} index calls recorded; answers:", {k: (len(v) if hasattr(v, '__len__') else v) for k, v in answers.items()})


def types_voyager():
    """`import voyager` inside the reference resolves to a module that only needs RecallError / Space here."""
    import types
    m = types.ModuleType("voyager")

    class RecallError(RuntimeError):
        pass

    m.RecallError = RecallError
    m.Space = types.SimpleNamespace(Cosine=2, Euclidean=0, InnerProduct=1)
    m.Index = rh.RecordingIndex
    return m


if __name__ == "__main__":
    main()
