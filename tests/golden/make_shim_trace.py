#!/usr/bin/env python
"""Golden record of how the reference's index builder / loader and its model factories use this package's shims.

    AUDIOMUSE_AI_SRC=<AudioMuse-AI checkout> python tests/golden/make_shim_trace.py   # writes tests/golden/shim_trace.json

Runs, UNMODIFIED and with `voyager` resolving to a recorder that forwards every call to
audiomuse_ai_b200.voyager_compat,

    tasks.voyager_manager.build_and_store_voyager_index    (:294-460; one row, or <name>_<i>_<n> segments of
                                                             <= VOYAGER_MAX_PART_SIZE bytes with id_map_json in part 1)
    tasks.voyager_manager.load_voyager_index_for_querying  (:145-293; single row, segmented rows, a missing segment,
                                                             a voyager HNSW blob left over from an old install)

over an in-memory database, and stores each voyager call (constructor arguments, array shapes / dtypes / sha256, the
kind of stream handed to Index.load, the bytes saved or loaded as length + sha256, attribute reads and writes, raised
exceptions) with the rows the reference wrote.  It also applies the INTEGRATION.md section-3 patch to the reference's
tasks.clustering_gpu and records which class each factory call constructs and with which arguments, and which of the
patched names exist upstream.  tests/test_reference_shims.py replays all of it without the reference tree.  The saved
bytes are the persisted index format, so a change to that format shows up as a mismatch here.
"""
import ast
import hashlib
import importlib.util
import io
import json
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from tests import ref_harness as rh  # noqa: E402

SEGMENT_PART_SIZE = 1 << 20    # 1 MiB parts instead of 50 MB, so a 4000-row index is stored as several rows


def fill(db, n, d, seed=3):
    """n seeded float32 rows as item0..item<n-1>, plus a NULL blob and a wrong-dimension blob that the builder skips
    (:353-363).  Returns the n rows."""
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, d)).astype(np.float32)
    db.embeddings = [(f"item{i}", x[i].tobytes()) for i in range(n)]
    db.embeddings.insert(5, ("broken", None))
    db.embeddings.insert(9, ("short", np.zeros(d - 1, np.float32).tobytes()))
    return x


def _sha(b: bytes) -> str:
    return hashlib.sha256(b).hexdigest()


def _arr(a):
    a = np.ascontiguousarray(a)
    return {"shape": list(a.shape), "dtype": str(a.dtype), "sha256": _sha(a.tobytes())}


def _blob(b: bytes):
    d = {"len": len(b), "sha256": _sha(b)}
    if len(b) <= 256:
        d["hex"] = b.hex()
    return d


def recording_voyager(vc, log):
    """A `voyager` module whose Index forwards to vc.Index and appends each call to `log`."""
    m = types.ModuleType("voyager")
    m.Space, m.RecallError, m.StorageDataType = vc.Space, vc.RecallError, vc.StorageDataType
    handles = [0]

    class Index:
        def __init__(self, *args, _inner=None, **kw):
            object.__setattr__(self, "_h", handles[0])
            handles[0] += 1
            if _inner is None:
                assert not args, "positional constructor arguments are not recorded"
                log.append({"op": "Index", "h": self._h,
                            "kwargs": {k: (v.name if isinstance(v, vc.Space) else v) for k, v in kw.items()}})
                _inner = vc.Index(**kw)
            object.__setattr__(self, "_inner", _inner)

        def add_items(self, vectors, ids=None, **kw):
            assert not kw
            log.append({"op": "add_items", "h": self._h, "vectors": _arr(vectors), "ids": _arr(ids)})
            return self._inner.add_items(vectors, ids=ids)

        def save(self, target):
            self._inner.save(target)
            assert isinstance(target, str), "only saving to a path is recorded"
            with open(target, "rb") as f:
                data = f.read()
            log.append({"op": "save", "h": self._h, "target": "path", "data": _blob(data)})

        @classmethod
        def load(cls, stream, *a, **kw):
            assert not a and not kw and hasattr(stream, "read")
            data = stream.read()
            rec = {"op": "load", "stream": "BytesIO" if isinstance(stream, io.BytesIO) else "TemporaryFile",
                   "data": _blob(data)}
            log.append(rec)
            try:
                inner = vc.Index.load(io.BytesIO(data))
            except Exception as e:
                rec["raises"] = type(e).__name__
                raise
            out = cls(_inner=inner)
            rec["h"] = out._h
            return out

        def __len__(self):
            n = len(self._inner)
            log.append({"op": "len", "h": self._h, "result": n})
            return n

        def __setattr__(self, name, value):
            log.append({"op": "set", "h": self._h, "attr": name, "value": value})
            setattr(self._inner, name, value)

        def __getattr__(self, name):
            value = getattr(self._inner, name)
            log.append({"op": "get", "h": self._h, "attr": name, "result": value})
            return value

    m.Index = Index
    return m


def index_rows(db):
    return {name: {"data": _blob(data), "id_map_json": _blob(id_map_json.encode()), "dim": dim}
            for name, (data, id_map_json, dim) in db.index_rows.items()}


def index_state(vm):
    if vm.voyager_index is None:
        return None
    return {"id_map_len": len(vm.id_map), "id_map_first": vm.id_map[0], "id_map_last": vm.id_map[len(vm.id_map) - 1]}


def voyager_scenarios(vc):
    log = []
    db = rh.FakeDB()
    ref = rh.load_reference(recording_voyager(vc, log), db)
    vm, d = ref.vm, ref.config.EMBEDDING_DIMENSION
    out = {"embedding_dimension": d, "index_name": ref.config.INDEX_NAME}

    def run(tag, fn):
        del log[:]
        fn()
        out[tag] = {"voyager_calls": list(log), "index_rows": index_rows(db), "commits": db.commits,
                    "loaded": index_state(vm)}

    def build_then_load(n):
        fill(db, n, d)
        vm.build_and_store_voyager_index(db)
        vm.voyager_index = None
        vm.load_voyager_index_for_querying(force_reload=True)

    run("single_row", lambda: build_then_load(500))
    db.index_rows.clear()
    db.commits = 0
    vm.VOYAGER_MAX_PART_SIZE = SEGMENT_PART_SIZE
    run("segmented_rows", lambda: build_then_load(4000))
    segments = sorted(db.index_rows, key=lambda s: int(s.split("_")[-2]))
    out["segmented_rows"]["row_order"] = segments

    def drop_a_segment():
        del db.index_rows[segments[1]]
        vm.load_voyager_index_for_querying(force_reload=True)

    run("missing_segment", drop_a_segment)
    db.index_rows.clear()

    def old_blob():
        db.index_rows[ref.config.INDEX_NAME] = (b"VOYA" + b"\x00" * 64, json.dumps({"0": "item0"}), d)
        vm.load_voyager_index_for_querying(force_reload=True)

    run("old_hnsw_blob", old_blob)
    return ref, out


def integration_scenario(ref):
    from audiomuse_ai_b200 import integration

    spec = importlib.util.spec_from_file_location("tasks.clustering_gpu", os.path.join(rh.REF, "tasks", "clustering_gpu.py"))
    ref_cg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref_cg)
    with open(os.path.join(rh.REF, "tasks", "clap_analyzer.py")) as f:
        clap_defs = sorted(n.name for n in ast.parse(f.read()).body if isinstance(n, ast.FunctionDef))
    vm_callers = sorted(name for name, fn in vars(ref.vm).items()
                        if isinstance(fn, types.FunctionType) and "_filter_by_distance" in fn.__code__.co_names)
    integration.apply(voyager_manager=ref.vm, clustering=ref_cg, allow_sklearn_fallback=False)

    constructed = []
    for cls_name in ("GPUKMeans", "GPUDBSCAN", "GPUPCA"):
        cls = getattr(ref_cg, cls_name)

        def recorder(*args, _cls=cls, _name=cls_name, **kw):
            constructed.append({"class": _name, "args": list(args), "kwargs": kw})
            return _cls(*args, **kw)

        setattr(ref_cg, cls_name, recorder)
    calls = [("get_clustering_model", ["kmeans", {"n_clusters": 7}], {"use_gpu": True}),
             ("get_clustering_model", ["dbscan", {"eps": 0.5, "min_samples": 4}], {"use_gpu": True}),
             ("get_pca_model", [12], {"use_gpu": True})]
    factories = []
    for fn, args, kw in calls:
        del constructed[:]
        getattr(ref_cg, fn)(*args, **kw)
        assert len(constructed) == 1, constructed
        factories.append({"call": fn, "args": args, "kwargs": kw, "constructs": constructed[0]})
    return {"clap_analyzer_functions": clap_defs, "filter_by_distance_callers": vm_callers, "factories": factories}


def main():
    if not rh.available():
        raise SystemExit("set AUDIOMUSE_AI_SRC to an AudioMuse-AI checkout")
    from audiomuse_ai_b200 import voyager_compat as vc

    ref, out = voyager_scenarios(vc)
    out["integration"] = integration_scenario(ref)
    with open(os.path.join(HERE, "shim_trace.json"), "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print({k: len(v["voyager_calls"]) for k, v in out.items() if isinstance(v, dict) and "voyager_calls" in v})


if __name__ == "__main__":
    main()
