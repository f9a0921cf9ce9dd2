"""The reference's OWN index builder / loader and model factories over the shims, by replay of what they did
(tests/golden/shim_trace.json, written by tests/golden/make_shim_trace.py with `voyager` resolving to voyager_compat):
tasks/voyager_manager.py:145-460 stores a flat AMIX blob in the `voyager_index_data` rows, one row or
<name>_<i>_<n> segments of <= VOYAGER_MAX_PART_SIZE bytes with id_map_json in part 1 only, and loads it back; the
INTEGRATION.md section-3 patch makes the reference's factories construct the B200 classes.  Every voyager call the
reference made is repeated here against voyager_compat on the same seeded rows, and every value the reference read
back (saved bytes, element counts, exceptions) must come out the same.  Queries need the GPU:
tests/test_gpu_ref_trace.py covers them the same way."""
import builtins
import hashlib
import io
import json
import os
import sys
import tempfile
import types

import numpy as np
import pytest

from tests import ref_harness as rh
from tests.golden import make_shim_trace as gen


@pytest.fixture(scope="module")
def trace(golden_dir):
    with open(os.path.join(golden_dir, "shim_trace.json")) as f:
        return json.load(f)


def _sha(b: bytes) -> str:
    return hashlib.sha256(b).hexdigest()


def _rows(trace, n):
    """The rows the reference read from the embedding table (seeded as when the trace was recorded)."""
    return gen.fill(rh.FakeDB(), n, trace["embedding_dimension"])


def replay(calls, arrays, tmp_path):
    """Repeats the recorded voyager calls against voyager_compat.  `arrays` maps sha256 -> the array the reference
    passed; loads read back bytes saved earlier in the replay (or recorded inline).  Returns the index handles."""
    from audiomuse_ai_b200 import voyager_compat as vc

    handles, saved = {}, {}
    for c in calls:
        op = c["op"]
        if op == "Index":
            kw = dict(c["kwargs"])
            kw["space"] = vc.Space[kw["space"]]
            handles[c["h"]] = vc.Index(**kw)
        elif op == "add_items":
            v, ids = arrays[c["vectors"]["sha256"]], arrays[c["ids"]["sha256"]]
            assert (list(v.shape), str(v.dtype), list(ids.shape), str(ids.dtype)) == \
                (c["vectors"]["shape"], c["vectors"]["dtype"], c["ids"]["shape"], c["ids"]["dtype"])
            handles[c["h"]].add_items(v, ids=ids)
        elif op == "save":
            path = tmp_path / f"index_{c['h']}.voyager"
            handles[c["h"]].save(str(path))
            data = path.read_bytes()
            assert (len(data), _sha(data)) == (c["data"]["len"], c["data"]["sha256"]), "saved index bytes differ"
            saved[_sha(data)] = data
        elif op == "load":
            data = bytes.fromhex(c["data"]["hex"]) if "hex" in c["data"] else saved[c["data"]["sha256"]]
            stream = io.BytesIO(data) if c["stream"] == "BytesIO" else tempfile.TemporaryFile()
            if c["stream"] != "BytesIO":
                stream.write(data)
                stream.seek(0)
            with stream:
                if "raises" in c:
                    with pytest.raises(getattr(vc, c["raises"], None) or getattr(builtins, c["raises"])):
                        vc.Index.load(stream)
                else:
                    handles[c["h"]] = vc.Index.load(stream)
        elif op == "set":
            setattr(handles[c["h"]], c["attr"], c["value"])
        elif op == "get":
            assert getattr(handles[c["h"]], c["attr"]) == c["result"], c
        elif op == "len":
            assert len(handles[c["h"]]) == c["result"], c
        else:
            raise AssertionError(f"unknown recorded call {op}")
    return handles


def _check_build_and_load(trace, sc, n, tmp_path):
    """Replays one build + load and checks the stored rows against the bytes voyager_compat saved.  Returns
    (loaded index, saved bytes, rows)."""
    from audiomuse_ai_b200 import voyager_compat as vc

    x = _rows(trace, n)
    ids = np.arange(n, dtype=np.int64)
    calls = sc["voyager_calls"]
    assert [c["op"] for c in calls][:3] == ["Index", "add_items", "save"]
    h = replay(calls, {_sha(x.tobytes()): x, _sha(ids.tobytes()): ids}, tmp_path)
    loads = [c for c in calls if c["op"] == "load"]
    assert len(loads) == 1
    blob = vc.Index(vc.Space.Cosine, trace["embedding_dimension"])
    blob.add_items(x, ids=ids)
    blob = blob.as_bytes()
    assert blob[:4] == b"AMIX" and _sha(blob) == loads[0]["data"]["sha256"]   # what was stored is what was loaded
    idx = h[loads[0]["h"]]
    assert isinstance(idx, vc.Index) and len(idx) == n == sc["loaded"]["id_map_len"]
    np.testing.assert_array_equal(idx._rows, x)             # float32 rows survive the round trip bit for bit
    # the id map the reference stored: dense ids over the valid rows ("broken" / "short" skipped)
    id_map_json = json.dumps({i: f"item{i}" for i in range(n)}).encode()
    rows = sc["index_rows"]
    assert all(r["dim"] == trace["embedding_dimension"] for r in rows.values())
    first = rows[sc.get("row_order", [trace["index_name"]])[0]]
    assert first["id_map_json"]["sha256"] == _sha(id_map_json)
    assert (sc["loaded"]["id_map_first"], sc["loaded"]["id_map_last"]) == ("item0", f"item{n - 1}")
    return idx, blob, rows


def test_build_store_load_single_row(trace, tmp_path):
    sc = trace["single_row"]
    idx, blob, rows = _check_build_and_load(trace, sc, 500, tmp_path)
    assert list(rows) == [trace["index_name"]] and sc["commits"] == 1
    assert rows[trace["index_name"]]["data"]["sha256"] == _sha(blob)
    ef = [c["value"] for c in sc["voyager_calls"] if c["op"] == "set" and c["attr"] == "ef"]
    assert ef and idx.ef == ef[-1]


def test_build_store_load_segmented_rows(trace, tmp_path):
    """An index larger than VOYAGER_MAX_PART_SIZE is stored as <INDEX_NAME>_<part>_<total> rows (:410-436) and
    reassembled by the loader (:186-283)."""
    sc = trace["segmented_rows"]
    idx, blob, rows = _check_build_and_load(trace, sc, 4000, tmp_path)
    names = sc["row_order"]
    total = len(names)
    assert total == -(-len(blob) // gen.SEGMENT_PART_SIZE) >= 3
    assert names == [f"{trace['index_name']}_{i}_{total}" for i in range(1, total + 1)] and sorted(rows) == sorted(names)
    off = 0
    for n in names:                                         # each row is the next slice of the saved bytes
        part = blob[off:off + gen.SEGMENT_PART_SIZE]
        assert rows[n]["data"] == {"len": len(part), "sha256": _sha(part)}
        off += len(part)
    assert off == len(blob)
    assert rows[names[0]]["id_map_json"]["len"] > 2 and all(rows[n]["id_map_json"]["len"] == 0 for n in names[1:])
    assert [c["stream"] for c in sc["voyager_calls"] if c["op"] == "load"] == ["TemporaryFile"]
    # a missing segment aborts the load instead of serving a corrupt index (:224-227): no blob reaches the shim
    gone = trace["missing_segment"]
    assert gone["voyager_calls"] == [] and gone["loaded"] is None and len(gone["index_rows"]) == total - 1


def test_an_old_hnsw_blob_is_refused_and_the_loader_survives(trace, tmp_path):
    from audiomuse_ai_b200 import voyager_compat as vc

    sc = trace["old_hnsw_blob"]
    assert [(c["op"], c.get("raises")) for c in sc["voyager_calls"]] == [("load", "RuntimeError")]
    replay(sc["voyager_calls"], {}, tmp_path)                 # voyager_compat refuses the same bytes the same way
    assert sc["loaded"] is None                               # logged, cache left empty: rebuild path
    with pytest.raises(RuntimeError):
        vc.Index.load(io.BytesIO(b"VOYA" + b"\x00" * 64))


def test_integration_patch_applies_to_the_reference_modules(trace):
    from audiomuse_ai_b200 import clap_analyzer as b200_clap, clustering_gpu as b200_cg, integration
    from audiomuse_ai_b200 import voyager_compat as vc

    g = trace["integration"]
    old_voyager = sys.modules.get("voyager")
    integration.install_voyager_shim()
    try:
        assert sys.modules["voyager"] is vc
    finally:
        if old_voyager is None:
            sys.modules.pop("voyager", None)
        else:
            sys.modules["voyager"] = old_voyager
    ref_clap = types.ModuleType("tasks.clap_analyzer")
    for name in integration.CLAP_NAMES:
        assert name in g["clap_analyzer_functions"], name    # every patched name exists upstream with that spelling
        setattr(ref_clap, name, object())
    ref_vm, ref_cg = types.ModuleType("tasks.voyager_manager"), types.ModuleType("tasks.clustering_gpu")
    old = os.environ.pop("B200_ALLOW_SKLEARN_FALLBACK", None)
    try:
        integration.apply(clap=ref_clap, voyager_manager=ref_vm, clustering=ref_cg)
        assert os.environ.get("B200_ALLOW_SKLEARN_FALLBACK") == "1"        # the reference's silent-fallback contract
    finally:
        os.environ.pop("B200_ALLOW_SKLEARN_FALLBACK", None)
        if old is not None:
            os.environ["B200_ALLOW_SKLEARN_FALLBACK"] = old
    assert all(getattr(ref_clap, n) is getattr(b200_clap, n) for n in integration.CLAP_NAMES)
    assert ref_cg.check_gpu_available is b200_cg.check_gpu_available
    # the reference's k-NN paths call the module-level _filter_by_distance, which the patch replaces
    assert g["filter_by_distance_callers"] and ref_vm._filter_by_distance.__name__ == "_filter_by_distance_b200"
    # get_clustering_model / get_pca_model of the REFERENCE look the classes up at call time and construct them with
    # the recorded arguments (clustering_gpu.py:338-422): after the patch those are the B200 classes
    want = {"GPUKMeans": {"n_clusters": 7}, "GPUDBSCAN": {"eps": 0.5, "min_samples": 4}, "GPUPCA": {"n_components": 12}}
    assert sorted(f["constructs"]["class"] for f in g["factories"]) == sorted(want)
    for f in g["factories"]:
        c = f["constructs"]
        cls = getattr(ref_cg, c["class"])
        assert cls is getattr(b200_cg, c["class"])
        m = cls(*c["args"], **c["kwargs"])
        assert isinstance(m, cls) and all(getattr(m, k) == v for k, v in want[c["class"]].items())
