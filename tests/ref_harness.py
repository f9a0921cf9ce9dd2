"""Golden-generator infrastructure: import the REFERENCE's own modules (read-only, from the AudioMuse-AI checkout
named by $AUDIOMUSE_AI_SRC) with inert stand-ins for the third-party packages that are not installed here (psycopg2,
voyager, the Flask app helpers), so their functions run unmodified -- over a recording brute-force index
(tests/golden/make_ref_trace.py), or over a recorder in front of audiomuse_ai_b200.voyager_compat
(tests/golden/make_shim_trace.py).

No test imports the reference: the tests replay what these generators stored under tests/golden/.
"""
from __future__ import annotations

import importlib.util
import json
import os
import re
import sys
import types
from typing import Dict, List, Optional

import numpy as np

REF = os.environ.get("AUDIOMUSE_AI_SRC", "")


def available() -> bool:
    return bool(REF) and os.path.isdir(os.path.join(REF, "tasks"))


# ------------------------------------------------------------------------------------------------ fake database
class FakeCursor:
    """Answers the handful of SQL statements tasks/voyager_manager.py and tasks/clap_text_search.py issue."""

    def __init__(self, db: "FakeDB", dict_rows: bool):
        self.db, self.dict_rows, self._rows = db, dict_rows, []

    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False

    def close(self):
        pass

    def execute(self, sql, params=None):
        s = " ".join(sql.split())
        db = self.db
        if s.startswith("SELECT item_id, embedding FROM embedding"):
            self._rows = [(i, e) for i, e in db.embeddings]
        elif s.startswith("SELECT item_id, embedding FROM clap_embedding") or "FROM clap_embedding" in s:
            self._rows = [(i, e) for i, e in db.clap_embeddings]
        elif s.startswith("DELETE FROM voyager_index_data") or s.startswith("DELETE FROM clap_index_data"):
            table = db.index_rows if "voyager_index_data" in s else db.clap_index_rows
            name = params[0]
            pat = re.compile("^" + re.escape(name) + r"_\d+_\d+$")
            for k in [k for k in table if k == name or pat.match(k)]:
                del table[k]
        elif s.startswith("INSERT INTO voyager_index_data") or s.startswith("INSERT INTO clap_index_data"):
            table = db.index_rows if "voyager_index_data" in s else db.clap_index_rows
            name, data, id_map_json, dim = params[:4]
            table[name] = (bytes(getattr(data, "adapted", data)), id_map_json, dim)
        elif s.startswith("SELECT index_data, id_map_json, embedding_dimension FROM"):
            table = db.index_rows if "voyager_index_data" in s else db.clap_index_rows
            r = table.get(params[0])
            self._rows = [r] if r else []
        elif s.startswith("SELECT index_name, index_data, id_map_json, embedding_dimension FROM"):
            table = db.index_rows if "voyager_index_data" in s else db.clap_index_rows
            self._rows = [(k,) + v for k, v in table.items()]
        elif "FROM score WHERE item_id = ANY" in s or "FROM score WHERE item_id IN" in s:
            ids = list(params[0])
            rows = [db.score[i] for i in ids if i in db.score]
            cols = [c.strip() for c in s[len("SELECT "):s.index(" FROM")].split(",")]
            self._rows = [DictRow({c: r.get(c) for c in cols}) if self.dict_rows else tuple(r.get(c) for c in cols) for r in rows]
        else:
            raise AssertionError(f"FakeDB: unexpected SQL: {s[:120]}")
        db.log.append(s[:60])

    def fetchone(self):
        return self._rows[0] if self._rows else None

    def fetchall(self):
        return list(self._rows)


class DictRow(dict):
    """psycopg2 DictRow stand-in: item access by column name, .get, and positional access."""

    def __getitem__(self, k):
        if isinstance(k, int):
            return list(self.values())[k]
        return dict.__getitem__(self, k)


class FakeDB:
    def __init__(self):
        self.embeddings: List = []        # (item_id, bytes)
        self.clap_embeddings: List = []
        self.index_rows: Dict[str, tuple] = {}
        self.clap_index_rows: Dict[str, tuple] = {}
        self.score: Dict[str, dict] = {}
        self.log: List[str] = []
        self.commits = 0

    def cursor(self, cursor_factory=None, **kw):
        return FakeCursor(self, cursor_factory is not None)

    def commit(self):
        self.commits += 1

    def rollback(self):
        pass


def make_score_table(n: int, seed: int = 0) -> Dict[str, dict]:
    """Track metadata with a few same-title/artist duplicates and prolific artists (exercises the reference's
    title/artist de-duplication and MAX_SONGS_PER_ARTIST cap)."""
    rng = np.random.default_rng(seed)
    artists = [f"Artist {a}" for a in range(max(4, n // 12))]
    out = {}
    for i in range(n):
        a = artists[int(rng.integers(0, len(artists)))]
        title = f"Song {i}" if i % 17 else f"Song {i - 1}"     # every 17th repeats its neighbour's title
        out[f"item{i}"] = {"item_id": f"item{i}", "title": title, "author": a, "album": f"Album {i % 50}",
                           "album_artist": a, "other_features": "danceable:0.5,aggressive:0.5,happy:0.5,party:0.5,relaxed:0.5,sad:0.5",
                           "mood_vector": "rock:0.5", "energy": 0.5, "tempo": 120.0, "key": "C", "scale": "major"}
    return out


# ------------------------------------------------------------------------------------------------ module loading
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


class Binary:
    """psycopg2.Binary stand-in."""

    def __init__(self, data):
        self.adapted = bytes(data)


def load_reference(voyager_module, db: FakeDB):
    """Imports the reference's config, tasks.voyager_manager and tasks.clap_text_search with `voyager` resolving to
    `voyager_module` and the database helpers to `db`.  Returns a namespace (config, vm, cts)."""
    if REF not in sys.path:
        sys.path.insert(0, REF)
    for k in [k for k in sys.modules if k == "tasks" or k.startswith("tasks.") or k in ("config", "app_helper", "voyager")]:
        del sys.modules[k]
    import config  # the reference's config.py (pure env-var defaults)

    sys.modules["voyager"] = voyager_module
    _stub("psycopg2", extras=None, OperationalError=Exception, Binary=Binary)
    _stub("psycopg2.extras", DictCursor=object)
    sys.modules["psycopg2"].extras = sys.modules["psycopg2.extras"]

    def get_score_data_by_ids(ids):
        return [dict(db.score[i]) for i in ids if i in db.score]

    _stub("app_helper", get_db=lambda: db, get_score_data_by_ids=get_score_data_by_ids)
    tasks_pkg = _stub("tasks")
    tasks_pkg.__path__ = [os.path.join(REF, "tasks")]
    _stub("tasks.mediaserver", create_instant_playlist=lambda *a, **k: None)
    vm = _load("tasks.voyager_manager", "tasks/voyager_manager.py")
    try:
        _load("tasks.memory_utils", "tasks/memory_utils.py")
    except Exception:
        pass
    cts = None
    try:
        cts = _load("tasks.clap_text_search", "tasks/clap_text_search.py")
    except Exception as e:  # optional: needs more of the app than the k-NN path
        cts = e
    return types.SimpleNamespace(config=config, vm=vm, cts=cts)


# ------------------------------------------------------------------------------------------------ recording index
class RecordingIndex:
    """Exact brute-force index with voyager's Cosine-space contract (unit-normalised stored rows, distance =
    1 - cos, ascending, ties by lower id: oracle/knn.py, itself pinned by the reference's DummyVoyagerIndex golden);
    every call the reference makes is appended to `trace`."""

    def __init__(self, rows: np.ndarray):
        from oracle import knn as oknn

        self._oknn = oknn
        self.rows = oknn.normalize_rows(rows)
        self.trace: List[dict] = []
        self.ef = 10

    def __len__(self):
        return len(self.rows)

    @property
    def num_elements(self):
        return len(self.rows)

    def get_vector(self, i):
        v = self.rows[int(i)].copy()
        self.trace.append({"op": "get_vector", "id": int(i), "vector": v})
        return v

    def query(self, vector, k):
        q = np.asarray(vector, dtype=np.float32)
        ids, dist = self._oknn.topk(self.rows, q[np.newaxis, :], int(k))
        ids, dist = ids[0].astype(np.uint64), dist[0].astype(np.float32)
        self.trace.append({"op": "query", "vector": q.copy(), "k": int(k), "ids": ids.astype(np.int64), "dist": dist.copy()})
        return ids, dist
