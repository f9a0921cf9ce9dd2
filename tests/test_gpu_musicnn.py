"""MusiCNN tower on the B200 vs the PyTorch oracle (oracle/musicnn.py), through the ONNX files the oracle exports."""
import numpy as np
import pytest

from oracle import musicnn as om
from tests import musicnn_export as me

pytestmark = pytest.mark.gpu


def _cos_rows(a, b):
    return np.sum(a * b, 1) / (np.linalg.norm(a, axis=1) * np.linalg.norm(b, axis=1))


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as ge
    ge.build()
    from audiomuse_ai_b200 import _lib
    _lib.check(_lib.load().am_init(0))


def _session(blob):
    from audiomuse_ai_b200 import musicnn as mm
    return mm.MusicnnSession(blob)


def _patches(n, seed):
    rng = np.random.default_rng(seed)
    # log10(1 + 10000 mel) lives in [0, ~5]
    return (rng.gamma(2.0, 0.6, size=(n, om.N_FRAMES, om.N_MELS))).astype(np.float32)


EXPORT = {"torch": (me.export_embedding, me.export_prediction), "tf": (me.export_embedding_tf, me.export_prediction_tf)}


@pytest.mark.parametrize("spelling", ["torch", "tf"])
@pytest.mark.parametrize("n", [1, 7, 300])
def test_embedding_matches_oracle(built, n, spelling):
    model = om.MusicnnEmbedding(seed=3)
    assert any((bn.weight < 0).any() for _, bn in model.timbral)   # negative BatchNorm scales are present
    sess = _session(EXPORT[spelling][0](model))
    x = _patches(n, n)
    got = sess.run(None, {om.EMB_IN: x})[0]
    want = om.embed_patches(model, x)
    cos = _cos_rows(got, want)
    print(f"{spelling} n={n} min cosine {cos.min():.6f}")
    assert got.shape == (n, 200) and 1.0 - cos.min() <= 1e-3


@pytest.mark.parametrize("spelling", ["torch", "tf"])
@pytest.mark.parametrize("variant", ["timbral", "temporal"])
def test_reduced_variants(built, variant, spelling):
    if variant == "timbral":
        model = om.MusicnnEmbedding(timbral=((7, 38, 204),), temporal=(), seed=5)
    else:
        model = om.MusicnnEmbedding(timbral=(), temporal=((128, 51),), seed=6)
    sess = _session(EXPORT[spelling][0](model))
    x = _patches(9, 11)
    cos = _cos_rows(sess.run(None, {om.EMB_IN: x})[0], om.embed_patches(model, x))
    print(f"{spelling} {variant}: min cosine {cos.min():.6f}")
    assert 1.0 - cos.min() <= 1e-3


@pytest.mark.parametrize("spelling", ["torch", "tf"])
def test_prediction_matches_oracle(built, spelling):
    pred = om.MusicnnPrediction(seed=2)
    sess = _session(EXPORT[spelling][1](pred))
    e = np.random.default_rng(0).standard_normal((33, 200)).astype(np.float32)
    got = sess.run([om.PRED_OUT], {om.PRED_IN: e})[0]
    np.testing.assert_allclose(got, om.predict(pred, e), rtol=1e-4, atol=1e-4)


def test_bulk_tracks_match_oracle_pipeline(built):
    from audiomuse_ai_b200 import musicnn as mm
    from oracle import mel as omel
    emb_m, pred_m = om.MusicnnEmbedding(seed=7), om.MusicnnPrediction(seed=8)
    es, ps = _session(me.export_embedding(emb_m)), _session(me.export_prediction(pred_m))
    rng = np.random.default_rng(4)
    lens = [16000 * 3 + 4000, 1000, 16000 * 9, 16000 * 6 + 123]   # 1 patch, too short, 3 patches, 2 patches
    tracks = [(0.3 * rng.standard_normal(L)).astype(np.float32) for L in lens]
    res = mm.analyze_tracks(tracks, es, ps)
    assert res[1] is None
    for w, r in zip(tracks, res):
        if r is None:
            continue
        p = np.asarray(omel.musicnn_patches(w), dtype=np.float32)
        ep = om.embed_patches(emb_m, p)
        want_e, want_m = om.track_result(ep, om.predict(pred_m, ep))
        e, moods, npch = r
        assert npch == p.shape[0]
        cos = float(np.dot(e, want_e) / (np.linalg.norm(e) * np.linalg.norm(want_e)))
        print(f"patches={npch} cosine {cos:.6f} max mood err {np.abs(moods - want_m).max():.2e}")
        assert 1.0 - cos <= 1e-3
        assert np.abs(moods - want_m).max() <= 1e-3


def _find_onnx_name(candidate_name, names):
    """tasks/analysis.py:110-127, restated: exact, without ':0', the last path component, '/' -> '_', else the first."""
    if candidate_name in names:
        return candidate_name
    stripped = candidate_name.split(":")[0]
    if stripped in names:
        return stripped
    if stripped.split("/")[-1] in names:
        return stripped.split("/")[-1]
    if stripped.replace("/", "_") in names:
        return stripped.replace("/", "_")
    return names[0] if names else None


def _run_inference(sess, feed_dict, output_tensor_name):
    """tasks/analysis.py:129-170, restated: map the feed names and the output name through the session's own lists."""
    input_names = [i.name for i in sess.get_inputs()]
    output_names = [o.name for o in sess.get_outputs()]
    mapped = {_find_onnx_name(k, input_names): v for k, v in feed_dict.items()}
    return sess.run([_find_onnx_name(output_tensor_name, output_names)], mapped)[0]


@pytest.mark.parametrize("spelling", ["torch", "tf"])
def test_sessions_through_the_ort_proxy_replay_run_inference(built, tmp_path, spelling):
    """The sessions integration.apply(analysis=...) hands out for the two model files answer run_inference with the
    names of DEFINED_TENSOR_NAMES (analysis.py:81-93)."""
    import types
    from audiomuse_ai_b200 import integration

    names = {"embedding": {"input": om.EMB_IN, "output": om.EMB_OUT},
             "prediction": {"input": om.PRED_IN, "output": om.PRED_OUT}}
    emb_m, pred_m = om.MusicnnEmbedding(seed=9), om.MusicnnPrediction(seed=10)
    (tmp_path / "musicnn_embedding.onnx").write_bytes(EXPORT[spelling][0](emb_m))
    (tmp_path / "musicnn_prediction.onnx").write_bytes(EXPORT[spelling][1](pred_m))
    real = types.SimpleNamespace(InferenceSession=lambda *a, **k: pytest.fail("routed to onnxruntime"),
                                 get_available_providers=lambda: ["CPUExecutionProvider"])
    analysis = types.SimpleNamespace(ort=real)
    integration.apply(analysis=analysis)
    providers = ["CPUExecutionProvider"]
    es = analysis.ort.InferenceSession(str(tmp_path / "musicnn_embedding.onnx"), providers=providers)
    ps = analysis.ort.InferenceSession(str(tmp_path / "musicnn_prediction.onnx"), providers=providers)
    x = _patches(4, 2)
    e = _run_inference(es, {names["embedding"]["input"]: x}, names["embedding"]["output"])
    logits = _run_inference(ps, {names["prediction"]["input"]: e}, names["prediction"]["output"])
    assert 1.0 - _cos_rows(e, om.embed_patches(emb_m, x)).min() <= 1e-3
    np.testing.assert_allclose(logits, om.predict(pred_m, e), rtol=1e-4, atol=1e-4)
    es.release_workspace()
    np.testing.assert_array_equal(e, _run_inference(es, {names["embedding"]["input"]: x}, names["embedding"]["output"]))
