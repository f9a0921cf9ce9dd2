"""The `ort` proxy integration.apply(analysis=...) installs into tasks.analysis, on a fake onnxruntime module."""
import types

import pytest


class _RuntimeException(Exception):
    pass


def _fake_ort():
    ort = types.SimpleNamespace()
    ort.made = []
    ort.InferenceSession = lambda path, *a, **kw: ort.made.append((path, a, kw)) or ("real", path)
    ort.get_available_providers = lambda: ["CUDAExecutionProvider", "CPUExecutionProvider"]
    ort.capi = types.SimpleNamespace(onnxruntime_pybind11_state=types.SimpleNamespace(RuntimeException=_RuntimeException))
    return ort


def test_proxy_routes_musicnn_files_and_delegates_the_rest(monkeypatch):
    from audiomuse_ai_b200 import integration, musicnn

    made = []

    class FakeSession:
        def __init__(self, path):
            made.append(path)

    monkeypatch.setattr(musicnn, "MusicnnSession", FakeSession)
    real = _fake_ort()
    analysis = types.SimpleNamespace(ort=real)
    integration.apply(analysis=analysis)
    ort = analysis.ort
    assert isinstance(ort, integration.OrtProxy)
    s1 = ort.InferenceSession("/models/musicnn_embedding.onnx", providers=["CUDAExecutionProvider"])
    s2 = ort.InferenceSession("/models/musicnn_prediction.onnx", providers=["CPUExecutionProvider"])
    assert isinstance(s1, FakeSession) and isinstance(s2, FakeSession)
    assert made == ["/models/musicnn_embedding.onnx", "/models/musicnn_prediction.onnx"] and real.made == []
    assert ort.InferenceSession("/models/other.onnx", providers=["CPUExecutionProvider"]) == ("real", "/models/other.onnx")
    assert real.made == [("/models/other.onnx", (), {"providers": ["CPUExecutionProvider"]})]
    # names the reference's code and except clauses use stay valid
    assert ort.get_available_providers() == ["CUDAExecutionProvider", "CPUExecutionProvider"]
    with pytest.raises(ort.capi.onnxruntime_pybind11_state.RuntimeException):
        raise _RuntimeException("Failed to allocate memory")
    # applying twice does not stack proxies
    integration.apply(analysis=analysis)
    assert analysis.ort is ort


def test_apply_without_analysis_leaves_ort_alone():
    from audiomuse_ai_b200 import integration

    real = _fake_ort()
    analysis = types.SimpleNamespace(ort=real)
    integration.apply()
    assert analysis.ort is real
