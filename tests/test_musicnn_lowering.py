"""CPU checks of the MusiCNN tower's ONNX path: the oracle's exports, the lowered program am_musicnn_describe_file
prints (no GPU needed) and the refusal of an unsupported node by name."""
import numpy as np
import pytest
import torch

from oracle import musicnn as om, onnx_ref
from tests import musicnn_export as me


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from audiomuse_ai_b200 import _lib
    return _lib.load()


@pytest.mark.parametrize("spelling", ["torch", "tf"])
def test_embedding_exports_match_module(spelling):
    """Both spellings of the embedding file, interpreted node by node, against the module (< 1e-5)."""
    from oracle import onnx_ref_ext
    model = om.MusicnnEmbedding(seed=3)
    blob = (me.export_embedding if spelling == "torch" else me.export_embedding_tf)(model)
    g = onnx_ref.load(blob)
    assert g.inputs == [om.EMB_IN] and g.outputs == [om.EMB_OUT]
    ops = {n.op for n in g.nodes}
    if spelling == "tf":
        assert {"Transpose", "MaxPool", "Squeeze", "Mul", "MatMul"} <= ops and "BatchNormalization" not in ops
    x = np.random.default_rng(0).gamma(2.0, 0.6, (3, om.N_FRAMES, om.N_MELS)).astype(np.float32)
    want = om.embed_patches(model, x)
    got = onnx_ref_ext.run(g, {om.EMB_IN: x})[0]
    assert np.abs(got - want).max() <= 1e-5 * max(1.0, float(np.abs(want).max()))


@pytest.mark.parametrize("spelling", ["torch", "tf"])
def test_prediction_exports_match_module(spelling):
    pred = om.MusicnnPrediction(seed=4)
    g = onnx_ref.load((me.export_prediction if spelling == "torch" else me.export_prediction_tf)(pred))
    e = np.random.default_rng(0).standard_normal((5, 200)).astype(np.float32)
    np.testing.assert_allclose(onnx_ref.run(g, {om.PRED_IN: e})[0], om.predict(pred, e), rtol=1e-5, atol=1e-5)


def test_both_spellings_lower_to_the_same_program(lib, tmp_path):
    from audiomuse_ai_b200 import musicnn as mm
    model, pred = om.MusicnnEmbedding(seed=1), om.MusicnnPrediction(seed=1)
    progs = []
    for i, (e, p) in enumerate(((me.export_embedding, me.export_prediction),
                                (me.export_embedding_tf, me.export_prediction_tf))):
        (tmp_path / f"e{i}.onnx").write_bytes(e(model))
        (tmp_path / f"p{i}.onnx").write_bytes(p(pred))
        progs.append([mm.describe_file(str(tmp_path / f"{k}{i}.onnx")).split("\n", 1)[1] for k in "ep"])
    strip = lambda d: d.replace(" (window 59)", "").replace(" (window 30)", "").replace(" (window 96)", "")
    assert strip(progs[1][0]) == progs[0][0] and progs[1][1] == progs[0][1]
    assert "(window 59)" in progs[1][0]


def test_pre_residual_read_and_mixed_input_normalisation_are_rejected(lib, tmp_path):
    from audiomuse_ai_b200 import _lib, musicnn as mm

    class PoolsPreResidual(om.MusicnnEmbedding):
        def forward(self, x):   # pools mid-end layer 1 before its residual add as well as after it
            x = self.bn_in(x.unsqueeze(1))
            xp = torch.nn.functional.pad(x, (0, 0, 3, 3))
            f = torch.cat([torch.amax(bn(torch.relu(conv(xp))), dim=3) for conv, bn in self.timbral], 1)
            (c0, b0), (c1, b1) = self.mid[0], self.mid[1]
            m0 = b0(torch.relu(c0(f)))
            y1 = b1(torch.relu(c1(m0)))
            z = torch.cat([f, m0, y1, y1 + m0], 1)
            return self.dense(self.bn_pool(torch.cat([z.amax(2), z.mean(2)], 1)))

    class SkipsInputNorm(om.MusicnnEmbedding):
        def forward(self, x):   # the second branch reads the raw input
            xr = x.unsqueeze(1)
            xn = self.bn_in(xr)
            outs = [torch.amax(bn(torch.relu(conv(v))), dim=3) for (conv, bn), v in zip(self.temporal, (xn, xr))]
            f = torch.cat(outs, 1)
            conv, bn = self.mid[0]
            m0 = bn(torch.relu(conv(f)))
            z = torch.cat([f, m0], 1)
            return self.dense(self.bn_pool(torch.cat([z.amax(2), z.mean(2)], 1)))

    cases = ((PoolsPreResidual(timbral=((7, 38, 32),), temporal=(), mid=16, n_mid=3, emb=8), "before its residual add"),
             (SkipsInputNorm(timbral=(), temporal=((16, 16), (8, 16)), mid=16, n_mid=1, emb=8), "different normalisations"))
    for model, msg in cases:
        p = tmp_path / "bad.onnx"
        p.write_bytes(me.export_embedding(model))
        with pytest.raises(_lib.B200Error) as ei:
            mm.describe_file(str(p))
        assert msg in str(ei.value), str(ei.value)


def test_oracle_track_math():
    e = np.arange(6, dtype=np.float32).reshape(3, 2)
    emb, moods = om.track_result(e, np.zeros((3, 2), np.float32))
    np.testing.assert_allclose(emb, [2.0, 3.0])
    np.testing.assert_allclose(moods, 1 / (1 + np.exp(-0.5)))


def test_describe_lists_the_program(lib, tmp_path):
    from audiomuse_ai_b200 import musicnn as mm
    p = tmp_path / "musicnn_embedding.onnx"
    p.write_bytes(me.export_embedding(om.MusicnnEmbedding(seed=1)))
    d = mm.describe_file(str(p))
    for line in ("front 0: conv 7x38 cout=204 pad_time=3/3", "front 1: conv 7x67 cout=204",
                 "front 2: conv 128x1 cout=51 pad_time=63/64", "front 3: conv 64x1 cout=51",
                 "front 4: conv 32x1 cout=51 pad_time=15/16 relu bn max_freq -> channels [510, 561)",
                 "mid 0: conv1d k=7 561->64 relu bn\n", "mid 1: conv1d k=7 64->64 relu bn +residual",
                 "mid 2: conv1d k=7 64->64 relu bn +residual", "pool time max|mean over [ front mid0 mid1 mid2 ] -> 1506",
                 "head affine width=1506", "head linear 1506->200 +bias"):
        assert line in d, (line, d)
    q = tmp_path / "musicnn_prediction.onnx"
    q.write_bytes(me.export_prediction(om.MusicnnPrediction()))
    d = mm.describe_file(str(q))
    assert "input rows 200" in d and "head unary act=2 width=200" in d and "head linear 200->50 +bias" in d


def test_dimensions_come_from_the_graph(lib, tmp_path):
    from audiomuse_ai_b200 import musicnn as mm
    model = om.MusicnnEmbedding(timbral=((5, 20, 100),), temporal=((16, 24),), mid=32, n_mid=2, emb=40)
    p = tmp_path / "small.onnx"
    p.write_bytes(me.export_embedding(model))
    d = mm.describe_file(str(p))
    assert "front 0: conv 5x20 cout=100 pad_time=2/2" in d and "front 1: conv 16x1 cout=24 pad_time=7/8" in d
    assert "mid 1: conv1d k=7 32->32 relu bn +residual" in d and "head linear 376->40 +bias" in d


def test_unsupported_node_rejected_by_name(lib, tmp_path):
    from audiomuse_ai_b200 import _lib, musicnn as mm

    class Tanh(om.MusicnnPrediction):
        def forward(self, e):
            return torch.tanh(super().forward(e))

    p = tmp_path / "bad.onnx"
    p.write_bytes(me.export_prediction(Tanh()))
    with pytest.raises(_lib.B200Error) as ei:
        mm.describe_file(str(p))
    assert "cannot lower node 'Tanh_" in str(ei.value) and "(Tanh)" in str(ei.value)
