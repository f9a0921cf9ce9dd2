"""Test helper: write the MusiCNN oracle modules (oracle/musicnn.py) to ONNX under the reference's tensor names
(tasks/analysis.py:81-93, DEFINED_TENSOR_NAMES), through the same TorchScript exporter stages as tests/onnx_export.py.
"""
from __future__ import annotations

import warnings

import torch


def _export(model: torch.nn.Module, x: torch.Tensor, in_name: str, out_name: str) -> bytes:
    from torch.onnx._internal.torchscript_exporter import utils as U

    model.eval()
    dyn = {in_name: {0: "batch"}}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        graph, params, _ = U._model_to_graph(model, (x,), input_names=[in_name], output_names=[out_name],
                                             do_constant_folding=True, dynamic_axes=dyn)
        proto = graph._export_onnx(params, 17, dyn, False, torch.onnx.OperatorExportTypes.ONNX, True, True, {}, True,
                                   "", {})[0]
    return bytes(proto)


def export_embedding(model: torch.nn.Module) -> bytes:
    from oracle import musicnn as om

    return _export(model, torch.randn(2, om.N_FRAMES, om.N_MELS), om.EMB_IN, om.EMB_OUT)


def export_prediction(model: torch.nn.Module, emb: int = 200) -> bytes:
    from oracle import musicnn as om

    return _export(model, torch.randn(2, emb), om.PRED_IN, om.PRED_OUT)


def _affine(bn) -> "tuple[torch.Tensor, torch.Tensor]":
    s = bn.weight / torch.sqrt(bn.running_var + bn.eps)
    return s.detach().clone(), (bn.bias - bn.running_mean * s).detach().clone()


class TfStyleEmbedding(torch.nn.Module):
    """The same function as an oracle MusicnnEmbedding, spelled the way tf2onnx writes the TF graph: NHWC input
    (Unsqueeze + Transpose), BatchNorm as constant Mul / Add, an explicit Pad before every convolution, the frequency
    max as MaxPool [1, W] + Squeeze, the mid-end as a [7, C] convolution over the padded (time, channel) image, and the
    dense layer as MatMul + Add."""

    def __init__(self, m, n_mels: int = 96):
        super().__init__()
        self.m = m
        s, h = _affine(m.bn_in)
        self.register_buffer("s_in", s.reshape(()))
        self.register_buffer("h_in", h.reshape(()))
        self.br = []
        for i, (conv, bn) in enumerate(list(m.timbral) + list(m.temporal)):
            kh, kw = conv.kernel_size
            timbral = i < len(m.timbral)
            top = m.front_pad if timbral else (kh - 1) // 2
            bot = m.front_pad if timbral else kh - 1 - (kh - 1) // 2
            s, h = _affine(bn)
            self.register_buffer(f"bs{i}", s.reshape(1, -1, 1, 1))
            self.register_buffer(f"bh{i}", h.reshape(1, -1, 1, 1))
            self.br.append((conv, top, bot, n_mels - kw + 1))
        for j, (conv, bn) in enumerate(m.mid):
            self.register_buffer(f"mw{j}", conv.weight.detach().permute(0, 2, 1).unsqueeze(1).contiguous())
            self.register_buffer(f"mb{j}", conv.bias.detach().clone())
            s, h = _affine(bn)
            self.register_buffer(f"ms{j}", s.reshape(1, -1, 1, 1))
            self.register_buffer(f"mh{j}", h.reshape(1, -1, 1, 1))
        s, h = _affine(m.bn_pool)
        self.register_buffer("ps", s)
        self.register_buffer("ph", h)
        self.register_buffer("dw", m.dense.weight.detach().t().contiguous())
        self.register_buffer("db", m.dense.bias.detach().clone())

    def forward(self, x):
        F = torch.nn.functional
        x = x.unsqueeze(3).permute(0, 3, 1, 2)                           # NHWC [B, T, F, 1] -> [B, 1, T, F]
        x = x * self.s_in + self.h_in
        outs = []
        for i, (conv, top, bot, w_out) in enumerate(self.br):
            y = torch.relu(F.conv2d(F.pad(x, (0, 0, top, bot)), conv.weight, conv.bias))
            y = y * getattr(self, f"bs{i}") + getattr(self, f"bh{i}")
            outs.append(F.max_pool2d(y, (1, w_out)).squeeze(3))           # [B, c, T]
        f = torch.cat(outs, 1)
        series, h = [f], f
        for j in range(len(self.m.mid)):
            img = F.pad(h.permute(0, 2, 1).unsqueeze(1), (0, 0, 3, 3))     # [B, 1, T + 6, C]
            y = torch.relu(F.conv2d(img, getattr(self, f"mw{j}"), getattr(self, f"mb{j}")))   # [B, 64, T, 1]
            y = (y * getattr(self, f"ms{j}") + getattr(self, f"mh{j}")).squeeze(3)
            h = y + h if j > 0 else y
            series.append(h)
        z = torch.cat(series, 1)
        p = torch.cat([z.amax(2), z.mean(2)], 1)
        return (p * self.ps + self.ph) @ self.dw + self.db


class TfStylePrediction(torch.nn.Module):
    """An oracle MusicnnPrediction as Relu -> Mul -> Add -> MatMul -> Add."""

    def __init__(self, m):
        super().__init__()
        s, h = _affine(m.bn)
        self.register_buffer("s", s)
        self.register_buffer("h", h)
        self.register_buffer("w", m.dense.weight.detach().t().contiguous())
        self.register_buffer("b", m.dense.bias.detach().clone())

    def forward(self, e):
        return (torch.relu(e) * self.s + self.h) @ self.w + self.b


def export_embedding_tf(model: torch.nn.Module) -> bytes:
    from oracle import musicnn as om

    return _export(TfStyleEmbedding(model), torch.randn(2, om.N_FRAMES, om.N_MELS), om.EMB_IN, om.EMB_OUT)


def export_prediction_tf(model: torch.nn.Module, emb: int = 200) -> bytes:
    from oracle import musicnn as om

    return _export(TfStylePrediction(model), torch.randn(2, emb), om.PRED_IN, om.PRED_OUT)
