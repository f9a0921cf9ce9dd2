"""PyTorch restatement of the MSD MusiCNN tower behind ``musicnn_embedding.onnx`` / ``musicnn_prediction.onnx``
(tasks/analysis.py:324-573), test infrastructure only.

The network is Pons & Serra's ``build_musicnn`` (musicnn/models.py) with front-end factor 1.6, 64 mid-end filters
and 200 back-end units, for 187 x 96 log-mel patches:

* input BatchNorm (one scalar channel);
* timbral branches: pad time by 3, conv 7 x int(0.4 * 96) and 7 x int(0.7 * 96), 204 filters each, valid;
  temporal branches: conv 128 x 1, 64 x 1, 32 x 1, 51 filters each, same padding; every branch is
  conv -> ReLU -> BatchNorm -> max over frequency;
* mid-end: three 7-tap convolutions over time (64 filters, zero padding 3), ReLU -> BatchNorm, residual adds on
  the second and third;
* back-end: [front | m1 | m2 | m3] -> max and mean over time -> BatchNorm -> dense; the embedding is the dense
  output BEFORE its ReLU (``model/dense/BiasAdd:0``);
* prediction model: ReLU -> BatchNorm -> dense to 50 logits.

Weights are seeded; BatchNorm statistics are realistic and include negative scales (a negative scale after the
ReLU turns the frequency max into a min, which the engine must honour).  Parity with the published ONNX files is
not pinned: they are not available offline.
"""
from __future__ import annotations

from typing import Sequence, Tuple

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

N_FRAMES, N_MELS = 187, 96
EMB_IN, EMB_OUT, PRED_IN, PRED_OUT = "model/Placeholder:0", "model/dense/BiasAdd:0", \
    "serving_default_model_Placeholder:0", "PartitionedCall:0"


def _bn(c: int, g: torch.Generator, d: int = 2) -> nn.Module:
    bn = (nn.BatchNorm2d if d == 2 else nn.BatchNorm1d)(c, eps=1e-3)
    with torch.no_grad():
        scale = 0.5 + torch.rand(c, generator=g)
        sign = torch.where(torch.rand(c, generator=g) < 0.2, -1.0, 1.0)
        bn.weight.copy_(scale * sign)
        bn.bias.copy_(0.1 * torch.randn(c, generator=g))
        bn.running_mean.copy_(0.2 * torch.randn(c, generator=g))
        bn.running_var.copy_(0.5 + torch.rand(c, generator=g))
    return bn


class MusicnnEmbedding(nn.Module):
    """[B, 187, 96] log-mel patches -> [B, emb] dense outputs before the ReLU."""

    def __init__(self, timbral: Sequence[Tuple[int, int, int]] = ((7, 38, 204), (7, 67, 204)),
                 temporal: Sequence[Tuple[int, int]] = ((128, 51), (64, 51), (32, 51)),
                 mid: int = 64, n_mid: int = 3, emb: int = 200, seed: int = 0):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.bn_in = _bn(1, g)
        self.timbral = nn.ModuleList()
        self.temporal = nn.ModuleList()
        for kh, kw, c in timbral:
            conv = nn.Conv2d(1, c, (kh, kw))
            self.timbral.append(nn.ModuleList([conv, _bn(c, g)]))
        for kh, c in temporal:
            conv = nn.Conv2d(1, c, (kh, 1), padding="same")
            self.temporal.append(nn.ModuleList([conv, _bn(c, g)]))
        self.front_pad = max([kh for kh, _, _ in timbral], default=1) // 2
        c_front = sum(c for _, _, c in timbral) + sum(c for _, c in temporal)
        self.mid = nn.ModuleList()
        cin = c_front
        for _ in range(n_mid):
            self.mid.append(nn.ModuleList([nn.Conv1d(cin, mid, 7, padding=3), _bn(mid, g, 1)]))
            cin = mid
        self.c_front, self.c_cat = c_front, c_front + n_mid * mid
        self.bn_pool = _bn(2 * self.c_cat, g, 1)
        self.dense = nn.Linear(2 * self.c_cat, emb)
        with torch.no_grad():
            for m in self.modules():
                if isinstance(m, (nn.Conv2d, nn.Conv1d, nn.Linear)):
                    fan_in = m.weight[0].numel()
                    m.weight.copy_(torch.randn(m.weight.shape, generator=g) * (1.5 / fan_in) ** 0.5)
                    m.bias.copy_(0.05 * torch.randn(m.bias.shape, generator=g))
        self.eval()

    def forward(self, x):
        x = self.bn_in(x.unsqueeze(1))                                   # [B, 1, 187, 96]
        xp = F.pad(x, (0, 0, self.front_pad, self.front_pad))
        outs = []
        for conv, bn in self.timbral:
            outs.append(torch.amax(bn(torch.relu(conv(xp))), dim=3))    # [B, c, 187]
        for conv, bn in self.temporal:
            outs.append(torch.amax(bn(torch.relu(conv(x))), dim=3))
        f = torch.cat(outs, 1)                                           # [B, 561, 187]
        series = [f]
        h = f
        for i, (conv, bn) in enumerate(self.mid):
            y = bn(torch.relu(conv(h)))
            h = y + h if i > 0 else y
            series.append(h)
        z = torch.cat(series, 1)                                         # [B, 753, 187]
        p = torch.cat([z.amax(2), z.mean(2)], 1)                         # [B, 1506]
        return self.dense(self.bn_pool(p))


class MusicnnPrediction(nn.Module):
    """[B, emb] embeddings -> [B, n_out] raw logits: ReLU -> BatchNorm -> dense."""

    def __init__(self, emb: int = 200, n_out: int = 50, seed: int = 1):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.bn = _bn(emb, g, 1)
        self.dense = nn.Linear(emb, n_out)
        with torch.no_grad():
            # logits of a few units around -2: per-patch tag probabilities mostly below 0.3, so the double sigmoid
            # lands in the 0.5-0.57 band the reference's comment describes for real tracks (analysis.py:513-520)
            self.dense.weight.copy_(torch.randn(n_out, emb, generator=g) * (0.02 / emb) ** 0.5)
            self.dense.bias.copy_(-2.0 + 0.5 * torch.randn(n_out, generator=g))
        self.eval()

    def forward(self, e):
        return self.dense(self.bn(torch.relu(e)))


def embed_patches(model: MusicnnEmbedding, patches: np.ndarray) -> np.ndarray:
    with torch.no_grad():
        return model(torch.as_tensor(np.ascontiguousarray(patches, dtype=np.float32))).numpy()


def predict(model: MusicnnPrediction, emb: np.ndarray) -> np.ndarray:
    with torch.no_grad():
        return model(torch.as_tensor(np.ascontiguousarray(emb, dtype=np.float32))).numpy()


def sigmoid(x: np.ndarray) -> np.ndarray:
    return 1.0 / (1.0 + np.exp(-x))


def track_result(emb_patches: np.ndarray, logits: np.ndarray):
    """The reference's track math: embedding = mean of the patch embeddings (analysis.py:544, no normalisation),
    moods = sigmoid(mean(sigmoid(logits))) (analysis.py:521-522)."""
    return emb_patches.mean(axis=0), sigmoid(sigmoid(logits).mean(axis=0))
