"""Operators the MusiCNN exports need on top of ``oracle/onnx_ref.py``: ReduceMax, MaxPool, Concat, and Conv in its
1-D form and with ``auto_pad`` SAME_UPPER / SAME_LOWER.  TEST INFRASTRUCTURE ONLY.

``run(g, feeds)`` walks the graph node by node like ``onnx_ref.run``; the operators above are interpreted here (fp32,
PyTorch CPU, opset 17 semantics) and every other node is handed to ``onnx_ref.run`` as a one-node graph, so the
existing interpreter stays the single definition of the operators it already covers.
"""
from __future__ import annotations

from typing import Dict, List

import numpy as np

from . import onnx_ref


def _conv(x, w, b, a):
    import torch
    import torch.nn.functional as F

    nd = w.dim() - 2
    k = list(w.shape[2:])
    strides = list(a.get("strides", [1] * nd))
    dil = list(a.get("dilations", [1] * nd))
    ap = a.get("auto_pad", "NOTSET")
    ap = ap.decode() if isinstance(ap, bytes) else ap
    if ap in ("SAME_UPPER", "SAME_LOWER"):
        if any(s != 1 for s in strides):
            raise NotImplementedError("auto_pad with strides")
        tot = [d * (kk - 1) for d, kk in zip(dil, k)]
        lo = [t // 2 if ap == "SAME_UPPER" else t - t // 2 for t in tot]
        pads = lo + [t - l for t, l in zip(tot, lo)]
    elif ap in ("NOTSET", "VALID", "", None):
        pads = list(a.get("pads", [0] * (2 * nd)))
    else:
        raise NotImplementedError(f"auto_pad {ap}")
    tp = []
    for d in range(nd - 1, -1, -1):
        tp += [pads[d], pads[d + nd]]
    x = F.pad(x, tp)
    conv = F.conv1d if nd == 1 else F.conv2d
    return conv(x, w, b, stride=tuple(strides), dilation=tuple(dil), groups=a.get("group", 1))


def run(g: onnx_ref.Graph, feeds: Dict[str, np.ndarray]) -> List[np.ndarray]:
    import torch
    import torch.nn.functional as F

    env: Dict[str, "torch.Tensor"] = {k: torch.as_tensor(np.asarray(v)) for k, v in g.initializers.items()}
    for k, v in feeds.items():
        env[k] = torch.as_tensor(np.ascontiguousarray(v))
    with torch.no_grad():
        for n in g.nodes:
            a = n.attrs
            x = [env[i] if i else None for i in n.inputs]
            if n.op == "Conv":
                y = _conv(x[0], x[1], x[2] if len(x) > 2 else None, a)
            elif n.op == "ReduceMax":
                axes = [int(v) for v in x[1].tolist()] if len(x) > 1 and x[1] is not None else a.get("axes")
                y = x[0]
                if axes is None:
                    axes = list(range(y.dim()))
                y = torch.amax(y, dim=tuple(axes), keepdim=bool(a.get("keepdims", 1)))
            elif n.op == "MaxPool":
                k = list(a["kernel_shape"])
                if a.get("pads") and any(a["pads"]) or any(d != 1 for d in a.get("dilations", [1] * len(k))):
                    raise NotImplementedError("MaxPool with pads / dilations")
                st = list(a.get("strides", [1] * len(k)))
                y = (F.max_pool2d if len(k) == 2 else F.max_pool1d)(x[0], tuple(k), tuple(st))
            elif n.op == "Concat":
                y = torch.cat(x, dim=int(a["axis"]))
            else:
                sub = onnx_ref.Graph([n], {}, [i for i in n.inputs if i], [n.outputs[0]], g.opset)
                y = torch.as_tensor(onnx_ref.run(sub, {i: env[i].numpy() for i in n.inputs if i})[0])
            env[n.outputs[0]] = y
    return [env[o].numpy() for o in g.outputs]
