"""MusiCNN tower on one B200: device-resident patches/s, tracks/s from host PCM through the moods, the front-end
kernel's time and share of the bf16 peak (algorithmic flops from the graph's shapes), a cuDNN arm running the same
front end in the same process (conv2d + ReLU + BatchNorm + amax per branch, measurement only) and the oracle on the CPU.

    python tools/musicnn_bench.py [--batches 256,1024,4096] [--tracks 64] [--out profiles/musicnn_bench.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PEAK_BF16 = 2.25e15  # dense bf16 FLOP/s of one B200 (data sheet, 1000 W)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, pl, clk = [s.strip() for s in q.split(",")]
        return {"gpu": name, "power_limit": pl, "max_sm_clock": clk}
    except Exception as e:  # noqa: BLE001
        return {"gpu": "unknown", "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="256,1024,4096")
    ap.add_argument("--tracks", type=int, default=64)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "musicnn_bench.json"))
    args = ap.parse_args()

    import torch
    import __graft_entry__ as ge
    ge.build()
    from audiomuse_ai_b200 import _lib, musicnn as mm
    from oracle import musicnn as om
    from tests import musicnn_export as me

    if not torch.cuda.is_available():
        raise SystemExit("musicnn_bench needs a CUDA device")
    _lib.check(_lib.load().am_init(0))
    emb_m, pred_m = om.MusicnnEmbedding(seed=0), om.MusicnnPrediction(seed=1)
    es, ps = mm.MusicnnSession(me.export_embedding(emb_m)), mm.MusicnnSession(me.export_prediction(pred_m))
    total_f, front_f = es.flops_per_patch(om.N_FRAMES, om.N_MELS)
    res = {"metric": "musicnn", **gpu_info(), "flops_per_patch": total_f, "front_flops_per_patch": front_f,
           "peak_bf16_datasheet": PEAK_BF16, "arms": {}}
    dev = torch.device("cuda:0")
    stream = torch.cuda.current_stream().cuda_stream

    # ---- device-resident patches/s
    for B in [int(b) for b in args.batches.split(",")]:
        x = (torch.rand(B, om.N_FRAMES, om.N_MELS, device=dev) * 4.0).contiguous()
        out = torch.empty(B, 200, device=dev)
        for _ in range(2):
            es.run_dev(x.data_ptr(), B, om.N_FRAMES, om.N_MELS, out.data_ptr(), stream)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.reps):
            es.run_dev(x.data_ptr(), B, om.N_FRAMES, om.N_MELS, out.data_ptr(), stream)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.reps
        # per-kernel device times (separate pass with per-launch events)
        _lib.profile_report()
        _lib.profile_enable(True)
        for _ in range(args.reps):
            es.run_dev(x.data_ptr(), B, om.N_FRAMES, om.N_MELS, out.data_ptr(), stream)
        torch.cuda.synchronize()
        _lib.profile_enable(False)
        prof = _lib.profile_report()
        kern = {k: v["ms"] / args.reps for k, v in prof.items()}
        front_ms = sum(v for k, v in kern.items() if "musicnn_front_kernel" in k)
        arm = {"batch": B, "ms_per_call": ms, "patches_per_s": B / ms * 1e3, "kernel_ms_per_call": kern,
               "front_kernel_ms": front_ms,
               "front_share_of_bf16_peak": (front_f * B / PEAK_BF16) / (front_ms * 1e-3) if front_ms else None,
               "whole_call_share_of_bf16_peak": (total_f * B / PEAK_BF16) / (ms * 1e-3)}

        # ---- cuDNN arm: the same front end in torch (bf16 conv2d + ReLU + BatchNorm + amax), same patches
        xin = (x * emb_m.bn_in.weight.item() / (emb_m.bn_in.running_var.item() + emb_m.bn_in.eps) ** 0.5).to(torch.bfloat16)
        mods = []
        for conv, bn in list(emb_m.timbral) + list(emb_m.temporal):
            mods.append((conv.to(dev, torch.bfloat16), bn.to(dev, torch.bfloat16), conv in [c for c, _ in emb_m.timbral]))
        xi = xin.unsqueeze(1)
        xp = torch.nn.functional.pad(xi, (0, 0, 3, 3))

        def torch_front():
            outs = []
            for conv, bn, timbral in mods:
                outs.append(torch.amax(bn(torch.relu(conv(xp if timbral else xi))), dim=3))
            return torch.cat(outs, 1)

        torch.backends.cudnn.benchmark = True
        with torch.no_grad():
            for _ in range(3):
                torch_front()
            torch.cuda.synchronize()
            e0.record()
            for _ in range(args.reps):
                torch_front()
            e1.record()
            torch.cuda.synchronize()
        cud_ms = e0.elapsed_time(e1) / args.reps
        emb_m.float().cpu()
        arm["cudnn_front_ms"] = cud_ms
        arm["front_speedup_vs_cudnn"] = cud_ms / front_ms if front_ms else None
        res["arms"][f"patches_{B}"] = arm
        print(json.dumps(arm), flush=True)
        del x, out, xin, xi, xp
        torch.cuda.empty_cache()

    # ---- tracks/s: 3-minute 16 kHz tracks from host PCM through the moods
    rng = np.random.default_rng(0)
    tracks = [(0.2 * rng.standard_normal(180 * 16000)).astype(np.float32) for _ in range(args.tracks)]
    mm.analyze_tracks(tracks[:2], es, ps)
    t0 = time.perf_counter()
    reps = 3
    for _ in range(reps):
        r = mm.analyze_tracks(tracks, es, ps)
    dt = (time.perf_counter() - t0) / reps
    res["arms"]["tracks_3min"] = {"tracks": args.tracks, "s_per_call": dt, "tracks_per_s": args.tracks / dt,
                                  "patches_per_track": r[0][2]}
    print(json.dumps(res["arms"]["tracks_3min"]), flush=True)

    # ---- CPU baseline: the oracle on the CPU
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    xc = np.random.default_rng(1).random((16, om.N_FRAMES, om.N_MELS), dtype=np.float32) * 4
    om.embed_patches(emb_m, xc[:2])
    t0 = time.perf_counter()
    om.embed_patches(emb_m, xc)
    cpu = time.perf_counter() - t0
    res["cpu_baseline"] = {"kind": "oracle (PyTorch fp32 CPU)", "threads": torch.get_num_threads(),
                           "patches_per_s": 16 / cpu}
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "arms"}))


if __name__ == "__main__":
    main()
