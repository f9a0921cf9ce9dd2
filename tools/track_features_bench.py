"""Track features (tempo / energy / tuning / chroma / key) on one B200: device-resident tracks/s for 3-minute tracks in
groups of 16, 64 and 256 (each call at most 2^26 samples), per-kernel ms, an HBM-bytes roofline view, end-to-end
tracks/s from host PCM for features + MusiCNN (all of analyze_track after decoding), and the numpy restatement's
seconds per track on the CPU.

    python tools/track_features_bench.py [--reps 5] [--out profiles/r04_track_features_bench.json]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

HBM_BW = 7.7e12   # bytes/s of one B200 (data sheet)
SR, TRACK = 16000, 180 * 16000


def hbm_bytes(n_samples, n_tracks):
    """Algorithmic HBM traffic of one call: PCM in, S written and read back by chroma, mel dB written and read by
    the onset pass, piptrack candidate slots written and read twice (median select: about 8 passes, histogram)."""
    T = n_samples // 512 + n_tracks
    pcm = 4 * n_samples
    s = 2 * 4 * 1025 * T
    d = 4 * 128 * T * 2 + 4 * T * 3
    cand = 8 * 40 * T * 10          # about 40 candidates per music frame, ~10 reads each
    return pcm + s + d + cand


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_track_features_bench.json"))
    args = ap.parse_args()

    import torch
    import __graft_entry__ as ge
    ge.build()
    from musicnn_bench import gpu_info
    from audiomuse_ai_b200 import _lib, musicnn as mm, track_features as tfm
    from oracle import musicnn as om, track_features as otf
    from tests import musicnn_export as me
    from tests.test_gpu_track_features import synthetic_music

    if not torch.cuda.is_available():
        raise SystemExit("track_features_bench needs a CUDA device")
    _lib.check(_lib.load().am_init(0))
    res = {"metric": "track_features", **gpu_info(), "track_seconds": 180, "hbm_datasheet_bytes_per_s": HBM_BW,
           "groups": {}}
    base = [synthetic_music(TRACK, 1000 + i) for i in range(16)]
    sess = tfm.FeatureSession()
    stream = torch.cuda.current_stream().cuda_stream
    per_call = (1 << 26) // TRACK   # 23 three-minute tracks per call
    for n in (16, 64, 256):
        pcm = torch.from_numpy(np.concatenate([base[i % 16] for i in range(n)])).cuda()
        offs = np.arange(n + 1, dtype=np.int64) * TRACK

        def group():
            for a in range(0, n, per_call):
                sess.run_dev(pcm.data_ptr(), offs[a:min(n, a + per_call) + 1], stream=stream)

        group()   # warm-up
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.reps):
            group()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / args.reps
        _lib.profile_report()
        _lib.profile_enable(True)
        group()
        torch.cuda.synchronize()
        prof = _lib.profile_report()
        _lib.profile_enable(False)
        b = hbm_bytes(n * TRACK, n)
        res["groups"][str(n)] = {"tracks": n, "calls": -(-n // per_call), "call_ms": dt * 1e3, "tracks_per_s": n / dt,
                                 "kernels_ms": prof, "hbm_bytes": b, "hbm_bound_ms": b / HBM_BW * 1e3,
                                 "share_of_hbm_bound": b / HBM_BW / dt}
        del pcm
    g = res["groups"][max(res["groups"], key=int)]
    ks = g["kernels_ms"]
    top = max(ks, key=lambda k: ks[k]["ms"] if isinstance(ks[k], dict) else ks[k]) if ks else None
    kind = "HBM bandwidth" if g["share_of_hbm_bound"] > 0.5 else "not HBM bandwidth (compute / latency)"
    res["bound"] = (f"{kind}: the call takes {g['call_ms']:.2f} ms against an HBM floor of {g['hbm_bound_ms']:.3f} ms; "
                    f"the largest kernel is {top}")

    # ---- end to end from host PCM: features + MusiCNN embedding + moods
    es = mm.MusicnnSession(me.export_embedding(om.MusicnnEmbedding(seed=0)))
    ps = mm.MusicnnSession(me.export_prediction(om.MusicnnPrediction(seed=1)))
    waves = [base[i % 16] for i in range(64)]
    tfm.track_features(waves[:4], session=sess)
    mm.analyze_tracks(waves[:4], es, ps)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    tfm.track_features(waves, session=sess)
    mm.analyze_tracks(waves, es, ps)
    dt = time.perf_counter() - t0
    res["end_to_end_from_host_pcm"] = {"tracks": 64, "seconds": dt, "tracks_per_s": 64 / dt}

    # ---- the numpy restatement on this host's CPU (not librosa)
    t0 = time.perf_counter()
    otf.analyze(base[0])
    res["cpu_numpy_restatement_seconds_per_track"] = time.perf_counter() - t0
    res["cpu_note"] = "oracle/track_features.py (numpy restatement), one 3-minute track; librosa itself not measured"
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
