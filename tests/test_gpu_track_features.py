"""Track features (tempo, energy, tuning, chroma, key) on the B200 vs the numpy restatement oracle/track_features.py,
and the analyze_track drop-in of integration.make_analyze_track."""
import types

import numpy as np
import pytest

from oracle import track_features as otf

pytestmark = pytest.mark.gpu

SR = 16000
# 1 sample, 511, 512, one MusiCNN patch, 30 s, 3 min, 10 min, and lengths off the hop grid
LENGTHS = [1, 511, 512, 48128, 30 * SR, 180 * SR, 600 * SR, 20 * SR + 77, 45 * SR + 511, 7 * SR + 1]


def synthetic_music(n, seed):
    """Harmonic notes with attack / decay envelopes on a beat grid, clicks and noise."""
    rng = np.random.default_rng(seed)
    y = (0.01 * rng.standard_normal(n)).astype(np.float64)
    if n < 64:
        return y.astype(np.float32)
    beat = int(rng.integers(5000, 12000))
    detune = rng.uniform(-0.45, 0.45)
    root = int(rng.integers(48, 60))
    scale = [0, 2, 4, 5, 7, 9, 11] if rng.random() < 0.5 else [0, 2, 3, 5, 7, 8, 10]
    for s in range(0, n, beat):
        L = min(beat * 2, n - s)
        t = np.arange(L) / SR
        env = np.exp(-t * rng.uniform(2, 6)) * np.minimum(1.0, t * 200)
        midi = root + scale[int(rng.integers(0, 7))] + 12 * int(rng.integers(0, 2)) + detune
        f0 = 440.0 * 2 ** ((midi - 69) / 12)
        note = sum((0.6 ** h) * np.sin(2 * np.pi * f0 * (h + 1) * t + rng.uniform(0, 6.28)) for h in range(5))
        y[s:s + L] += 0.2 * env * note
        y[s:s + min(40, L)] += 0.5 * rng.standard_normal(min(40, L))
    return y.astype(np.float32)


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as ge
    ge.build()
    from audiomuse_ai_b200 import _lib
    _lib.check(_lib.load().am_init(0))


@pytest.fixture(scope="module")
def tracks():
    return [synthetic_music(L, 100 + i) for i, L in enumerate(LENGTHS)]


@pytest.fixture(scope="module")
def device_run(built, tracks):
    from audiomuse_ai_b200 import track_features as tfm
    sess = tfm.FeatureSession()
    feats, tg = sess.run(tracks, tempogram=True)
    return sess, feats, tg


@pytest.fixture(scope="module")
def oracle_runs(tracks):
    return [otf.analyze(y) for y in tracks]


def test_continuous_values(device_run, oracle_runs, tracks):
    _, feats, tg = device_run
    for y, f, o, g in zip(tracks, feats, oracle_runs, tg):
        assert f.n_frames == otf.n_frames(len(y))
        assert abs(f.energy - o["energy"]) <= 1e-5 * abs(o["energy"]), (len(y), f.energy, o["energy"])
        cm = np.array(f.chroma_mean[:], np.float32)
        # chroma depends on the tuning: compare where both chose the same bin
        if f.tuning == o["tuning"]:
            assert np.abs(cm - o["chroma_mean"]).max() <= 1e-4, (len(y), cm, o["chroma_mean"])
        if o["tempogram"] is not None:
            assert np.abs(g - o["tempogram"]).max() <= 1e-5, (len(y), np.abs(g - o["tempogram"]).max())
        counts = np.array(f.tuning_counts[:])
        assert abs(f.n_pitches - o["n_kept"]) <= max(1, 1e-3 * o["n_kept"])
        assert np.abs(counts - o["counts"]).max() <= max(2, 1e-3 * o["n_kept"]), (len(y), counts, o["counts"])
        print(f"L={len(y)} energy rel {abs(f.energy - o['energy']) / max(o['energy'], 1e-30):.1e} "
              f"chroma {np.abs(cm - o['chroma_mean']).max():.1e} pitches {f.n_pitches}/{o['n_kept']}")


def test_discrete_values_where_the_oracle_is_decisive(device_run, oracle_runs, tracks):
    _, feats, tg = device_run
    decisive = 0
    for y, f, o, g in zip(tracks, feats, oracle_runs, tg):
        assert f.is_major == 0                                    # the reference always stores 'minor'
        if o["tempogram"] is None:
            assert f.tempo == 0.0 and f.period == 0
            continue
        tg_o = o["tempogram"]
        sc = otf.tempo_scores(tg_o)
        err = float(np.abs(g - tg_o).max())
        # d score / d tg = 1e6 / (1 + 1e6 tg): the score error the measured tempogram error can cause, per lag
        e = 1e6 * err / (1 + 1e6 * np.maximum(tg_o - err, 0.0))
        k1 = int(np.argmax(sc))
        others = np.array([k for k in range(otf.WIN) if k != k1 and np.isfinite(sc[k])])
        tempo_margin = float(np.min(sc[k1] - sc[others] - e[k1] - e[others]))
        c = np.sort(o["counts"])[::-1]
        count_err = int(np.abs(np.array(f.tuning_counts[:]) - o["counts"]).max())
        kc = np.sort(otf.key_correlations(o["chroma_mean"]))[::-1]
        print(f"L={len(y)} tempo margin over error {tempo_margin:.3g} tuning margin {c[0] - c[1]} (count error "
              f"{count_err}) key margin {kc[0] - kc[1]:.3g}")
        ok = 0
        if tempo_margin > 0:
            assert f.tempo == o["tempo"] and f.period == o["period"]
            ok += 1
        if c[0] - c[1] > 2 * count_err:
            assert f.tuning == o["tuning"]
            ok += 1
        if f.tuning == o["tuning"] and kc[0] - kc[1] > 1e-3:
            assert otf.KEYS[f.key] == o["key"]
            ok += 1
        decisive += ok == 3
    assert decisive >= 3      # of the 7 tracks with a non-zero onset envelope


def test_device_entry_equals_host_entry_and_runs_are_bit_identical(device_run, tracks):
    import torch
    from audiomuse_ai_b200 import _lib
    sess, feats, tg = device_run
    feats2, tg2 = sess.run(tracks, tempogram=True)
    b1 = b"".join(bytes(f) for f in feats)
    assert b"".join(bytes(f) for f in feats2) == b1
    np.testing.assert_array_equal(tg2, tg)
    lens = np.array([len(t) for t in tracks], np.int64)
    offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    dev = torch.from_numpy(np.concatenate(tracks)).cuda()
    feats3, tg3 = sess.run_dev(dev.data_ptr(), offs, tempogram=True)
    assert b"".join(bytes(f) for f in feats3) == b1
    np.testing.assert_array_equal(tg3, tg)
    sess.release_workspace()
    feats4, _ = sess.run(tracks)
    assert b"".join(bytes(f) for f in feats4) == b1


def test_track_features_api(built, tracks, oracle_runs):
    from audiomuse_ai_b200 import track_features as tfm
    waves = tracks[3:6] + [np.zeros(SR, np.float32), np.zeros(0, np.float32)]
    res = tfm.track_features(waves, max_samples=60 * SR)                 # forces several calls
    assert res[-1] is None and res[-2] is None
    for r, o in zip(res[:3], oracle_runs[3:6]):
        assert r["scale"] == "minor" and set(r) == {"tempo", "key", "scale", "energy"}
        assert abs(r["energy"] - float(o["energy"])) <= 1e-5 * float(o["energy"])


@pytest.mark.parametrize("spelling", ["torch", "tf"])
def test_analyze_track_drop_in(built, tmp_path, spelling):
    from audiomuse_ai_b200 import integration, musicnn as mm
    from oracle import mel as omel, musicnn as om
    from tests import musicnn_export as me

    export = {"torch": (me.export_embedding, me.export_prediction),
              "tf": (me.export_embedding_tf, me.export_prediction_tf)}[spelling]
    emb_m, pred_m = om.MusicnnEmbedding(seed=11), om.MusicnnPrediction(seed=12)
    paths = {"embedding": str(tmp_path / "musicnn_embedding.onnx"),
             "prediction": str(tmp_path / "musicnn_prediction.onnx")}
    (tmp_path / "musicnn_embedding.onnx").write_bytes(export[0](emb_m))
    (tmp_path / "musicnn_prediction.onnx").write_bytes(export[1](pred_m))
    audio = {"song.mp3": synthetic_music(20 * SR + 300, 7), "short.mp3": synthetic_music(2000, 8),
             "silent.mp3": np.zeros(SR * 5, np.float32), "broken.mp3": None}
    mod = types.SimpleNamespace(ort=types.SimpleNamespace(InferenceSession=lambda *a, **k: pytest.fail("onnxruntime")),
                                analyze_track=None,
                                robust_load_audio_with_fallback=lambda p, target_sr=16000: (audio[p], target_sr))
    integration.apply(analysis=mod, analyze_track=True)
    labels = [f"mood{i}" for i in range(50)]
    sessions = {"embedding": mm.MusicnnSession(paths["embedding"]), "prediction": mm.MusicnnSession(paths["prediction"])}
    y = audio["song.mp3"]
    want_f = otf.track_features(y)
    p = omel.musicnn_patches(y)
    ep = om.embed_patches(emb_m, p)
    want_e, want_m = om.track_result(ep, om.predict(pred_m, ep))
    for onnx_sessions in (None, sessions):
        for ret_audio in (False, True):
            out = mod.analyze_track("song.mp3", labels, paths, onnx_sessions=onnx_sessions, return_audio=ret_audio)
            assert len(out) == (4 if ret_audio else 2)
            res, emb = out[0], out[1]
            if ret_audio:
                assert out[3] == 16000 and np.array_equal(out[2], y)
            assert res["key"] == want_f["key"] and res["scale"] == "minor" and res["tempo"] == want_f["tempo"]
            assert abs(res["energy"] - want_f["energy"]) <= 1e-5 * want_f["energy"]
            assert emb.dtype == np.float32 and emb.shape == (200,)
            cos = float(np.dot(emb, want_e) / (np.linalg.norm(emb) * np.linalg.norm(want_e)))
            assert 1.0 - cos <= 1e-3
            assert list(res["moods"]) == labels
            assert np.abs(np.array(list(res["moods"].values())) - want_m).max() <= 1e-3
        for name in ("short.mp3", "silent.mp3", "broken.mp3"):
            assert mod.analyze_track(name, labels, paths, onnx_sessions=onnx_sessions) == (None, None)
            assert mod.analyze_track(name, labels, paths, onnx_sessions=onnx_sessions,
                                     return_audio=True) == (None, None, None, None)
