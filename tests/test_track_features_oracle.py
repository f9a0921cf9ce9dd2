"""The numpy restatement of analyze_track's tempo / energy / tuning / key (oracle/track_features.py) on signals whose
answers are known, and the analyze_track switch of integration.apply.  No GPU."""
import types

import numpy as np
import pytest

from oracle import track_features as tf

SR = 16000


def _clicks(period, seconds=30, seed=0):
    rng = np.random.default_rng(seed)
    y = (0.01 * rng.standard_normal(SR * seconds)).astype(np.float32)
    y[::period] += 1.0
    return y


def _tones(midis, detune, seconds=10.0):
    t = np.arange(int(SR * seconds)) / SR
    y = sum(np.sin(2 * np.pi * 440.0 * 2 ** ((m - 69 + detune) / 12) * t) for m in midis)
    return (0.2 * y).astype(np.float32)


@pytest.mark.parametrize("period,bpm,lag", [(7680, 125.0, 15), (10240, 93.75, 20), (5120, 93.75, 20)])
def test_click_train_tempo(period, bpm, lag):
    """Clicks every `period` samples = every period / 512 frames.  125 and 93.75 BPM are reported as played.  A
    187.5 BPM train is reported at half tempo: its autocorrelation at twice the period is nearly as strong, and the
    log-normal prior around 120 BPM (one octave = a penalty of 0.5) favours 93.75 over 187.5."""
    assert tf.tempo(_clicks(period)) == (bpm, lag)


def test_single_impulse_gives_zero_envelope_and_zero_tempo():
    y = np.zeros(5 * SR, np.float32)
    y[0] = 1.0
    assert not tf.onset_envelope(y).any()
    assert tf.tempo(y) == (0.0, 0)


def test_detuned_tones_tuning():
    """Peak interpolation biases the estimate by about a hundredth of a semitone."""
    S = tf.power_spectrum(_tones([60, 64, 67, 71], 0.234))
    tuning, counts, n_kept = tf.estimate_tuning(S)
    assert abs(tuning - 0.234) <= 0.02
    assert counts.sum() == n_kept > 0


def test_c_major_scale_is_stored_as_a_minor():
    """The reference's key block can only answer 'minor': its minor profile is the major one rolled by 3, so the
    relative minor of C major (A) wins the tie that the strict `major_max > minor_max` always resolves to minor."""
    y = np.concatenate([_tones([m], 0.0, 1.0) for m in (60, 62, 64, 65, 67, 69, 71)])
    feats = tf.track_features(y)
    assert feats["key"] == "A" and feats["scale"] == "minor"
    assert abs(tf.analyze(y)["tuning"]) <= 0.05


def test_minor_profile_is_major_rolled_by_three():
    np.testing.assert_array_equal(tf.MINOR_PROFILE, np.roll(tf.MAJOR_PROFILE, 3))


def test_key_scale_equals_the_loop_restatement():
    rng = np.random.default_rng(17)
    for i in range(1000):
        cm = rng.random(12).astype(np.float32)
        if i % 100 == 0:
            cm[:] = cm[0]                         # constant chroma: every correlation is NaN -> 'C' minor
        assert tf.key_scale(cm) == tf.key_scale_loop(cm), cm
    assert tf.key_scale(np.full(12, 0.5, np.float32)) == ("C", "minor")


def test_energy_is_mean_frame_rms():
    y = np.full(SR, 0.5, np.float32)
    e = tf.energy(y)
    frames = tf._frames(y)
    assert e == pytest.approx(np.mean(np.sqrt(np.mean(frames.astype(np.float64) ** 2, axis=1))), rel=1e-6)


def test_empty_and_silent_tracks_have_no_features():
    assert tf.track_features(np.zeros(0, np.float32)) is None
    assert tf.track_features(np.zeros(SR, np.float32)) is None


def _fake_analysis():
    m = types.SimpleNamespace(ort=types.SimpleNamespace(InferenceSession=lambda *a, **k: None))
    m.analyze_track = lambda *a, **k: "librosa"
    m.robust_load_audio_with_fallback = lambda path, target_sr=16000: (None, target_sr)
    return m


def test_apply_leaves_analyze_track_alone_by_default():
    from audiomuse_ai_b200 import integration
    m = _fake_analysis()
    orig = m.analyze_track
    integration.apply(analysis=m)
    assert m.analyze_track is orig


def test_apply_replaces_analyze_track_idempotently():
    from audiomuse_ai_b200 import integration
    m = _fake_analysis()
    integration.apply(analysis=m, analyze_track=True)
    first = m.analyze_track
    assert first is not None and getattr(first, "_b200", False)
    integration.apply(analysis=m, analyze_track=True)
    assert m.analyze_track is first
    # a failed load gives the reference's None tuples without touching the device
    assert first("x.mp3", [], {}) == (None, None)
    assert first("x.mp3", [], {}, return_audio=True) == (None, None, None, None)


def test_apply_analyze_track_needs_the_module():
    from audiomuse_ai_b200 import integration
    with pytest.raises(ValueError):
        integration.apply(analyze_track=True)
