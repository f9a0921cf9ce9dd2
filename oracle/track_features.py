"""Oracle: analyze_track's tempo, energy, tuning, chroma and key.  TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

Restates ``tasks/analysis.py:344-365``:

    tempo, _ = librosa.beat.beat_track(y=audio, sr=sr)
    average_energy = np.mean(librosa.feature.rms(y=audio))
    chroma = librosa.feature.chroma_stft(y=audio, sr=sr)     # then the key / scale block

for mono float32 audio at sr = 16000.  librosa==0.11.0 (requirements/common.txt:27) is a third-party dependency that
is not importable here; its published algorithm is restated below with its dtype discipline.

PARITY UNPINNED: librosa cannot be run here, so nothing in this file has been compared with librosa's own output.
What is restated, and where this reading of librosa 0.11 makes a choice:

  * framing: n_fft 2048, hop 512, center=True with ZERO padding (pad_mode='constant', librosa's default since 0.10),
    T = 1 + L // 512, periodic Hann in float64, rFFT in float64 stored as complex64, power |X|^2 in float32;
  * energy: rms over the same zero-padded frames without a window (a float32 mean over the frame axis), then the
    float32 mean over frames;
  * tempo (beat_track's tempo only; its beat positions are discarded by the caller, so the dynamic-programming
    tracker is not restated): onset_strength(aggregate=np.median) on power_to_db(128 Slaney mels, fmax sr/2,
    top_db=80 against the whole track's max); env[i] = 0 for i < 3 and env[i] = median_b max(0, D[b,i-2]-D[b,i-3]);
    an all-zero envelope gives tempo 0.0 (beat_track's early return); tempogram with win_length
    floor(8 * sr / 512) = 250, linear_ramp padding of 125 frames to zero on each side, periodic Hann, a float64
    autocorrelation per frame normalised by its largest |value|, mean over frames; then
    argmax_k log1p(1e6 tg[k]) - 0.5 (log2 bpm[k] - log2 120)^2 over bpm[k] = 60 sr / (512 k) < 320 (k >= 6);
  * tuning: estimate_tuning on the POWER spectrogram (chroma_stft passes S=power): piptrack with threshold 0.1 of
    each frame's max over all bins, fmin 150, fmax 4000, local maxima of the masked spectrum, parabolic shift from
    the unmasked one (0 where |b| >= |a|), mag = S + 0.5 b shift; the float32 median of the candidate mags is the
    threshold; residuals 12 log2(p / 27.5) mod 1 in float32, histogram over linspace(-0.5, 0.5, 101) with numpy's
    bin rules, tuning = the left edge of the first maximal bin;
  * chroma: librosa.filters.chroma(sr, 2048, tuning) (ctroct 5, octwidth 2, L2 column norm, base_c) built in
    float64 and stored as float32, fb @ S, each frame divided by its max (frames whose max is below float32 tiny
    are divided by 1), float32 mean over frames;
  * key / scale: np.corrcoef against the binary major and minor profiles rotated by i.  The minor profile is the
    major one rolled by 3, so both sets hold the same twelve numbers and the strict `major_max > minor_max` is never
    true: the reference always stores scale 'minor', key = the first argmax of the minor correlations ('C' when a
    constant chroma makes every correlation NaN).  That behaviour is reproduced, not corrected.
"""
from __future__ import annotations

import numpy as np

from . import mel as omel

SR = 16000
N_FFT = 2048
HOP = 512
N_MELS = 128
TOP_DB = 80.0
AC_SIZE = 8.0
WIN = int(np.floor(AC_SIZE * SR / HOP))      # 250 tempogram lags
START_BPM = 120.0
MAX_TEMPO = 320.0
KEYS = ["C", "C#", "D", "D#", "E", "F", "F#", "G", "G#", "A", "A#", "B"]
MAJOR_PROFILE = np.array([1, 0, 1, 0, 1, 1, 0, 1, 0, 1, 0, 1])
MINOR_PROFILE = np.array([1, 0, 1, 1, 0, 1, 0, 1, 1, 0, 1, 0])
PIP_FMIN, PIP_FMAX, PIP_THRESHOLD = 150.0, 4000.0, 0.1


def n_frames(n_samples: int) -> int:
    return 1 + int(n_samples) // HOP


def _frames(y):
    """Zero-padded (center=True, pad_mode='constant') frames, f32[T, 2048]."""
    y = np.asarray(y, dtype=np.float32).reshape(-1)
    ypad = np.pad(y, N_FFT // 2, mode="constant")
    T = n_frames(len(y))
    idx = np.arange(N_FFT)[None, :] + HOP * np.arange(T)[:, None]
    return ypad[idx]


def power_spectrum(y):
    """|STFT|^2, f32[1025, T]."""
    spec = np.fft.rfft(omel.hann_periodic(N_FFT)[None, :] * _frames(y), axis=1).astype(np.complex64)
    return (np.abs(spec) ** 2).T.astype(np.float32, copy=False)


def energy(y) -> np.float32:
    """np.mean(librosa.feature.rms(y=y)) in float32."""
    x = _frames(y).T                                   # [2048, T]: the mean runs over the frame axis
    rms = np.sqrt(np.mean(x * x, axis=0))
    return np.float32(np.mean(rms[None, :]))


def onset_db(S):
    """power_to_db(128 Slaney mels of S, top_db=80), f32[128, T]."""
    mel = omel.mel_filterbank(SR, N_FFT, N_MELS, 0.0, SR / 2.0) @ S
    D = omel.power_to_db(mel)
    return np.maximum(D, D.max() - np.float32(TOP_DB)).astype(np.float32, copy=False)


def onset_envelope(y=None, S=None):
    """onset_strength(y, sr, hop_length=512, aggregate=np.median), f32[T]."""
    if S is None:
        S = power_spectrum(y)
    D = onset_db(S)
    T = D.shape[1]
    env = np.zeros(T, dtype=np.float32)
    if T > 3:
        diff = np.maximum(np.float32(0.0), D[:, 1:T - 2] - D[:, 0:T - 3])   # column i-3 -> env[i]
        env[3:] = np.median(diff, axis=0)
    return env


def tempogram_mean(env):
    """np.mean(librosa.feature.tempogram(onset_envelope=env, win_length=250), axis=1), f64[250]."""
    env = np.asarray(env, dtype=np.float32)
    T = len(env)
    padded = np.pad(env, WIN // 2, mode="linear_ramp", end_values=(0, 0))
    idx = np.arange(WIN)[None, :] + np.arange(T)[:, None]
    x = padded[idx] * omel.hann_periodic(WIN)[None, :]               # float64 [T, 250]
    n_pad = 2 * WIN                                                   # >= 2W - 1: a linear, not circular, correlation
    r = np.fft.irfft(np.abs(np.fft.rfft(x, n=n_pad, axis=1)) ** 2, n=n_pad, axis=1)[:, :WIN]
    m = np.abs(r).max(axis=1, keepdims=True)
    m[m < np.finfo(np.float64).tiny] = 1.0
    return np.mean(r / m, axis=0)


def tempo_bpms():
    bpm = np.empty(WIN, dtype=np.float64)
    bpm[0] = np.inf
    bpm[1:] = 60.0 * SR / (HOP * np.arange(1.0, WIN))
    return bpm


def tempo_scores(tg):
    """Per-lag score with the log-normal prior around 120 BPM; -inf for bpm >= 320."""
    bpm = tempo_bpms()
    with np.errstate(divide="ignore", invalid="ignore"):
        logprior = -0.5 * ((np.log2(bpm) - np.log2(START_BPM)) / 1.0) ** 2
    logprior[: int(np.argmax(bpm < MAX_TEMPO))] = -np.inf
    return np.log1p(1e6 * tg) + logprior


def tempo(y=None, env=None):
    """beat_track's tempo: (tempo, period k); (0.0, 0) when the onset envelope is all zero."""
    if env is None:
        env = onset_envelope(y)
    if not env.any():
        return 0.0, 0
    k = int(np.argmax(tempo_scores(tempogram_mean(env))))
    return float(tempo_bpms()[k]), k


def piptrack(S):
    """librosa.piptrack(S=S, sr=16000, n_fft=2048, fmin=150, fmax=4000, threshold=0.1) restricted to its candidates:
    (pitch f32[n], mag f32[n]) in frame-major order."""
    S = np.asarray(S, dtype=np.float32)
    n_bins = S.shape[0]
    freqs = np.arange(n_bins) * (SR / N_FFT)
    avg = np.zeros_like(S)
    avg[1:-1] = (S[2:] - S[:-2]) / 2                                  # np.gradient, interior
    a = S[2:] + S[:-2] - 2 * S[1:-1]
    b = (S[2:] - S[:-2]) / 2
    shift = np.zeros_like(S)
    with np.errstate(divide="ignore", invalid="ignore"):
        sh = -b / a
    sh[np.abs(b) >= np.abs(a)] = 0
    shift[1:-1] = sh
    dskew = 0.5 * avg * shift
    ref = np.float32(PIP_THRESHOLD) * S.max(axis=0, keepdims=True)
    Sm = S * (S > ref)
    lm = np.zeros_like(S, dtype=bool)                                 # librosa.util.localmax along bins
    lm[1:-1] = (Sm[1:-1] > Sm[:-2]) & (Sm[1:-1] >= Sm[2:])
    freq_mask = ((PIP_FMIN <= freqs) & (freqs < PIP_FMAX))[:, None]
    f, t = np.nonzero(freq_mask & lm)
    order = np.lexsort((f, t))
    f, t = f[order], t[order]
    pitch = ((f + shift[f, t]) * np.float32(SR / N_FFT)).astype(np.float32)
    mag = (S[f, t] + dskew[f, t]).astype(np.float32)
    return pitch, mag


def tuning_residuals(pitch):
    res = np.mod(np.float32(12) * np.log2(pitch.astype(np.float32) / np.float32(440.0 / 16)), np.float32(1.0))
    res[res >= 0.5] -= np.float32(1.0)
    return res.astype(np.float32)


def estimate_tuning(S):
    """librosa.estimate_tuning(S=S, sr=16000, n_fft=2048): (tuning, histogram counts int64[100], kept pitch count)."""
    pitch, mag = piptrack(S)
    threshold = np.median(mag) if len(mag) else np.float32(0.0)
    kept = pitch[(mag >= threshold) & (pitch > 0)]
    if len(kept) == 0:
        return 0.0, np.zeros(100, dtype=np.int64), 0
    counts, edges = np.histogram(tuning_residuals(kept), np.linspace(-0.5, 0.5, 101))
    return float(edges[int(np.argmax(counts))]), counts.astype(np.int64), len(kept)


def chroma_filterbank(tuning=0.0, n_chroma=12):
    """librosa.filters.chroma(sr=16000, n_fft=2048, tuning=tuning), f32[12, 1025]."""
    frequencies = np.linspace(0, SR, N_FFT, endpoint=False)[1:]
    a440 = 440.0 * 2.0 ** (tuning / n_chroma)
    frqbins = n_chroma * np.log2(frequencies / (a440 / 16))
    frqbins = np.concatenate(([frqbins[0] - 1.5 * n_chroma], frqbins))
    binwidthbins = np.concatenate((np.maximum(frqbins[1:] - frqbins[:-1], 1.0), [1]))
    D = np.subtract.outer(frqbins, np.arange(0, n_chroma, dtype="d")).T
    n_chroma2 = np.round(float(n_chroma) / 2)
    D = np.remainder(D + n_chroma2 + 10 * n_chroma, n_chroma) - n_chroma2
    wts = np.exp(-0.5 * (2 * D / np.tile(binwidthbins, (n_chroma, 1))) ** 2)
    length = np.sqrt(np.sum(wts ** 2, axis=0, keepdims=True))
    length[length < np.finfo(np.float64).tiny] = 1.0
    wts = wts / length
    wts *= np.tile(np.exp(-0.5 * (((frqbins / n_chroma - 5.0) / 2) ** 2)), (n_chroma, 1))
    wts = np.roll(wts, -3 * (n_chroma // 12), axis=0)
    return np.ascontiguousarray(wts[:, : 1 + N_FFT // 2], dtype=np.float32)


def chroma_mean(S, tuning):
    """np.mean(librosa.feature.chroma_stft(S=S, tuning=tuning), axis=1), f32[12]."""
    chroma = chroma_filterbank(tuning) @ np.asarray(S, dtype=np.float32)
    mx = np.abs(chroma).max(axis=0, keepdims=True)
    mx[mx < np.finfo(np.float32).tiny] = 1.0
    return np.mean(chroma / mx, axis=1).astype(np.float32)


def key_correlations(cm):
    """np.corrcoef(chroma_mean, roll(major, i))[0, 1] for i in 0..11, f64[12]."""
    x = np.asarray(cm, dtype=np.float64)
    P = np.stack([np.roll(MAJOR_PROFILE, i) for i in range(12)]).astype(np.float64)
    xc = x - x.mean()
    pc = P - P.mean(axis=1, keepdims=True)
    with np.errstate(divide="ignore", invalid="ignore"):
        c = (pc @ xc) / np.sqrt((pc * pc).sum(axis=1) * (xc @ xc))
    return np.clip(c, -1.0, 1.0)


def key_scale(cm):
    """The key / scale block, vectorised: the minor correlations are the major ones rotated by 3
    (MINOR_PROFILE == np.roll(MAJOR_PROFILE, 3)), so both maxima are the same number."""
    major = key_correlations(cm)
    minor = np.roll(major, -3)                    # minor[i] = major[(i + 3) % 12]
    mi, ni = int(np.argmax(major)), int(np.argmax(minor))
    if major[mi] > minor[ni]:
        return KEYS[mi], "major"
    return KEYS[ni], "minor"


def key_scale_loop(cm):
    """The key / scale block written out rotation by rotation, one np.corrcoef each."""
    cm = np.asarray(cm)
    major_corrs, minor_corrs = [], []
    for i in range(12):
        major_corrs.append(np.corrcoef(cm, np.roll(MAJOR_PROFILE, i))[0, 1])
    for i in range(12):
        minor_corrs.append(np.corrcoef(cm, np.roll(MINOR_PROFILE, i))[0, 1])
    best_major = int(np.argmax(major_corrs))
    best_minor = int(np.argmax(minor_corrs))
    if major_corrs[best_major] > minor_corrs[best_minor]:
        return KEYS[best_major], "major"
    return KEYS[best_minor], "minor"


def analyze(y):
    """Every intermediate the device path reports: dict with tempo, period, energy, tuning, counts, n_kept,
    chroma_mean, key, scale, tempogram (f64[250] or None), env."""
    y = np.asarray(y, dtype=np.float32).reshape(-1)
    S = power_spectrum(y)
    env = onset_envelope(S=S)
    tg = tempogram_mean(env) if env.any() else None
    k = 0 if tg is None else int(np.argmax(tempo_scores(tg)))
    t = 0.0 if tg is None else float(tempo_bpms()[k])
    tuning, counts, n_kept = estimate_tuning(S)
    cm = chroma_mean(S, tuning)
    key, scale = key_scale(cm)
    return {"tempo": t, "period": k, "energy": energy(y), "tuning": tuning, "counts": counts, "n_kept": n_kept,
            "chroma_mean": cm, "key": key, "scale": scale, "tempogram": tg, "env": env}


def track_features(y):
    """{"tempo", "key", "scale", "energy"} as analyze_track stores them, or None for an empty or all-zero track."""
    y = np.asarray(y, dtype=np.float32).reshape(-1)
    if y.size == 0 or not np.any(y):
        return None
    a = analyze(y)
    return {"tempo": a["tempo"], "key": a["key"], "scale": a["scale"], "energy": float(a["energy"])}
