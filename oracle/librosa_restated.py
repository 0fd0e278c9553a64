"""
numpy/scipy restatement of the librosa 0.10.2+/0.11 functions the reference's
hot path calls (TEST INFRASTRUCTURE — see oracle/__init__.py).

librosa itself is absent from this image (requirements.txt:22 pins only
``librosa>=0.10.1``), so every function here is restated from SURVEY.md
Appendix A; **parity with real librosa is unpinned**.  Call sites in the
reference (paths relative to /root/reference/nightcore_analyzer):

  io.py:54,76   tempo.py:44,45,58,63,158,159,168   pitch.py:58
  xcorr.py:92,93,206,207,210,211

Deliberate, documented deviations from real librosa:

* beat tracking (local score, DP, trim) runs in float64 on the float32 onset
  envelope (librosa's numba kernels may run in float32 for float32 input);
* ``resample`` is a Kaiser-windowed-sinc polyphase filter, not soxr_hq.
"""
from __future__ import annotations

import math
import numpy as np
import scipy.fft
import scipy.signal

# --------------------------------------------------------------------------- helpers


def tiny(x) -> float:
    """librosa.util.tiny: smallest positive normal number of x's float dtype."""
    dt = np.asarray(x).dtype
    if not np.issubdtype(dt, np.floating) and not np.issubdtype(dt, np.complexfloating):
        dt = np.dtype(np.float32)
    return float(np.finfo(dt).tiny)


def hann_periodic(n: int) -> np.ndarray:
    """scipy.signal.get_window('hann', n, fftbins=True), float64 (Appendix A.1)."""
    return scipy.signal.get_window("hann", n, fftbins=True)


def frames_to_time(frames, sr=22050, hop_length=512):
    """librosa.frames_to_time (Appendix A.5) — tempo.py:168."""
    return np.asanyarray(frames) * hop_length / float(sr)


def localmax(x: np.ndarray) -> np.ndarray:
    """librosa.util.localmax along the last axis: x[i] > x[i-1] and x[i] >= x[i+1];
    the first sample is never a maximum; the last is compared with itself (edge pad)."""
    x = np.asarray(x)
    out = np.zeros(x.shape, dtype=bool)
    if x.shape[-1] < 2:
        return out
    xp = np.concatenate([x, x[..., -1:]], axis=-1)
    out[..., 1:] = (x[..., 1:] > x[..., :-1]) & (x[..., 1:] >= xp[..., 2:])
    return out


# --------------------------------------------------------------------------- STFT


def stft(y: np.ndarray, n_fft: int = 2048, hop_length: int = 512, window="hann") -> np.ndarray:
    """librosa.stft(center=True, pad_mode='constant') (Appendix A.1).

    The float64 window times the float32 frames gives a float64 FFT; the
    result is stored as complex64 (float32 input)."""
    y = np.asarray(y)
    if window == "ones":
        w = np.ones(n_fft)
    else:
        w = hann_periodic(n_fft)
    pad = n_fft // 2
    yp = np.concatenate([np.zeros(pad, y.dtype), y, np.zeros(pad, y.dtype)])
    n_frames = 1 + len(y) // hop_length
    idx = np.arange(n_fft)[:, None] + hop_length * np.arange(n_frames)[None, :]
    out = np.empty((n_fft // 2 + 1, n_frames), dtype=np.complex64 if y.dtype == np.float32 else np.complex128)
    step = 4096
    for s in range(0, n_frames, step):
        e = min(n_frames, s + step)
        out[:, s:e] = scipy.fft.rfft(w[:, None] * yp[idx[:, s:e]], axis=0)
    return out


# --------------------------------------------------------------------------- mel


def _hz_to_mel(f):
    f = np.asanyarray(f, dtype=float)
    f_sp = 200.0 / 3
    mels = f / f_sp
    min_log_hz = 1000.0
    min_log_mel = min_log_hz / f_sp
    logstep = np.log(6.4) / 27.0
    return np.where(f >= min_log_hz, min_log_mel + np.log(np.maximum(f, 1e-300) / min_log_hz) / logstep, mels)


def _mel_to_hz(m):
    m = np.asanyarray(m, dtype=float)
    f_sp = 200.0 / 3
    freqs = f_sp * m
    min_log_hz = 1000.0
    min_log_mel = min_log_hz / f_sp
    logstep = np.log(6.4) / 27.0
    return np.where(m >= min_log_mel, min_log_hz * np.exp(logstep * (m - min_log_mel)), freqs)


def mel_filter(sr: int = 22050, n_fft: int = 2048, n_mels: int = 128, fmin: float = 0.0, fmax=None) -> np.ndarray:
    """librosa.filters.mel(htk=False, norm='slaney', dtype=float32) (Appendix A.2)."""
    if fmax is None:
        fmax = sr / 2.0
    fftfreqs = np.fft.rfftfreq(n=n_fft, d=1.0 / sr)
    mel_f = _mel_to_hz(np.linspace(_hz_to_mel(fmin), _hz_to_mel(fmax), n_mels + 2))
    fdiff = np.diff(mel_f)
    ramps = np.subtract.outer(mel_f, fftfreqs)
    weights = np.zeros((n_mels, 1 + n_fft // 2), dtype=np.float32)
    for i in range(n_mels):
        lower = -ramps[i] / fdiff[i]
        upper = ramps[i + 2] / fdiff[i + 1]
        weights[i] = np.maximum(0, np.minimum(lower, upper))
    enorm = 2.0 / (mel_f[2 : n_mels + 2] - mel_f[:n_mels])
    weights *= enorm[:, np.newaxis]          # float32 *= float64: computed in float64, stored as float32
    return weights


_MEL_CACHE: dict = {}


def _mel_cached(sr, n_fft, n_mels):
    key = (sr, n_fft, n_mels)
    if key not in _MEL_CACHE:
        _MEL_CACHE[key] = mel_filter(sr, n_fft, n_mels)
    return _MEL_CACHE[key]


# --------------------------------------------------------------------------- onset strength


def power_to_db(S: np.ndarray, amin: float = 1e-10, top_db: float = 80.0) -> np.ndarray:
    """librosa.power_to_db(ref=1.0) — the max is over the whole call (Appendix A.2)."""
    log_spec = 10.0 * np.log10(np.maximum(amin, S))
    if top_db is not None:
        log_spec = np.maximum(log_spec, log_spec.max() - top_db)
    return log_spec


def logmel_db(y: np.ndarray, sr: int = 22050, hop_length: int = 512, n_fft: int = 2048, n_mels: int = 128,
              top_db=80.0) -> np.ndarray:
    """melspectrogram(power=2) -> power_to_db; float32 [n_mels, n_frames]."""
    y = np.asarray(y, dtype=np.float32)
    D = stft(y, n_fft=n_fft, hop_length=hop_length)
    S = np.abs(D) ** 2.0
    mel = np.einsum("ft,mf->mt", S, _mel_cached(sr, n_fft, n_mels), optimize=True)
    return power_to_db(mel, top_db=top_db)


def onset_strength(y: np.ndarray, sr: int = 22050, hop_length: int = 512, n_fft: int = 2048,
                   n_mels: int = 128) -> np.ndarray:
    """librosa.onset.onset_strength(y=, sr=, hop_length=) (Appendix A.2) — tempo.py:44,158.

    lag=1, max_size=1, detrend=False, center=True, aggregate=np.mean."""
    S = logmel_db(y, sr, hop_length, n_fft, n_mels)
    return onset_from_logmel(S, n_fft, hop_length)


def onset_from_logmel(S: np.ndarray, n_fft: int, hop_length: int) -> np.ndarray:
    lag = 1
    onset_env = S[:, lag:] - S[:, :-lag]
    onset_env = np.maximum(0.0, onset_env)
    onset_env = np.mean(onset_env, axis=0)
    pad_width = lag + n_fft // (2 * hop_length)
    onset_env = np.pad(onset_env, (int(pad_width), 0), mode="constant")
    return onset_env[: S.shape[-1]]


# --------------------------------------------------------------------------- tempogram / tempo


def autocorrelate(y: np.ndarray, axis: int = 0) -> np.ndarray:
    """librosa.autocorrelate along `axis` (FFT route, real input)."""
    n = y.shape[axis]
    n_pad = scipy.fft.next_fast_len(2 * n - 1, real=True)
    spec = scipy.fft.rfft(y, n=n_pad, axis=axis)
    powspec = spec.real ** 2 + spec.imag ** 2
    ac = scipy.fft.irfft(powspec, n=n_pad, axis=axis)
    sl = [slice(None)] * ac.ndim
    sl[axis] = slice(n)
    return ac[tuple(sl)]


def _normalize_inf(S: np.ndarray, axis: int) -> np.ndarray:
    """librosa.util.normalize(norm=inf, fill=None)."""
    mag = np.abs(S).astype(float)
    length = np.max(mag, axis=axis, keepdims=True)
    length[length < tiny(S)] = 1.0
    return S / length


def tempogram_frames(onset_envelope: np.ndarray, win_length: int):
    """The padded envelope used by librosa.feature.tempogram(center=True, linear_ramp)."""
    onset_envelope = np.asarray(onset_envelope)
    p = int(win_length // 2)
    return np.pad(onset_envelope, (p, p), mode="linear_ramp", end_values=[0, 0])


def tempogram(onset_envelope: np.ndarray, win_length: int = 384, t0: int = 0, t1=None) -> np.ndarray:
    """librosa.feature.tempogram(onset_envelope=, win_length=, center=True, window='hann', norm=inf)
    (Appendix A.3) — tempo.py:58.  Returns [win_length, n] (optionally only frames t0:t1)."""
    n = len(onset_envelope)
    if t1 is None:
        t1 = n
    padded = tempogram_frames(onset_envelope, win_length)
    w = hann_periodic(win_length)
    idx = np.arange(win_length)[:, None] + np.arange(t0, t1)[None, :]
    frames = padded[idx] * w[:, None]          # float32 * float64 -> float64
    return _normalize_inf(autocorrelate(frames, axis=0), axis=0)


def tempo_frequencies(n_bins: int, hop_length: int, sr: float) -> np.ndarray:
    bpms = np.zeros(n_bins, dtype=np.float64)
    bpms[0] = np.inf
    bpms[1:] = 60.0 * sr / (hop_length * np.arange(1.0, n_bins))
    return bpms


def tempogram_mean(onset_envelope: np.ndarray, win_length: int, block: int = 2048) -> np.ndarray:
    """mean over frames of the tempogram, streamed over frame blocks (identical per-frame math)."""
    n = len(onset_envelope)
    acc = np.zeros(win_length, dtype=np.float64)
    for s in range(0, n, block):
        e = min(n, s + block)
        acc += tempogram(onset_envelope, win_length, s, e).sum(axis=1)
    return acc / n


def tempo_lag_from_mean(tg: np.ndarray, sr: float = 22050, hop_length: int = 512, start_bpm: float = 120.0,
                        std_bpm: float = 1.0, max_tempo: float = 320.0) -> int:
    """The prior-weighted argmax of librosa.feature.tempo over a time-averaged tempogram (Appendix A.3)."""
    win_length = len(tg)
    bpms = tempo_frequencies(win_length, hop_length, sr)
    with np.errstate(divide="ignore"):
        logprior = -0.5 * ((np.log2(bpms) - np.log2(start_bpm)) / std_bpm) ** 2
    max_idx = int(np.argmax(bpms < max_tempo))
    logprior[:max_idx] = -np.inf
    return int(np.argmax(np.log1p(1e6 * tg) + logprior))


def tempo_lag(onset_envelope: np.ndarray, sr: float = 22050, hop_length: int = 512, start_bpm: float = 120.0,
              std_bpm: float = 1.0, ac_size: float = 8.0, max_tempo: float = 320.0) -> int:
    """Best autocorrelation lag of librosa.feature.tempo (Appendix A.3) — tempo.py:63."""
    win_length = int(np.floor(ac_size * sr / hop_length))
    tg = tempogram_mean(onset_envelope, win_length)
    return tempo_lag_from_mean(tg, sr, hop_length, start_bpm, std_bpm, max_tempo)


def tempo(onset_envelope: np.ndarray, sr: float = 22050, hop_length: int = 512, start_bpm: float = 120.0) -> np.ndarray:
    """librosa.feature.tempo(onset_envelope=, sr=, hop_length=, start_bpm=) -> 1-element array."""
    win_length = int(np.floor(8.0 * sr / hop_length))
    lag = tempo_lag(onset_envelope, sr, hop_length, start_bpm)
    return np.array([tempo_frequencies(win_length, hop_length, sr)[lag]])


# --------------------------------------------------------------------------- beat tracking


def _beat_local_score(onset_norm: np.ndarray, fpb: float) -> np.ndarray:
    """librosa.beat.__beat_local_score, static-tempo branch (Appendix A.4).

    Restated literally, including the loop bound ``min(i + K//2, K)`` which
    excludes the tap that would touch onset[0] for small i."""
    N = len(onset_norm)
    window = np.exp(-0.5 * (np.arange(-fpb, fpb + 1) * 32.0 / fpb) ** 2)
    K = len(window)
    from . import native
    return native.local_score(np.ascontiguousarray(onset_norm, dtype=np.float64), window.astype(np.float64), K)


def beat_track_frames(onset_envelope: np.ndarray, bpm: float, sr: float = 22050, hop_length: int = 512,
                      tightness: float = 100.0, trim: bool = True, return_debug: bool = False):
    """librosa.beat.__beat_tracker with a given bpm (Appendix A.4): frames of the detected beats."""
    onset = np.asarray(onset_envelope, dtype=np.float64)
    fpb = float(np.round((float(sr) / hop_length) * 60.0 / bpm))
    norm = onset.std(ddof=1)
    onset_norm = onset / (norm + tiny(np.float64(0)))
    out, debug = beat_track_from_norm(onset_norm, fpb, tightness=tightness, trim=trim)
    return (out, debug) if return_debug else out


def beat_track_from_norm(onset_norm: np.ndarray, fpb: float, window=None, pen=None, tightness: float = 100.0,
                         trim: bool = True):
    """The chain of beat_track_frames after the normalisation: local score → DP → last beat → backtrack → trim.

    ``window`` (2·fpb + 1 taps) and ``pen`` (the transition penalty tightness·ln²(d / fpb) for d = round(fpb/2) .. 2·fpb)
    replace the values this module would compute, so that the chain can run on another machine's float64 exp and log.
    → (beat frames, debug dict: localscore, cumscore, backlink, tail, threshold, fpb, median of the local-maximum
    scores, margin = each frame's best-versus-second predecessor score gap, relative, pen = the penalty table used)."""
    from . import native
    fpb = float(fpb)
    if window is None:
        localscore = _beat_local_score(onset_norm, fpb)
    else:
        localscore = native.local_score(onset_norm, window, len(window))
    backlink, cumscore, margin = native.beat_dp_pen(localscore, fpb, tightness, pen)
    if pen is None:           # the table the C DP computed: tightness·(log(d) − log(fpb))² with the same C library log
        logf = math.log(fpb)
        pen = np.array([tightness * ((math.log(d) - logf) * (math.log(d) - logf))
                        for d in range(int(np.round(fpb / 2.0)), int(2.0 * fpb) + 1)])
    # last beat
    mask = localmax(cumscore)
    if mask.any():
        med = float(np.median(cumscore[mask]))
    else:
        med = float("nan")
    thr = 0.5 * med
    n = len(cumscore) - 1
    tail = n
    while n >= 0:
        if mask[n] and cumscore[n] >= thr:
            tail = n
            break
        n -= 1
    beats = np.zeros(len(onset_norm), dtype=bool)
    n = tail
    while n >= 0:
        beats[n] = True
        n = backlink[n]
    # trim
    w = np.hanning(5)
    smooth = np.convolve(localscore[beats], w)[len(w) // 2 : len(localscore) + len(w) // 2]
    threshold = 0.5 * ((smooth ** 2).mean() ** 0.5) if trim else 0.0
    n = 0
    while n < len(localscore) and localscore[n] <= threshold:
        beats[n] = False
        n += 1
    n = len(localscore) - 1
    while n >= 0 and localscore[n] <= threshold:
        beats[n] = False
        n -= 1
    out = np.flatnonzero(beats)
    return out, dict(localscore=localscore, cumscore=cumscore, backlink=backlink, tail=tail, threshold=threshold,
                     fpb=fpb, median=med, margin=margin, pen=pen)


def beat_track(onset_envelope: np.ndarray, sr: float = 22050, hop_length: int = 512, start_bpm: float = 120.0):
    """librosa.beat.beat_track(onset_envelope=, sr=, hop_length=, start_bpm=) -> (tempo, frames)
    (Appendix A.4) — tempo.py:45,159."""
    onset_envelope = np.asarray(onset_envelope)
    if not onset_envelope.any():
        return 0.0, np.array([], dtype=int)
    bpm = tempo(onset_envelope, sr=sr, hop_length=hop_length, start_bpm=start_bpm)
    beats = beat_track_frames(onset_envelope, float(bpm[0]), sr=sr, hop_length=hop_length)
    return bpm, beats


# --------------------------------------------------------------------------- rms / trim


def rms(y: np.ndarray, frame_length: int = 2048, hop_length: int = 512) -> np.ndarray:
    """librosa.feature.rms(y=, frame_length=, hop_length=, center=True, pad_mode='constant')[0]
    (Appendix A.6/A.7) — xcorr.py:210."""
    y = np.asarray(y)
    pad = frame_length // 2
    yp = np.concatenate([np.zeros(pad, y.dtype), y, np.zeros(pad, y.dtype)])
    n_frames = 1 + len(y) // hop_length
    out = np.empty(n_frames, dtype=y.dtype)
    step = 8192
    for s in range(0, n_frames, step):
        e = min(n_frames, s + step)
        idx = np.arange(frame_length)[:, None] + hop_length * np.arange(s, e)[None, :]
        x = yp[idx]
        out[s:e] = np.sqrt(np.mean(np.abs(x) ** 2, axis=0))
    return out


def trim(y: np.ndarray, top_db: float = 60.0, frame_length: int = 2048, hop_length: int = 512):
    """librosa.effects.trim (Appendix A.6) — io.py:76.  Returns (y[start:end], (start, end))."""
    y = np.asarray(y)
    mse = rms(y, frame_length, hop_length)
    amin = 1e-5
    mag = np.abs(mse)
    ref = np.max(mag)
    db = 10.0 * np.log10(np.maximum(amin ** 2, mag ** 2)) - 10.0 * np.log10(np.maximum(amin ** 2, ref ** 2))
    non_silent = np.flatnonzero(db > -top_db)
    if non_silent.size > 0:
        start = int(non_silent[0] * hop_length)
        end = min(len(y), int((non_silent[-1] + 1) * hop_length))
    else:
        start, end = 0, 0
    return y[start:end], np.asarray([start, end])


# --------------------------------------------------------------------------- resample (own FIR, NOT soxr)

HALFBAND_TAPS = 127
HALFBAND_BETA = 10.0


def halfband_fir() -> np.ndarray:
    """Linear-phase low-pass used for every 2:1 decimation (documented deviation: librosa uses
    soxr_hq, which cannot be reproduced here).  Kaiser-windowed sinc, 127 taps, beta 10,
    cut-off at a quarter of the input rate; DC gain exactly 1."""
    n = np.arange(HALFBAND_TAPS) - (HALFBAND_TAPS - 1) // 2
    h = 0.5 * np.sinc(0.5 * n) * np.kaiser(HALFBAND_TAPS, HALFBAND_BETA)
    return h / h.sum()


def decimate2(y: np.ndarray, scale: bool = True) -> np.ndarray:
    """resample(y, orig_sr=2, target_sr=1, scale=True): out[i] = sqrt(2)·sum_k h[k]·y[2i+k-63]; len ceil(n/2)."""
    y = np.asarray(y)
    h = halfband_fir()
    c = (HALFBAND_TAPS - 1) // 2
    n_out = (len(y) + 1) // 2
    yp = np.concatenate([np.zeros(c), y.astype(np.float64), np.zeros(c + 1)])
    full = np.convolve(yp, h[::-1], mode="valid")      # full[j] = sum_k h[k] yp[j+k] = sum_k h[k] y[j+k-c]
    out = full[0 : 2 * n_out : 2]
    if scale:
        out = out * np.sqrt(2.0)
    return out.astype(y.dtype)


def resample(y: np.ndarray, orig_sr: float, target_sr: float, scale: bool = False) -> np.ndarray:
    """Stand-in for librosa.resample (xcorr.py:206-207).  2:1 uses `decimate2`; other ratios use
    scipy.signal.resample_poly.  NOT soxr-compatible."""
    y = np.asarray(y)
    if orig_sr == target_sr:
        return y
    if orig_sr == 2 * target_sr:
        out = decimate2(y, scale=False)
    else:
        from fractions import Fraction
        fr = Fraction(int(target_sr), int(orig_sr))
        out = scipy.signal.resample_poly(y.astype(np.float64), fr.numerator, fr.denominator).astype(y.dtype)
        n_out = int(math.ceil(len(y) * target_sr / orig_sr))
        out = out[:n_out]
    if scale:
        out = out / np.sqrt(target_sr / orig_sr)
    return out.astype(y.dtype)


# --------------------------------------------------------------------------- tuning / CQT / chroma

C1_HZ = 32.70319566257483          # librosa.note_to_hz('C1') = 440·2^((24-69)/12)... exact below


def note_c1_hz() -> float:
    return 440.0 * (2.0 ** ((12 * (1 + 1) + 0 - 69) / 12.0))


def piptrack_peaks(y: np.ndarray, sr: float = 22050, n_fft: int = 2048, hop_length: int = 512,
                   fmin: float = 150.0, fmax: float = 4000.0, threshold: float = 0.1):
    """librosa.piptrack restricted to what estimate_tuning needs: (pitches, mags) of all peaks."""
    S = np.abs(stft(np.asarray(y, dtype=np.float32), n_fft=n_fft, hop_length=hop_length))
    fmax = min(fmax, sr / 2.0)
    fft_freqs = np.fft.rfftfreq(n=n_fft, d=1.0 / sr)
    avg = np.gradient(S, axis=0)
    a = S[2:] + S[:-2] - 2 * S[1:-1]
    b = (S[2:] - S[:-2]) / 2
    shift = np.zeros_like(S)
    with np.errstate(divide="ignore", invalid="ignore"):
        sh = np.where(np.abs(b) >= np.abs(a), 0.0, -b / a)
    shift[1:-1] = sh
    dskew = 0.5 * avg * shift
    freq_mask = ((fmin <= fft_freqs) & (fft_freqs < fmax))[:, None]
    ref_value = threshold * np.max(S, axis=0, keepdims=True)
    Sm = S * (S > ref_value)
    lm = localmax(Sm.T).T
    idx = np.nonzero(freq_mask & lm)
    pitches = ((idx[0] + shift[idx]) * float(sr) / n_fft)
    mags = S[idx] + dskew[idx]
    return pitches, mags


def pitch_tuning(frequencies: np.ndarray, resolution: float = 0.01, bins_per_octave: int = 12) -> float:
    frequencies = np.atleast_1d(frequencies)
    frequencies = frequencies[frequencies > 0]
    if not np.any(frequencies):
        return 0.0
    residual = np.mod(bins_per_octave * np.log2(frequencies / (440.0 / 16)), 1.0)
    residual[residual >= 0.5] -= 1.0
    bins = np.linspace(-0.5, 0.5, int(np.ceil(1.0 / resolution)) + 1)
    counts, tuning = np.histogram(residual, bins)
    return float(tuning[np.argmax(counts)])


def estimate_tuning(y: np.ndarray, sr: float = 22050, bins_per_octave: int = 12, return_index: bool = False):
    """librosa.estimate_tuning(y=, sr=, bins_per_octave=) (§3.4)."""
    pitch, mag = piptrack_peaks(y, sr)
    pitch_mask = pitch > 0
    if pitch_mask.any():
        threshold = np.median(mag[pitch_mask])
    else:
        threshold = 0.0
    t = pitch_tuning(pitch[(mag >= threshold) & pitch_mask], bins_per_octave=bins_per_octave)
    if return_index:  # histogram bin 0..99 (left edges -0.50 ... +0.49)
        return t, int(round((t + 0.5) * 100))
    return t


def cqt_octave_basis(sr: float, fmin: float, bins_per_octave: int = 36, n_bins: int = 252, sparsity: float = 0.01):
    """FFT basis of the TOP octave at the full rate (Appendix A.8): complex [36, 513], plus n_fft and
    the full-rate filter lengths of all n_bins.  Every lower octave uses the same matrix times sqrt(2^oct)."""
    freqs = fmin * 2.0 ** (np.arange(n_bins) / bins_per_octave)
    r = 2.0 ** (1.0 / bins_per_octave)
    alpha = (r ** 2 - 1) / (r ** 2 + 1)
    Q = 1.0 / alpha
    lengths_all = Q * sr / freqs
    freqs_top = freqs[-bins_per_octave:]
    lengths = Q * sr / freqs_top
    filters = []
    for ilen, freq in zip(lengths, freqs_top):
        t = np.arange(-ilen // 2, ilen // 2, dtype=float)
        sig = np.exp(1j * t * 2 * np.pi * freq / sr)
        sig = sig * hann_periodic(len(sig))
        sig = sig / np.sum(np.abs(sig))
        filters.append(sig)
    max_len = int(2.0 ** (np.ceil(np.log2(max(lengths)))))
    basis = np.zeros((len(filters), max_len), dtype=np.complex128)
    for i, f in enumerate(filters):
        lpad = (max_len - len(f)) // 2
        basis[i, lpad : lpad + len(f)] = f
    n_fft = max_len
    basis *= lengths[:, None] / float(n_fft)
    fft_basis = scipy.fft.fft(basis, n=n_fft, axis=1)[:, : n_fft // 2 + 1]
    # util.sparsify_rows(quantile=0.01)
    out = np.zeros_like(fft_basis)
    mags = np.abs(fft_basis)
    norms = np.sum(mags, axis=1, keepdims=True)
    mag_sort = np.sort(mags, axis=1)
    cumulative_mag = np.cumsum(mag_sort / norms, axis=1)
    threshold_idx = np.argmin(cumulative_mag < sparsity, axis=1)
    for i, j in enumerate(threshold_idx):
        keep = mags[i] >= mag_sort[i, j]
        out[i, keep] = fft_basis[i, keep]
    return out.astype(np.complex64), n_fft, lengths_all


def cqt_mag(y: np.ndarray, sr: float = 22050, hop_length: int = 512, bins_per_octave: int = 36,
            n_octaves: int = 7, tuning=None) -> np.ndarray:
    """|librosa.cqt| as chroma_cqt calls it (§3.4 / Appendix A.8): float32 [252, n_frames]."""
    y = np.asarray(y, dtype=np.float32)
    n_bins = n_octaves * bins_per_octave
    if tuning is None:
        tuning = estimate_tuning(y, sr, bins_per_octave=bins_per_octave)
    fmin = note_c1_hz() * 2.0 ** (tuning / bins_per_octave)
    fft_basis, n_fft, lengths = cqt_octave_basis(sr, fmin, bins_per_octave, n_bins)
    resp = []
    my_y, my_hop = y, hop_length
    for i in range(n_octaves):
        D = stft(my_y, n_fft=n_fft, hop_length=my_hop, window="ones")
        resp.append((fft_basis * np.float32(np.sqrt(2.0 ** i))).astype(np.complex64).dot(D))
        if my_hop % 2 == 0:
            my_hop //= 2
            my_y = decimate2(my_y, scale=True)
    max_col = min(c.shape[-1] for c in resp)
    V = np.empty((n_bins, max_col), dtype=np.complex64)
    end = n_bins
    for c in resp:
        n_oct = c.shape[0]
        V[end - n_oct : end] = c[:, :max_col]
        end -= n_oct
    V /= np.sqrt(lengths)[:, None].astype(np.float32)
    return np.abs(V)


def cq_to_chroma(n_input: int = 252, bins_per_octave: int = 36, n_chroma: int = 12) -> np.ndarray:
    """librosa.filters.cq_to_chroma(fmin=C1) (Appendix A.8): float32 [12, 252]."""
    n_merge = bins_per_octave // n_chroma
    cq = np.repeat(np.eye(n_chroma), n_merge, axis=1)
    cq = np.roll(cq, -(n_merge // 2), axis=1)
    n_octaves = int(np.ceil(n_input / bins_per_octave))
    cq = np.tile(cq, n_octaves)[:, :n_input]
    # fmin = C1 -> midi 24 -> roll = round(24 % 12 · n_chroma/12) = 0
    return cq.astype(np.float32)


def chroma_cqt(y: np.ndarray, sr: float = 22050, hop_length: int = 512, bins_per_octave: int = 36,
               n_chroma: int = 12, n_octaves: int = 7, tuning=None) -> np.ndarray:
    """librosa.feature.chroma_cqt(y=, sr=, bins_per_octave=, hop_length=) — pitch.py:58.  [12, n_frames]."""
    C = cqt_mag(y, sr, hop_length, bins_per_octave, n_octaves, tuning)
    chroma = cq_to_chroma(C.shape[0], bins_per_octave, n_chroma).dot(C)
    chroma[chroma < 0.0] = 0.0
    return _normalize_inf(chroma, axis=0)


# --------------------------------------------------------------------------- spectral statistics (spectral.py:38-103)


def fft_frequencies(sr: float = 22050, n_fft: int = 2048) -> np.ndarray:
    """librosa.fft_frequencies = np.fft.rfftfreq(n_fft, 1/sr)."""
    return np.fft.rfftfreq(n=n_fft, d=1.0 / sr)


def _normalize_l1(S: np.ndarray, axis: int) -> np.ndarray:
    """librosa.util.normalize(norm=1, fill=None): divide by the sum of magnitudes; columns below tiny stay unscaled."""
    mag = np.abs(S).astype(float)
    length = np.sum(mag, axis=axis, keepdims=True)
    length[length < tiny(S)] = 1.0
    return S / length


def spectral_centroid(y: np.ndarray, sr: float = 22050, n_fft: int = 2048, hop_length: int = 512) -> np.ndarray:
    """librosa.feature.spectral_centroid(y=, sr=) → [1, n_frames]: sum(freq · normalize(|STFT|, norm=1))."""
    S = np.abs(stft(np.asarray(y, dtype=np.float32), n_fft=n_fft, hop_length=hop_length))
    freq = fft_frequencies(sr, n_fft)
    return np.sum(freq[:, None] * _normalize_l1(S, axis=0), axis=0, keepdims=True)


def spectral_rolloff(y: np.ndarray, sr: float = 22050, n_fft: int = 2048, hop_length: int = 512,
                     roll_percent: float = 0.85) -> np.ndarray:
    """librosa.feature.spectral_rolloff → [1, n_frames]: lowest bin frequency whose cumulative magnitude reaches
    roll_percent of the frame total."""
    S = np.abs(stft(np.asarray(y, dtype=np.float32), n_fft=n_fft, hop_length=hop_length))
    freq = fft_frequencies(sr, n_fft)[:, None]
    total_energy = np.cumsum(S, axis=0)
    threshold = roll_percent * total_energy[-1]
    ind = np.where(total_energy < threshold[None, :], np.nan, 1)
    return np.nanmin(ind * freq, axis=0, keepdims=True)


def amplitude_to_db(S: np.ndarray, ref=1.0, amin: float = 1e-5, top_db: float = 80.0) -> np.ndarray:
    """librosa.amplitude_to_db(S, ref=np.max) = power_to_db(S², ref=ref², amin=amin², top_db)."""
    magnitude = np.abs(S)
    ref_value = ref(magnitude) if callable(ref) else np.abs(ref)
    power = np.square(magnitude)
    log_spec = 10.0 * np.log10(np.maximum(amin ** 2, power))
    log_spec = log_spec - 10.0 * np.log10(np.maximum(amin ** 2, ref_value ** 2))
    if top_db is not None:
        log_spec = np.maximum(log_spec, log_spec.max() - top_db)
    return log_spec
