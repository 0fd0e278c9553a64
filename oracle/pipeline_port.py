"""
CPU port of the reference's array-level pipeline (TEST / BASELINE INFRASTRUCTURE — see oracle/__init__.py).

Same control flow and parameters as /root/reference/nightcore_analyzer/{io,tempo,pitch,consensus,
pipeline}.py, executed on oracle/librosa_restated.py.  The reference itself cannot travel to the
GPU box (and needs librosa), so this port is what ``bench.py --impl reference`` / ``cpu_baseline``
time and what the full-pipeline parity tests compare against.  tests/test_reference_golden.py checks,
in the build container, that the port agrees with the reference's own modules run unmodified over
the librosa shim (oracle/reference_shim.py).

Returns plain numbers (lists, tuples); the AnalysisResult dataclass and its strings are product
code checked separately against the reference's golden vectors.
"""
from __future__ import annotations

from typing import Callable, List, Optional

import numpy as np

from . import librosa_restated as lr
from . import native

SAMPLE_RATE = 22050
MIN_BEATS = 4            # tempo.py:22
AGREEMENT_TOLERANCE = 0.08
HOP_LENGTH = 512
IBI_HOP_LENGTH = 64      # tempo.py:116
CHUNK_SEC = 20.0         # pitch.py:44
MIN_CHUNKS = 3
N_BOOTSTRAP = 2000       # consensus.py:52
MIN_VALID = 3


# ---------------------------------------------------------------------------------- io.py
def rms_db(audio: np.ndarray) -> float:
    """io.py:38-40."""
    rms = float(np.sqrt(np.mean(audio.astype(np.float64) ** 2)))
    return 20.0 * np.log10(max(rms, 1e-10))


def strip_silence(audio: np.ndarray, sr: int, top_db: float = 60.0):
    """io.py:58-79."""
    trimmed, (start, end) = lr.trim(audio, top_db=top_db)
    return trimmed, start / sr, (len(audio) - end) / sr


def slice_windows(audio: np.ndarray, sr: int, window_sec: float = 10.0, hop_sec: float = 5.0):
    """io.py:82-112 → list of (chunk, start_sec, end_sec, energy_db)."""
    win_n, hop_n = int(window_sec * sr), int(hop_sec * sr)
    out = []
    start = 0
    while start + win_n <= len(audio):
        chunk = audio[start : start + win_n]
        out.append((chunk, start / sr, (start + win_n) / sr, rms_db(chunk)))
        start += hop_n
    return out


def energy_gate(windows, threshold_db: float = -40.0):
    """io.py:115-126."""
    if not windows:
        return windows
    peak = max(w[3] for w in windows)
    return [w for w in windows if w[3] >= peak + threshold_db]


# ---------------------------------------------------------------------------------- tempo.py
def estimate_tempo(y: np.ndarray, sr: int, start_bpm: float = 120.0, faithful_cost: bool = True) -> Optional[float]:
    """tempo.py:27-77, including the unused tempogram (tempo.py:58) and the repeated
    feature.tempo call (tempo.py:63) when `faithful_cost` — that is what the reference's CPU does."""
    onset_env = lr.onset_strength(y, sr, HOP_LENGTH)
    tempo_default, beat_frames = lr.beat_track(onset_env, sr, HOP_LENGTH, start_bpm)
    tempo_default = float(np.atleast_1d(tempo_default)[0])
    if len(beat_frames) < MIN_BEATS:
        return None
    if faithful_cost:
        lr.tempogram(onset_env, 384)
        tempo_tempogram = float(np.atleast_1d(lr.tempo(onset_env, sr, HOP_LENGTH, start_bpm))[0])
    else:
        tempo_tempogram = tempo_default
    if tempo_default > 0:
        if abs(tempo_default - tempo_tempogram) / tempo_default <= AGREEMENT_TOLERANCE:
            return float((tempo_default + tempo_tempogram) / 2.0)
    return tempo_default if tempo_default > 0 else (tempo_tempogram if tempo_tempogram > 0 else None)


def ibis_from_beats(beat_frames, sr: int, hop_length: int = IBI_HOP_LENGTH, min_ibis: int = 4) -> Optional[np.ndarray]:
    """tempo.py:165-173."""
    beat_frames = np.atleast_1d(beat_frames)
    if len(beat_frames) < min_ibis + 1:
        return None
    t = lr.frames_to_time(beat_frames, sr, hop_length)
    ibis = np.diff(t)
    ibis = ibis[ibis > 0.05]
    if len(ibis) < min_ibis:
        return None
    return ibis


def estimate_ibis_global(y: np.ndarray, sr: int, hop_length: int = IBI_HOP_LENGTH, min_ibis: int = 4,
                         start_bpm: float = 120.0) -> Optional[np.ndarray]:
    """tempo.py:120-173."""
    onset_env = lr.onset_strength(y, sr, hop_length)
    _, beat_frames = lr.beat_track(onset_env, sr, hop_length, start_bpm)
    return ibis_from_beats(beat_frames, sr, hop_length, min_ibis)


# ---------------------------------------------------------------------------------- pitch.py
def mean_chroma(audio: np.ndarray, sr: int) -> np.ndarray:
    """pitch.py:55-64 (12 chroma bins: n_chroma is librosa's default)."""
    return lr.chroma_cqt(audio, sr, 512, 36).mean(axis=1)


def cyclic_xcorr_peak(src_chroma: np.ndarray, nc_chroma: np.ndarray) -> int:
    """pitch.py:67-85."""
    n = len(src_chroma)
    xc = np.array([float(np.dot(src_chroma, np.roll(nc_chroma, -k))) for k in range(n)])
    lag = int(np.argmax(xc))
    if lag > n // 2:
        lag -= n
    return lag


def chunk_pairs(src_audio: np.ndarray, nc_audio: np.ndarray, sr: int):
    """pitch.py:120-138: same-index 20 s chunks, or the whole files when either is shorter."""
    chunk_n = int(CHUNK_SEC * sr)
    n_chunks = min(len(src_audio) // chunk_n, len(nc_audio) // chunk_n)
    if n_chunks < 1:
        return [(src_audio, nc_audio)]
    return [(src_audio[i * chunk_n : (i + 1) * chunk_n], nc_audio[i * chunk_n : (i + 1) * chunk_n])
            for i in range(n_chunks)]


def estimate_pitch_chroma(src_audio: np.ndarray, nc_audio: np.ndarray, sr: int):
    """pitch.py:100-173 → (src_hz, nc_hz, point_st, (lo_st, hi_st), n_chunks, lags)."""
    pairs = chunk_pairs(src_audio, nc_audio, sr)
    lags = [cyclic_xcorr_peak(mean_chroma(s, sr), mean_chroma(n, sr)) for s, n in pairs]
    shift = np.array([lag / 3.0 for lag in lags])
    n_chunks = len(pairs)
    point = float(np.median(shift))
    if n_chunks >= MIN_CHUNKS:
        boots = native.bootstrap(shift, None, 2000, 0)
        lo, hi = float(np.percentile(boots, 2.5)), float(np.percentile(boots, 97.5))
    else:
        lo = hi = point
    src_hz = [440.0] * n_chunks
    nc_hz = [440.0 * (2.0 ** (st / 12.0)) for st in shift]
    return src_hz, nc_hz, point, (lo, hi), n_chunks, lags


# ---------------------------------------------------------------------------------- consensus.py
def valid(values) -> np.ndarray:
    """consensus.py:236-240."""
    return np.array([v for v in values if v is not None and np.isfinite(v) and v > 0], dtype=np.float64)


def bootstrap_ratio(first: np.ndarray, second: np.ndarray, n_boot: int = N_BOOTSTRAP, ci: float = 0.95):
    """median(first)/median(second) + CI, `first` resampled first (consensus.py:243-267 with
    first = nc; consensus.py:270-312 with first = src)."""
    point = float(np.median(first) / np.median(second))
    boot = native.bootstrap(first, second, n_boot, 42)
    alpha = (1.0 - ci) / 2.0
    return point, (float(np.percentile(boot, alpha * 100)), float(np.percentile(boot, (1.0 - alpha) * 100)))


# ---------------------------------------------------------------------------------- pipeline.py
def run_arrays(nc_audio: np.ndarray, src_audio: np.ndarray, sr: int = SAMPLE_RATE, *, window_sec: float = 10.0,
               hop_sec: float = 5.0, energy_gate_db: float = -40.0, silence_strip_db: Optional[float] = 60.0,
               compute_pitch: bool = True, compute_ibi: bool = True, faithful_cost: bool = True,
               log: Optional[Callable[[str], None]] = None, return_window_count: bool = False):
    """pipeline.py:81-216 from the point where both files are loaded."""
    if silence_strip_db is not None:
        nc_audio, _, _ = strip_silence(nc_audio, sr, silence_strip_db)
        src_audio, _, _ = strip_silence(src_audio, sr, silence_strip_db)
    nc_w = energy_gate(slice_windows(nc_audio, sr, window_sec, hop_sec), energy_gate_db)
    src_w = energy_gate(slice_windows(src_audio, sr, window_sec, hop_sec), energy_gate_db)
    if not nc_w or not src_w:
        raise RuntimeError(
            "All windows were discarded by the energy gate.  "
            "Try raising --energy-gate (e.g. --energy-gate -60)."
        )
    out = {}
    if compute_pitch:
        src_hz, nc_hz, point_st, ci_st, n_chunks, lags = estimate_pitch_chroma(src_audio, nc_audio, sr)
        out.update(src_hz=src_hz, nc_hz=nc_hz, pitch_point_st=point_st, pitch_ci_st=ci_st, chunk_lags=lags)
    else:
        src_hz, nc_hz = [], []
        out.update(src_hz=[], nc_hz=[], chunk_lags=[])
    src_tempos = [estimate_tempo(w[0], sr, 120.0, faithful_cost) for w in src_w]
    nc_duration, src_duration = len(nc_audio) / sr, len(src_audio) / sr
    nc_start_bpm = 120.0
    valid_src = [t for t in src_tempos if t is not None]
    if valid_src and nc_duration > 0 and src_duration > 0:
        nc_start_bpm = float(np.median(valid_src)) * (src_duration / nc_duration)
    nc_tempos = [estimate_tempo(w[0], sr, nc_start_bpm, faithful_cost) for w in nc_w]
    out.update(src_tempos=src_tempos, nc_tempos=nc_tempos, nc_start_bpm=nc_start_bpm, nc_duration=nc_duration,
               src_duration=src_duration)
    src_t, nc_t = valid(src_tempos), valid(nc_tempos)
    if len(src_t) < MIN_VALID or len(nc_t) < MIN_VALID:
        raise ValueError(
            f"Insufficient valid tempo windows (source: {len(src_t)}, "
            f"nightcore: {len(nc_t)}).  Need ≥ {MIN_VALID} each."
        )
    src_p, nc_p = valid(src_hz), valid(nc_hz)
    out["pitch"] = bootstrap_ratio(nc_p, src_p) if len(src_p) >= MIN_VALID and len(nc_p) >= MIN_VALID else None
    out["tempo"] = bootstrap_ratio(nc_t, src_t)
    out["ibi"] = None
    if compute_ibi:
        nc_ibis = estimate_ibis_global(nc_audio, sr, start_bpm=nc_start_bpm)
        src_ibis = estimate_ibis_global(src_audio, sr)
        if nc_ibis is not None and len(nc_ibis) >= 4 and src_ibis is not None and len(src_ibis) >= 4:
            out["ibi"] = bootstrap_ratio(src_ibis, nc_ibis)
            out["n_ibis"] = (len(nc_ibis), len(src_ibis))
    if return_window_count:
        return out, len(src_w) + len(nc_w)
    return out


# ---------------------------------------------------------------------------------------------- xcorr.py
XCORR_RMS_GATE = 1e-3     # xcorr.py:38
ALIGN_SR = 11025          # xcorr.py:45
ALIGN_HOP = 512


def speed_xcorr_arrays(ya: np.ndarray, yb: np.ndarray, sr: int = 22050, n_windows: int = 20, window_sec: float = 3.0,
                       search_range: float = 0.05, skip_edges: float = 0.10, return_indices: bool = False,
                       stride: Optional[int] = None):
    """xcorr.py:95-162 from the point where both files are loaded at `sr`: edge trim, 20 reference
    windows of A, strided float32 cosine search in B (stride = win//4 unless given, first strict maximum), polyfit
    slope + median quality.  Returns (slope, quality) [+ (a_pos, best_pb or -1 per window)]."""
    min_len = min(len(ya), len(yb))
    s, e = int(min_len * skip_edges), int(min_len * (1.0 - skip_edges))
    ya, yb = ya[s:e], yb[s:e]
    win = int(window_sec * sr)
    search = int(search_range * len(yb))
    if stride is None:
        stride = max(1, win // 4)
    if len(ya) < win or len(yb) < win:
        return ((1.0, 0.0), (np.zeros(0, np.int64), np.zeros(0, np.int64))) if return_indices else (1.0, 0.0)
    a_positions = np.linspace(0, len(ya) - win, n_windows).astype(int)
    picks = np.full(len(a_positions), -1, dtype=np.int64)
    quals = np.zeros(len(a_positions))
    for i, pa in enumerate(a_positions):
        wa = ya[pa : pa + win]
        if float(np.sqrt(np.mean(wa ** 2))) < XCORR_RMS_GATE:
            continue
        expected = int(pa * len(yb) / len(ya))
        lo_b, hi_b = max(0, expected - search), min(len(yb) - win, expected + search)
        if lo_b >= hi_b:
            continue
        norm_a = float(np.linalg.norm(wa))
        if norm_a < 1e-10:
            continue
        best_c, best_pb = -1.0, expected
        for pb in range(lo_b, hi_b, stride):
            wb = yb[pb : pb + win]
            norm_b = float(np.linalg.norm(wb))
            if norm_b < 1e-10:
                continue
            c = float(np.dot(wa, wb) / (norm_a * norm_b))
            if c > best_c:
                best_c, best_pb = c, pb
        if best_c > 0:
            picks[i], quals[i] = best_pb, best_c
    keep = picks >= 0
    if keep.sum() < 3:
        res = (1.0, 0.0)
    else:
        res = (float(np.polyfit(a_positions[keep].astype(float), picks[keep].astype(float), 1)[0]),
               float(np.median(quals[keep])))
    return (res, (a_positions.astype(np.int64), picks)) if return_indices else res


def content_offset(src_audio: np.ndarray, nc_audio: np.ndarray, sr: int, speed_lo: float = 1.03, speed_hi: float = 1.50,
                   n_speeds: int = 30, max_offset_sec: float = 120.0, return_debug: bool = False):
    """xcorr.py:165-259: RMS envelopes at 11 025 Hz (hop 512), 30 candidate speeds, np.interp stretch,
    np.correlate('valid') over the first max_offset frames, cosine-normalised peak."""
    src_env = lr.rms(lr.resample(src_audio, sr, ALIGN_SR), 2048, ALIGN_HOP).astype(np.float64)
    nc_env = lr.rms(lr.resample(nc_audio, sr, ALIGN_SR), 2048, ALIGN_HOP).astype(np.float64)
    hop_sec = ALIGN_HOP / ALIGN_SR
    max_frames = int(max_offset_sec / hop_sec)
    best = (-1.0, 0.0, (speed_lo + speed_hi) / 2.0)
    dbg = []
    for speed in np.linspace(speed_lo, speed_hi, n_speeds):
        n_st = int(len(nc_env) / speed)
        if n_st < 4 or n_st >= len(src_env):
            dbg.append(None)
            continue
        stretched = np.interp(np.linspace(0.0, 1.0, n_st), np.linspace(0.0, 1.0, len(nc_env)), nc_env)
        search_len = min(max_frames, len(src_env) - n_st)
        if search_len <= 0:
            dbg.append(None)
            continue
        corr = np.correlate(src_env[: search_len + n_st], stretched, mode="valid")[: search_len + 1]
        pk = int(np.argmax(corr))
        denom = np.sqrt(float(np.sum(src_env[pk : pk + n_st] ** 2)) * float(np.sum(stretched ** 2)))
        score = float(corr[pk]) / denom if denom > 1e-12 else 0.0
        dbg.append((pk, score))
        if score > best[0]:
            best = (score, pk * hop_sec, speed)
    return ((best[1], best[2]), dbg) if return_debug else (best[1], best[2])


# ---------------------------------------------------------------------------------------------- spectral.py
def spectral_stats(y: np.ndarray, sr: int) -> dict:
    """spectral.analyze (spectral.py:54-103) from the point where the file is loaded at its native rate."""
    y = np.asarray(y, dtype=np.float32)
    centroid = float(np.mean(lr.spectral_centroid(y, sr)))
    rolloff = float(np.mean(lr.spectral_rolloff(y, sr, roll_percent=0.85)))
    rms = lr.rms(y, 2048, 512)
    stft = np.abs(lr.stft(y))
    freqs = lr.fft_frequencies(sr)

    def band(lo, hi):
        mask = (freqs >= lo) & (freqs < hi)
        return float(np.mean(stft[mask, :])) if mask.any() else 0.0

    loud = rms[rms > np.percentile(rms, 75)]
    stft_db = lr.amplitude_to_db(stft, ref=np.max)
    freq_avg_db = np.mean(stft_db, axis=1)
    significant = freq_avg_db > (np.max(freq_avg_db) - 60.0)
    bw = float(freqs[np.where(significant)[0][-1]]) if significant.any() else float(freqs[-1])
    return dict(centroid=centroid, rolloff=rolloff, rms_mean=float(np.mean(rms)), rms_variance=float(np.var(rms)),
                sub_bass=band(20, 80), bass=band(80, 250), midrange=band(250, 2000), presence=band(2000, 6000),
                brilliance=band(6000, 20000), decay_rate=float(np.mean(np.diff(loud))) if len(loud) > 1 else 0.0,
                duration=len(y) / float(sr), effective_bandwidth_hz=bw, freq_avg_db=freq_avg_db)
