"""
Per-window tempo and full-signal inter-beat intervals — drop-in for the reference's
``nightcore_analyzer/tempo.py`` (tempo.py:22-173: same names, signatures, constants, ``None``
sentinels and log lines).

All windows of a call go through three batched kernel families (libncfa): onset strength
(STFT → mel → dB → flux), tempo (streamed tempogram autocorrelation + log-normal prior argmax) and
the beat-tracking DP.  The reference's second estimator (tempo.py:58-66) is the same
``librosa.feature.tempo`` call that ``beat_track`` already made, so the averaged value equals the
first; the unused tempogram at tempo.py:58 is not computed.
"""
from __future__ import annotations

from typing import Callable, List, Optional

import numpy as np

from . import _engine
from .io import AudioWindow

# ── tunables (tempo.py:22-24) ────────────────────────────────────────────────
MIN_BEATS: int = 4
AGREEMENT_TOLERANCE: float = 0.08
HOP_LENGTH: int = 512

IBI_HOP_LENGTH: int = 64   # tempo.py:116
IBI_MIN_IBIS: int = 4      # tempo.py:117


def _bpm_of_lag(lag: int, sr: int, hop: int) -> float:
    """librosa.tempo_frequencies: 60·sr / (hop·lag) in float64."""
    return float(60.0 * sr / (hop * float(lag)))


def _consensus(lag: int, n_beats: int, sr: int, hop: int) -> Optional[float]:
    """tempo.py:51-77 with both estimators equal to bpms[lag]."""
    if n_beats < MIN_BEATS:
        return None
    tempo_default = _bpm_of_lag(lag, sr, hop) if lag > 0 else 0.0
    tempo_tempogram = tempo_default
    if tempo_default > 0:
        rel_diff = abs(tempo_default - tempo_tempogram) / tempo_default
        if rel_diff <= AGREEMENT_TOLERANCE:
            return float((tempo_default + tempo_tempogram) / 2.0)
    return tempo_default if tempo_default > 0 else (tempo_tempogram if tempo_tempogram > 0 else None)


def _tempo_windows(windows: List[AudioWindow], start_bpm: float) -> List[Optional[float]]:
    if not windows:
        return []
    eng = _engine.get_engine()
    results: List[Optional[float]] = [None] * len(windows)
    # group by (sample rate, resident track) so that windows of one track share one device buffer
    groups: dict = {}
    for i, w in enumerate(windows):
        key = (w.sample_rate, id(w._track) if w._track is not None else None)
        groups.setdefault(key, []).append(i)
    for (sr, tid), idxs in groups.items():
        ws = [windows[i] for i in idxs]
        if tid is not None:
            audio = ws[0]._track.tensor
            seg_off = np.array([w._start for w in ws], dtype=np.int64)
            seg_len = np.array([len(w.audio) for w in ws], dtype=np.int32)
        else:
            audio, seg_off, seg_len = eng.pack([w.audio for w in ws])
        bpm = np.full(len(ws), float(start_bpm), dtype=np.float64)
        _, _, _, lag, _, n_beats = eng.tempo_segments_dev(audio, seg_off, seg_len, bpm, HOP_LENGTH, sr)
        hl, hn = lag.cpu().numpy(), _engine.check_beat_counts(n_beats.cpu().numpy())
        for j, i in enumerate(idxs):
            results[i] = _consensus(int(hl[j]), int(hn[j]), sr, HOP_LENGTH)
    return results


def estimate_tempo(window: AudioWindow, start_bpm: float = 120.0) -> Optional[float]:
    """tempo.py:27-77 — BPM estimate for *window*, or None with fewer than MIN_BEATS beats."""
    return _tempo_windows([window], start_bpm)[0]


def batch_estimate_tempo(
    windows: List[AudioWindow],
    log: Optional[Callable[[str], None]] = None,
    start_bpm: float = 120.0,
) -> List[Optional[float]]:
    """tempo.py:80-111 — all windows in one batched device pass; the per-window progress lines are
    emitted in the reference's order."""
    results = _tempo_windows(list(windows), start_bpm)
    n = len(windows)
    if log:
        for i, w in enumerate(windows):
            log(f"    tempo window {i + 1}/{n}  [{w.start_sec:.1f}–{w.end_sec:.1f} s]")
    valid = sum(1 for r in results if r is not None)
    if log:
        log(f"    {valid}/{n} windows yielded a confident tempo estimate")
    return results


def _ibis_from_beats(beat_frames: np.ndarray, sr: int, hop_length: int, min_ibis: int) -> Optional[np.ndarray]:
    """tempo.py:165-173."""
    beat_frames = np.atleast_1d(beat_frames)
    if len(beat_frames) < min_ibis + 1:
        return None
    t = np.asanyarray(beat_frames) * hop_length / float(sr)   # librosa.frames_to_time
    ibis = np.diff(t)
    ibis = ibis[ibis > 0.05]
    if len(ibis) < min_ibis:
        return None
    return ibis


def estimate_ibis_global(
    y: np.ndarray,
    sr: int,
    hop_length: int = IBI_HOP_LENGTH,
    min_ibis: int = IBI_MIN_IBIS,
    start_bpm: float = 120.0,
) -> Optional[np.ndarray]:
    """tempo.py:120-173 — beat-track the whole signal at hop 64 and return the inter-beat
    intervals in seconds (sub-50 ms intervals dropped), or None."""
    eng = _engine.get_engine()
    _, beats = eng.tempo_and_beats([np.ascontiguousarray(y, dtype=np.float32)], [float(start_bpm)], hop_length, sr)
    return _ibis_from_beats(beats[0], sr, hop_length, min_ibis)
