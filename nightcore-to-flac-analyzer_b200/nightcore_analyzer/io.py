"""
Audio I/O, windowing, energy gating and silence stripping — drop-in for the reference's
``nightcore_analyzer/io.py`` (same names, signatures, constants and return types; io.py:19-126).

The reductions run on the GPU (libncfa: ``ncfa_window_energy`` in float64 for ``_rms_db`` /
``slice_windows``, ``ncfa_rms_frames`` for ``strip_silence``).  ``slice_windows`` uploads the
track once and every returned ``AudioWindow`` remembers where its samples live on the device, so
``tempo.batch_estimate_tempo`` does not copy them again.
"""
from __future__ import annotations

import wave
from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np

from . import _engine

# ── defaults (io.py:19-23) ───────────────────────────────────────────────────
SAMPLE_RATE: int = 22050
WINDOW_SEC: float = 10.0
HOP_SEC: float = 5.0
ENERGY_GATE_DB: float = -40.0
SILENCE_STRIP_DB: float = 60.0


class DeviceTrack:
    """A whole track resident in HBM (float32, mono)."""

    __slots__ = ("tensor", "n", "sr")

    def __init__(self, tensor, n: int, sr: int):
        self.tensor, self.n, self.sr = tensor, n, sr


@dataclass
class AudioWindow:
    """One time slice of an audio file (io.py:27-34)."""
    audio: np.ndarray
    sample_rate: int
    start_sec: float
    end_sec: float
    energy_db: float
    # device residency (not part of the reference record; ignored by comparisons)
    _track: Optional[DeviceTrack] = field(default=None, repr=False, compare=False)
    _start: int = field(default=0, repr=False, compare=False)


def upload_track(audio: np.ndarray, sr: int) -> DeviceTrack:
    eng = _engine.get_engine()
    a = np.ascontiguousarray(audio, dtype=np.float32)
    return DeviceTrack(eng.to_dev(a if len(a) else np.zeros(4, np.float32)), len(a), sr)


def _db_from_meansq(meansq: float) -> float:
    rms = float(np.sqrt(meansq))
    return 20.0 * np.log10(max(rms, 1e-10))


def _rms_db(audio: np.ndarray) -> float:
    """io.py:38-40 — the float64 mean square is reduced on the device."""
    eng = _engine.get_engine()
    a = np.ascontiguousarray(audio, dtype=np.float32)
    if len(a) == 0:
        return _db_from_meansq(float("nan"))
    d = eng.to_dev(a)
    ms = eng.window_energy_dev(d, eng.to_dev(np.zeros(1, np.int64)), eng.to_dev(np.array([len(a)], np.int32)))
    return _db_from_meansq(float(ms.cpu().numpy()[0]))


def read_wav(path: str) -> tuple[np.ndarray, int, int]:
    """PCM ``.wav`` → (frames float32 [n, channels], sample rate, sample width in bytes).  8-bit (unsigned), 16-, 24- and
    32-bit (signed) samples are scaled by 2^(bits−1) into [−1, 1)."""
    with wave.open(str(path), "rb") as w:
        n, ch, sw, fr = w.getnframes(), w.getnchannels(), w.getsampwidth(), w.getframerate()
        raw = w.readframes(n)
    if sw == 2:
        y = np.frombuffer(raw, dtype="<i2").astype(np.float32) / 32768.0
    elif sw == 3:
        b = np.frombuffer(raw, dtype=np.uint8).reshape(-1, 3).astype(np.int32)
        v = b[:, 0] | (b[:, 1] << 8) | (b[:, 2] << 16)
        y = (v - ((v & 0x800000) << 1)).astype(np.float32) / 8388608.0
    elif sw == 4:
        y = np.frombuffer(raw, dtype="<i4").astype(np.float32) / 2147483648.0
    elif sw == 1:
        y = (np.frombuffer(raw, dtype=np.uint8).astype(np.float32) - 128.0) / 128.0
    else:
        raise ValueError(f"unsupported WAV sample width {sw}")
    return y.reshape(-1, ch), fr, sw


def write_wav(path: str, frames: np.ndarray, rate: int, sample_width: int = 2) -> None:
    """frames ([n] or [n, channels], float, full scale ±1) → PCM ``.wav`` of `sample_width` bytes (1, 2, 3 or 4): scaled
    by 2^(bits−1), rounded half to even and clipped to the integer range, without dither.  Writing what ``read_wav``
    returned reproduces a 8-, 16- or 24-bit file's samples exactly."""
    if sample_width not in (1, 2, 3, 4):
        raise ValueError(f"unsupported WAV sample width {sample_width}")
    y = np.asarray(frames, dtype=np.float64)
    y = y.reshape(len(y), -1)
    full = float(1 << (8 * sample_width - 1))
    q = np.clip(np.rint(y * full), -full, full - 1).astype(np.int64)
    if sample_width == 1:
        raw = (q + 128).astype(np.uint8).tobytes()
    elif sample_width == 3:
        raw = (q.reshape(-1, 1) >> np.array([0, 8, 16])).astype(np.uint8).tobytes()
    else:
        raw = q.astype(f"<i{sample_width}").tobytes()
    with wave.open(str(path), "wb") as w:
        w.setnchannels(y.shape[1])
        w.setsampwidth(sample_width)
        w.setframerate(int(rate))
        w.writeframes(raw)


def load_audio(path: str, sr: int = SAMPLE_RATE) -> tuple[np.ndarray, int]:
    """io.py:44-55.  Decoding is out of scope (no librosa/soundfile on the box): accepts ``.npy``
    (float mono already at *sr*) and PCM ``.wav`` read by ``read_wav`` (8-, 16-, 24- or 32-bit; 24-bit files load since
    ``read_wav`` was added, before that they raised ``ValueError``), averaged to mono; a WAV at another rate is
    resampled with scipy's polyphase filter (NOT soxr_hq — documented deviation)."""
    path = str(path)
    if path.endswith(".npy"):
        return np.load(path).astype(np.float32), (sr or SAMPLE_RATE)
    frames, fr, _ = read_wav(path)
    y = frames.mean(axis=1).astype(np.float32) if frames.shape[1] > 1 else frames[:, 0]
    if sr is not None and fr != sr:
        from fractions import Fraction
        import scipy.signal
        f = Fraction(int(sr), int(fr))
        y = scipy.signal.resample_poly(y.astype(np.float64), f.numerator, f.denominator).astype(np.float32)
    return y.astype(np.float32), (sr or fr)


def strip_silence(audio: np.ndarray, sr: int, top_db: float = SILENCE_STRIP_DB) -> tuple[np.ndarray, float, float]:
    """io.py:58-79 — librosa.effects.trim(top_db): framed RMS (2048/512, centred) on the device,
    first/last frame above −top_db relative to the loudest frame."""
    eng = _engine.get_engine()
    a = np.ascontiguousarray(audio, dtype=np.float32)
    n = len(a)
    if n == 0:
        return audio[0:0], 0.0, 0.0
    bounds = eng.to_host(eng.trim_bounds_dev(eng.to_dev(a), np.zeros(1, np.int64), np.array([n], np.int32), top_db))
    start, end = int(bounds[0, 0]), int(bounds[0, 1])
    trimmed = audio[start:end]
    return trimmed, start / sr, (len(audio) - end) / sr


def slice_windows(audio: np.ndarray, sr: int, window_sec: float = WINDOW_SEC, hop_sec: float = HOP_SEC,
                  ) -> List[AudioWindow]:
    """io.py:82-112 — fixed-length overlapping windows; the per-window energies come from one
    batched float64 reduction on the device."""
    win_n = int(window_sec * sr)
    hop_n = int(hop_sec * sr)
    starts = []
    start = 0
    while start + win_n <= len(audio):
        starts.append(start)
        start += hop_n
    if not starts:
        return []
    eng = _engine.get_engine()
    track = upload_track(audio, sr)
    seg_off = np.asarray(starts, dtype=np.int64)
    seg_len = np.full(len(starts), win_n, dtype=np.int32)
    if win_n > 0:
        ms = eng.window_energy_dev(track.tensor, eng.to_dev(seg_off), eng.to_dev(seg_len)).cpu().numpy()
    else:
        ms = np.full(len(starts), np.nan)
    return [
        AudioWindow(audio=audio[s : s + win_n], sample_rate=sr, start_sec=s / sr, end_sec=(s + win_n) / sr,
                    energy_db=_db_from_meansq(float(m)), _track=track, _start=int(s))
        for s, m in zip(starts, ms)
    ]


def energy_gate(windows: List[AudioWindow], threshold_db: float = ENERGY_GATE_DB) -> List[AudioWindow]:
    """io.py:115-126."""
    if not windows:
        return windows
    peak_db = max(w.energy_db for w in windows)
    return [w for w in windows if w.energy_db >= peak_db + threshold_db]
