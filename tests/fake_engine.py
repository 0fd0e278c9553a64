"""CPU stand-in for ``nightcore_analyzer._engine.Engine`` — TEST INFRASTRUCTURE.

Same method contracts as the real engine (names, argument meaning, return shapes and dtypes), but every "device"
tensor is a CPU torch tensor and the arithmetic is the oracle's (oracle/librosa_restated.py, oracle/native.py).  It lets
the ``-m "not gpu"`` tier execute the product's HOST logic — io / tempo / pitch / consensus / pipeline and the batch
path of batch.analyse_staged: segment tables, gating, priors, log lines, result assembly — end to end without a GPU,
against the same golden vectors the CUDA path is held to.  Nothing in the product imports this file."""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from nightcore_analyzer._engine import aligned_layout
from oracle import librosa_restated as lr
from oracle import native


class FakeEngine:
    device = torch.device("cpu")

    def __init__(self):
        self.launches = 0
        self.h2d_bytes = 0
        self.d2h_bytes = 0

    # ---- transfers
    def to_dev(self, a, dtype=None) -> torch.Tensor:
        t = torch.from_numpy(np.ascontiguousarray(a).copy())
        return t if dtype is None else t.to(dtype)

    def to_host(self, t: torch.Tensor) -> np.ndarray:
        self.d2h_bytes += t.numel() * t.element_size()
        return t.cpu().numpy()

    def pack(self, arrays: Sequence[np.ndarray]) -> Tuple[torch.Tensor, np.ndarray, np.ndarray]:
        lens = np.array([len(a) for a in arrays], dtype=np.int32)
        starts, pos = aligned_layout(lens)
        host = torch.zeros(max(pos, 4), dtype=torch.float32)
        for a, s, n in zip(arrays, starts, lens):
            host.numpy()[s : s + n] = np.asarray(a, dtype=np.float32)
        return host, starts, lens

    @staticmethod
    def _seg(audio: torch.Tensor, off, ln) -> np.ndarray:
        return audio.numpy()[int(off) : int(off) + int(ln)]

    # ---- io.py
    def window_energy_dev(self, audio, seg_off: torch.Tensor, seg_len: torch.Tensor) -> torch.Tensor:
        out = [float(np.mean(self._seg(audio, o, n).astype(np.float64) ** 2)) if int(n) else 0.0
               for o, n in zip(seg_off.tolist(), seg_len.tolist())]
        return torch.tensor(out, dtype=torch.float64)

    def trim_bounds_dev(self, audio, seg_off: np.ndarray, seg_len: np.ndarray, top_db: float) -> torch.Tensor:
        out = np.zeros((len(seg_len), 2), dtype=np.int64)
        for i, (o, n) in enumerate(zip(seg_off, seg_len)):
            _, (s, e) = lr.trim(self._seg(audio, o, n), top_db=top_db)
            out[i] = (s, e)
        return torch.from_numpy(out)

    # ---- tempo.py
    def tempo_segments_dev(self, audio, seg_off: np.ndarray, seg_len: np.ndarray, start_bpm: np.ndarray, hop: int, sr: int):
        lags, beats = [], []
        for o, n, bpm in zip(seg_off, seg_len, np.asarray(start_bpm, dtype=np.float64)):
            env = lr.onset_strength(self._seg(audio, o, n), sr, hop)
            lag = int(lr.tempo_lag(env, sr, hop, float(bpm)))
            lags.append(lag)
            beats.append(np.asarray(lr.beat_track_frames(env, 60.0 * sr / (hop * float(lag)), sr, hop), dtype=np.int32)
                         if lag > 0 else np.zeros(0, np.int32))
        width = max([len(b) for b in beats] + [1])
        table = np.zeros((len(beats), width), dtype=np.int32)
        for i, b in enumerate(beats):
            table[i, : len(b)] = b
        n_beats = np.array([len(b) for b in beats], dtype=np.int32)
        return None, None, None, torch.tensor(lags, dtype=torch.int32), torch.from_numpy(table), torch.from_numpy(n_beats)

    def tempo_and_beats(self, arrays, start_bpm, hop: int, sr: int, want_beats: bool = True):
        audio, off, ln = self.pack(arrays)
        _, _, _, lag, beats, n_beats = self.tempo_segments_dev(audio, off, ln, np.asarray(start_bpm, np.float64), hop, sr)
        hl, hn, hb = lag.numpy(), n_beats.numpy(), beats.numpy()
        if not want_beats:
            return hl, hn
        return hl, [hb[i, : hn[i]].copy() for i in range(len(arrays))]

    # ---- pitch.py
    def chroma_mean_dev(self, audio, seg_off: np.ndarray, seg_len: np.ndarray, sr: int, tuning_idx=None):
        rows = [lr.chroma_cqt(self._seg(audio, o, n), sr, 512, 36).mean(axis=1) for o, n in zip(seg_off, seg_len)]
        return torch.from_numpy(np.asarray(rows, dtype=np.float64).reshape(len(rows), 12)), None

    def cyclic_xcorr_dev(self, src: torch.Tensor, nc: torch.Tensor) -> torch.Tensor:
        lags = []
        for a, b in zip(src.numpy(), nc.numpy()):
            n = len(a)
            xc = np.array([float(np.dot(a, np.roll(b, -k))) for k in range(n)])
            lag = int(np.argmax(xc))
            lags.append(lag - n if lag > n // 2 else lag)
        return torch.tensor(lags, dtype=torch.int32)

    # ---- consensus.py / pitch.py bootstraps
    def bootstrap(self, jobs, seed: int, n_boot: int, q_lo: float, q_hi: float, want_boot: bool = False,
                  want_idx: bool = False):
        out = np.zeros((len(jobs), 3))
        for j, (a, b) in enumerate(jobs):
            a = np.ascontiguousarray(a, dtype=np.float64)
            b = None if b is None else np.ascontiguousarray(b, dtype=np.float64)
            boot = native.bootstrap(a, b, n_boot, seed)
            point = float(np.median(a)) if b is None else float(np.median(a) / np.median(b))
            out[j] = (point, float(np.percentile(boot, q_lo)), float(np.percentile(boot, q_hi)))
        return out, None, None

    # ---- xcorr.py: the candidate loop of estimate_speed_xcorr (xcorr.py:113-148), float32 dots like numpy's
    def xcorr_search_dev(self, a, b, a_pos: np.ndarray, b_lo: np.ndarray, n_cand: np.ndarray, win: int, stride: int,
                         rms_gate: float):
        ya, yb = a.numpy(), b.numpy()
        best_j = np.full(len(a_pos), -1, dtype=np.int32)
        best_c = np.zeros(len(a_pos), dtype=np.float64)
        for w, (pa, lo, nc) in enumerate(zip(a_pos, b_lo, n_cand)):
            wa = ya[int(pa) : int(pa) + win]
            if float(np.sqrt(np.mean(wa ** 2))) < rms_gate:
                continue
            norm_a = float(np.linalg.norm(wa))
            if norm_a < 1e-10:
                continue
            best, bj = -1.0, -1
            for j in range(int(nc)):
                wb = yb[int(lo) + j * stride : int(lo) + j * stride + win]
                norm_b = float(np.linalg.norm(wb))
                if norm_b < 1e-10:
                    continue
                c = float(np.dot(wa, wb)) / (norm_a * norm_b)
                if c > best:
                    best, bj = c, j
            if bj >= 0 and best > 0.0:
                best_j[w], best_c[w] = bj, best
        return torch.from_numpy(best_j), torch.from_numpy(best_c)

    # ---- xcorr.py: intro alignment (xcorr.py:206-252)
    def align_envelope(self, audio: np.ndarray, sr: int, target_sr: int, hop: int) -> torch.Tensor:
        return torch.from_numpy(lr.rms(lr.resample(audio, sr, target_sr), 2048, hop).astype(np.float64))

    def align_search(self, src_env: torch.Tensor, nc_env: torch.Tensor, n_str: np.ndarray, n_lag: np.ndarray):
        s, n = src_env.numpy(), nc_env.numpy()
        peak = np.full(len(n_str), -1, dtype=np.int32)
        score = np.zeros(len(n_str), dtype=np.float64)
        for i, (ns, nl) in enumerate(zip(n_str, n_lag)):
            if nl <= 0:
                continue
            stretched = np.interp(np.linspace(0.0, 1.0, int(ns)), np.linspace(0.0, 1.0, len(n)), n)
            corr = np.correlate(s[: int(nl) - 1 + int(ns)], stretched, mode="valid")[: int(nl)]
            pk = int(np.argmax(corr))
            denom = np.sqrt(float(np.sum(s[pk : pk + int(ns)] ** 2)) * float(np.sum(stretched ** 2)))
            peak[i], score[i] = pk, (float(corr[pk]) / denom if denom > 1e-12 else 0.0)
        return peak, score
