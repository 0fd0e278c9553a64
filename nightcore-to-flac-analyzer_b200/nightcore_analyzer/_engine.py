"""Device engine: torch owns memory and streams, libncfa.so does the arithmetic.

A *segment* is a contiguous run of samples inside one device audio buffer (an analysis window,
a pitch chunk or a whole track).  Every method that ends in ``_dev`` takes and returns device
tensors and never synchronises; the list-of-numpy convenience wrappers upload, run and download.
"""
from __future__ import annotations

import math
import threading
import weakref
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _native
from ._native import check, lib

# Intermediate log-mel tiles are sized to stay resident in the 126 MB L2 between the STFT kernel
# and the flux kernel (DESIGN.md "onset front-end").
ONSET_WS_TARGET_BYTES = 96 << 20
MAX_SEGS_PER_CALL = 65535
# tuning peak lists / decimation pyramids of one launch (HBM scratch, reused across sub-batches)
CHROMA_WS_TARGET_BYTES = 4 << 30
# pinned staging ring for parameter uploads (to_dev)
PARAM_RING_BYTES = 128 << 20


def _ptr(t: Optional[torch.Tensor]) -> int:
    return 0 if t is None else t.data_ptr()


def aligned_layout(lengths) -> Tuple[np.ndarray, int]:
    """Offsets (int64) of arrays of the given lengths laid end to end in one buffer, each starting on a 4-sample (16 B)
    boundary, and the buffer's total length.  Aligned starts put the kernels on their vector-load fast paths; any other
    start gives the same results (tests/test_gpu_segment_placement.py)."""
    padded = (np.asarray(lengths, dtype=np.int64) + 3) // 4 * 4
    off = np.zeros(len(padded), dtype=np.int64)
    np.cumsum(padded[:-1], out=off[1:])
    return off, int(padded.sum())


class Engine:
    def __init__(self, device: Optional[torch.device] = None):
        if not torch.cuda.is_available():
            raise _native.NcfaError("nightcore_analyzer needs a CUDA device (sm_100a); there is no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self._ws: dict = {}
        self._lock = threading.Lock()
        self.launches = 0  # kernels launched through this engine (bench.py's gpu_launches)
        self._ring: Optional[torch.Tensor] = None  # pinned parameter ring (to_dev)
        self._ring_pos = 0
        self.h2d_bytes = 0
        self.d2h_bytes = 0

    # ------------------------------------------------------------------ plumbing
    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def workspace(self, name: str, nbytes: int) -> torch.Tensor:
        nbytes = max(256, int(nbytes))
        t = self._ws.get(name)
        if t is None or t.numel() < nbytes:
            self._ws[name] = None
            t = torch.empty(int(nbytes * 1.25) if t is not None else nbytes, dtype=torch.uint8, device=self.device)
            self._ws[name] = t
        return t

    def to_dev(self, a: np.ndarray, dtype=None) -> torch.Tensor:
        """Host array → device tensor on the current stream.  Parameter-sized arrays (segment tables, priors, bootstrap
        values) do not use the DMA engine: a copy queued there waits behind any bulk audio upload in flight (65 ms for
        a 125-pair sub-batch) and every such wait is a hole in the kernel stream.  They are written into a pinned ring
        and moved by a small kernel that reads the ring over PCIe (ncfa_param_upload)."""
        t = torch.from_numpy(np.ascontiguousarray(a))
        if dtype is not None:
            t = t.to(dtype)
        nbytes = t.numel() * t.element_size()
        self.h2d_bytes += nbytes
        if nbytes == 0 or nbytes > PARAM_RING_BYTES // 8:
            return t.to(self.device, non_blocking=True)
        out = torch.empty(t.shape, dtype=t.dtype, device=self.device)
        off = self._ring_reserve(nbytes)
        self._ring[off : off + nbytes].copy_(t.reshape(-1).view(torch.uint8))
        with torch.cuda.device(self.device):
            check(lib.ncfa_param_upload(out.data_ptr(), self._ring.data_ptr() + off, nbytes, self._stream()),
                  "ncfa_param_upload")
        self.launches += 1
        return out

    def _ring_reserve(self, nbytes: int) -> int:
        """16-byte aligned slot of the pinned parameter ring.  Slots are reused only after a wrap, and a wrap waits for
        the device once (every PARAM_RING_BYTES of parameters, i.e. every few dozen sub-batches)."""
        if self._ring is None:
            self._ring = torch.empty(PARAM_RING_BYTES, dtype=torch.uint8, pin_memory=True)
            self._ring_pos = 0
        need = (nbytes + 15) // 16 * 16
        if self._ring_pos + need > PARAM_RING_BYTES:
            torch.cuda.synchronize(self.device)
            self._ring_pos = 0
        off = self._ring_pos
        self._ring_pos += need
        return off

    def to_host(self, t: torch.Tensor) -> np.ndarray:
        self.d2h_bytes += t.numel() * t.element_size()
        return t.cpu().numpy()

    def pack(self, arrays: Sequence[np.ndarray]) -> Tuple[torch.Tensor, np.ndarray, np.ndarray]:
        """Concatenate float32 arrays into one device buffer → (audio, seg_off int64, seg_len int32) (host descriptors)."""
        lens = np.array([len(a) for a in arrays], dtype=np.int32)
        starts, pos = aligned_layout(lens)
        host = torch.zeros(max(pos, 4), dtype=torch.float32)
        hn = host.numpy()
        for a, s, n in zip(arrays, starts, lens):
            hn[s : s + n] = np.asarray(a, dtype=np.float32)
        self.h2d_bytes += host.numel() * 4
        return host.to(self.device, non_blocking=True), starts, lens

    # ------------------------------------------------------------------ io.py: energies
    def window_energy_dev(self, audio: torch.Tensor, seg_off: torch.Tensor, seg_len: torch.Tensor) -> torch.Tensor:
        n = seg_off.numel()
        out = torch.empty(n, dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            check(lib.ncfa_window_energy(_ptr(audio), _ptr(seg_off), _ptr(seg_len), n, _ptr(out), self._stream()),
                  "ncfa_window_energy")
        self.launches += 1
        return out

    def rms_frames_dev(self, audio: torch.Tensor, n: int, frame_length: int, hop: int) -> torch.Tensor:
        out = torch.empty(1 + n // hop, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            check(lib.ncfa_rms_frames(_ptr(audio), int(n), int(frame_length), int(hop), _ptr(out), self._stream()),
                  "ncfa_rms_frames")
        self.launches += 1
        return out

    def trim_bounds_dev(self, audio: torch.Tensor, seg_off: np.ndarray, seg_len: np.ndarray, top_db: float) -> torch.Tensor:
        """librosa.effects.trim bounds of every segment → int64 [n_seg, 2] (start, end) on the device."""
        n_seg = len(seg_len)
        out = torch.zeros((max(n_seg, 1), 2), dtype=torch.int64, device=self.device)
        if n_seg == 0:
            return out[:0]
        d_off, d_len = self.to_dev(seg_off.astype(np.int64)), self.to_dev(seg_len.astype(np.int32))
        with torch.cuda.device(self.device):
            st = self._stream()
            for s in range(0, n_seg, MAX_SEGS_PER_CALL):
                e = min(n_seg, s + MAX_SEGS_PER_CALL)
                mx = int(seg_len[s:e].max())
                ws = self.workspace("trim", lib.ncfa_trim_workspace_bytes(e - s, mx))
                check(lib.ncfa_trim_bounds_batched(_ptr(audio), d_off.data_ptr() + 8 * s, d_len.data_ptr() + 4 * s, e - s, mx,
                                                   float(top_db), out.data_ptr() + 16 * s, _ptr(ws), ws.numel(), st),
                      "ncfa_trim_bounds_batched")
                self.launches += 2
        return out[:n_seg]

    # ------------------------------------------------------------------ onset strength
    @staticmethod
    def env_layout(seg_len: np.ndarray, hop: int) -> Tuple[np.ndarray, np.ndarray, int]:
        env_len = (1 + seg_len.astype(np.int64) // hop).astype(np.int32)
        return (env_len, *aligned_layout(env_len))

    def onset_strength_dev(self, audio: torch.Tensor, seg_off: np.ndarray, seg_len: np.ndarray, hop: int, sr: int,
                           d_seg_off: Optional[torch.Tensor] = None, d_seg_len: Optional[torch.Tensor] = None):
        """librosa.onset.onset_strength for every segment → (onset f32 packed, env_off (host int64),
        env_len (host int32), d_env_off, d_env_len)."""
        n_seg = len(seg_len)
        env_len, env_off, total = self.env_layout(seg_len, hop)
        onset = torch.empty(max(total, 4), dtype=torch.float32, device=self.device)
        d_env_off = self.to_dev(env_off)
        d_env_len = self.to_dev(env_len)
        if d_seg_off is None:
            d_seg_off = self.to_dev(seg_off.astype(np.int64))
        if d_seg_len is None:
            d_seg_len = self.to_dev(seg_len.astype(np.int32))
        if n_seg == 0:
            return onset, env_off, env_len, d_env_off, d_env_len
        # chunk the batch so the log-mel workspace of one launch stays L2-resident
        order_max = int(seg_len.max())
        per_seg = (1 + order_max // hop) * 128 * 4
        per_call = max(1, min(MAX_SEGS_PER_CALL, ONSET_WS_TARGET_BYTES // max(1, per_seg)))
        with torch.cuda.device(self.device):
            st = self._stream()
            for s in range(0, n_seg, per_call):
                e = min(n_seg, s + per_call)
                mx = int(seg_len[s:e].max())
                need = lib.ncfa_onset_workspace_bytes(e - s, mx, hop)
                ws = self.workspace("onset", need)
                check(
                    lib.ncfa_onset_strength_batched(
                        _ptr(audio), d_seg_off.data_ptr() + 8 * s, d_seg_len.data_ptr() + 4 * s, e - s, mx, hop, sr,
                        _ptr(onset), d_env_off.data_ptr() + 8 * s, _ptr(ws), ws.numel(), st),
                    "ncfa_onset_strength_batched")
                self.launches += 2
        return onset, env_off, env_len, d_env_off, d_env_len

    # ------------------------------------------------------------------ tempo (tempogram argmax)
    def tempo_lag_dev(self, onset: torch.Tensor, d_env_off: torch.Tensor, d_env_len: torch.Tensor, env_len: np.ndarray,
                      hop: int, sr: int, d_start_bpm: torch.Tensor) -> torch.Tensor:
        n_seg = len(env_len)
        lag = torch.zeros(max(n_seg, 1), dtype=torch.int32, device=self.device)
        if n_seg == 0:
            return lag[:0]
        W = int(math.floor(8.0 * sr / hop))
        if not 4 <= W <= 5000:
            # the tempogram kernels keep one 8-second window of the envelope per CTA in shared memory
            raise ValueError(f"unsupported sr / hop for the tempogram: its 8 s window is {W} onset frames at sr={sr}, "
                             f"hop={hop}; supported: 4..5000 frames (sr/hop <= 625, e.g. sr <= 40000 Hz at hop 64)")
        with torch.cuda.device(self.device):
            st = self._stream()
            for s in range(0, n_seg, MAX_SEGS_PER_CALL):
                e = min(n_seg, s + MAX_SEGS_PER_CALL)
                mx = int(env_len[s:e].max())
                need = lib.ncfa_tempo_workspace_bytes(e - s, mx, W)
                ws = self.workspace("tempo", need)
                check(
                    lib.ncfa_tempo_lag_batched(
                        _ptr(onset), d_env_off.data_ptr() + 8 * s, d_env_len.data_ptr() + 4 * s, e - s, mx, hop, sr,
                        d_start_bpm.data_ptr() + 8 * s, lag.data_ptr() + 4 * s, _ptr(ws), ws.numel(), st),
                    "ncfa_tempo_lag_batched")
                self.launches += 8
        return lag[:n_seg]

    # ------------------------------------------------------------------ beat tracker
    @staticmethod
    def max_beats_for(max_env_len: int, hop: int, sr: int) -> int:
        k_min = 1
        while not (60.0 * sr / (hop * k_min) < 320.0):
            k_min += 1
        near = max(1, int(round(k_min / 2.0)))
        return max_env_len // near + 2

    def beat_track_dev(self, onset: torch.Tensor, d_env_off: torch.Tensor, d_env_len: torch.Tensor, env_len: np.ndarray,
                       lag: torch.Tensor, hop: int, sr: int):
        n_seg = len(env_len)
        W = int(math.floor(8.0 * sr / hop))
        mx = int(env_len.max()) if n_seg else 1
        max_beats = self.max_beats_for(mx, hop, sr)
        beats = torch.empty((max(n_seg, 1), max_beats), dtype=torch.int32, device=self.device)
        n_beats = torch.zeros(max(n_seg, 1), dtype=torch.int32, device=self.device)
        if n_seg == 0:
            return beats[:0], n_beats[:0]
        with torch.cuda.device(self.device):
            need = lib.ncfa_beat_workspace_bytes(n_seg, mx, W)
            ws = self.workspace("beat", need)
            check(
                lib.ncfa_beat_track_batched(_ptr(onset), _ptr(d_env_off), _ptr(d_env_len), n_seg, mx, _ptr(lag), W,
                                            _ptr(beats), max_beats, _ptr(n_beats), _ptr(ws), ws.numel(),
                                            self._stream()),
                "ncfa_beat_track_batched")
            self.launches += 3  # prep, local score, DP
        return beats[:n_seg], n_beats[:n_seg]

    # ------------------------------------------------------------------ fused: segments → (lag, n_beats[, beats])
    def tempo_segments_dev(self, audio: torch.Tensor, seg_off: np.ndarray, seg_len: np.ndarray, start_bpm: np.ndarray,
                           hop: int, sr: int):
        onset, env_off, env_len, d_env_off, d_env_len = self.onset_strength_dev(audio, seg_off, seg_len, hop, sr)
        d_bpm = self.to_dev(np.asarray(start_bpm, dtype=np.float64))
        lag = self.tempo_lag_dev(onset, d_env_off, d_env_len, env_len, hop, sr, d_bpm)
        beats, n_beats = self.beat_track_dev(onset, d_env_off, d_env_len, env_len, lag, hop, sr)
        return onset, env_off, env_len, lag, beats, n_beats

    # ------------------------------------------------------------------ bootstrap (consensus.py / pitch.py)
    @staticmethod
    def pcg64_state(seed: int) -> Tuple[int, int, int, int]:
        """(state_hi, state_lo, inc_hi, inc_lo) of numpy's PCG64(seed); the SeedSequence hashing is numpy's own."""
        st = np.random.PCG64(seed).state["state"]
        s, i = int(st["state"]), int(st["inc"])
        m = (1 << 64) - 1
        return (s >> 64) & m, s & m, (i >> 64) & m, i & m

    def bootstrap_dev(self, d_a: torch.Tensor, a_off: np.ndarray, a_len: np.ndarray, d_b: Optional[torch.Tensor],
                      b_off: Optional[np.ndarray], b_len: Optional[np.ndarray], seed: int, n_boot: int, q_lo: float,
                      q_hi: float, want_boot: bool = False, want_idx: bool = False):
        """Batched PCG64-exact bootstrap; job j: boot = median(a_j*) / median(b_j*) with a drawn first.
        Returns (out[n_jobs,3] = point, lo, hi; boot[n_jobs,n_boot] | None; idx | None) on the device."""
        import ctypes
        n_jobs = len(a_len)
        out = torch.empty((max(n_jobs, 1), 3), dtype=torch.float64, device=self.device)
        if n_jobs == 0:
            return out[:0], None, None
        max_a = int(a_len.max())
        max_b = int(b_len.max()) if b_len is not None else 0
        boot = torch.empty((n_jobs, n_boot), dtype=torch.float64, device=self.device) if want_boot else None
        idx = None
        if want_idx:
            if n_jobs != 1:
                raise ValueError("resample indices are only returned for a single job")
            idx = torch.empty(n_boot * (max_a + max_b), dtype=torch.int32, device=self.device)
        d_a_off, d_a_len = self.to_dev(a_off.astype(np.int64)), self.to_dev(a_len.astype(np.int32))
        d_b_off = self.to_dev(b_off.astype(np.int64)) if d_b is not None else None
        d_b_len = self.to_dev(b_len.astype(np.int32)) if d_b is not None else None
        state = (ctypes.c_uint64 * 4)(*self.pcg64_state(seed))
        with torch.cuda.device(self.device):
            need = lib.ncfa_bootstrap_workspace_bytes(n_jobs, max_a, max_b, n_boot)
            ws = self.workspace("bootstrap", need)
            check(
                lib.ncfa_bootstrap_ratio_batched(_ptr(d_a), _ptr(d_a_off), _ptr(d_a_len), _ptr(d_b), _ptr(d_b_off),
                                                 _ptr(d_b_len), n_jobs, max_a, max_b, n_boot, state, float(q_lo),
                                                 float(q_hi), _ptr(out), _ptr(boot), _ptr(idx), _ptr(ws), ws.numel(),
                                                 self._stream()),
                "ncfa_bootstrap_ratio_batched")
            self.launches += 5
        return out, boot, idx

    def bootstrap(self, jobs: Sequence[Tuple[np.ndarray, Optional[np.ndarray]]], seed: int, n_boot: int, q_lo: float,
                  q_hi: float, want_boot: bool = False, want_idx: bool = False):
        """Host convenience: jobs = [(a, b | None), ...] (all with b or all without)."""
        has_b = jobs[0][1] is not None
        a_list = [np.ascontiguousarray(j[0], dtype=np.float64) for j in jobs]
        a_len = np.array([len(a) for a in a_list], dtype=np.int32)
        a_off = np.concatenate([[0], np.cumsum(a_len)[:-1]]).astype(np.int64)
        d_a = self.to_dev(np.concatenate(a_list) if a_list else np.zeros(1))
        d_b = b_off = b_len = None
        if has_b:
            b_list = [np.ascontiguousarray(j[1], dtype=np.float64) for j in jobs]
            b_len = np.array([len(b) for b in b_list], dtype=np.int32)
            b_off = np.concatenate([[0], np.cumsum(b_len)[:-1]]).astype(np.int64)
            d_b = self.to_dev(np.concatenate(b_list))
        out, boot, idx = self.bootstrap_dev(d_a, a_off, a_len, d_b, b_off, b_len, seed, n_boot, q_lo, q_hi,
                                            want_boot, want_idx)
        return (out.cpu().numpy(), None if boot is None else boot.cpu().numpy(),
                None if idx is None else idx.cpu().numpy())

    # ------------------------------------------------------------------ pitch.py: tuning, CQT chroma, cyclic xcorr
    def chroma_mean_dev(self, audio: torch.Tensor, seg_off: np.ndarray, seg_len: np.ndarray, sr: int,
                        tuning_idx: Optional[torch.Tensor] = None):
        """pitch._mean_chroma for every segment → (chroma float64 [n_seg, 12], tuning_idx int32 [n_seg]) on the
        device.  ``tuning_idx`` given: skip librosa.estimate_tuning and use those histogram bins."""
        n_seg = len(seg_len)
        chroma = torch.empty((max(n_seg, 1), 12), dtype=torch.float64, device=self.device)
        tun = torch.empty(max(n_seg, 1), dtype=torch.int32, device=self.device)
        if n_seg == 0:
            return chroma[:0], tun[:0]
        if tuning_idx is not None:
            tun[:n_seg] = tuning_idx.to(self.device, torch.int32)
        d_off = self.to_dev(seg_off.astype(np.int64))
        d_len = self.to_dev(seg_len.astype(np.int32))
        mx_all = int(seg_len.max())
        per_seg = max(lib.ncfa_tuning_workspace_bytes(1, mx_all), lib.ncfa_chroma_workspace_bytes(1, mx_all), 1)
        per_call = max(1, min(MAX_SEGS_PER_CALL, CHROMA_WS_TARGET_BYTES // per_seg))
        with torch.cuda.device(self.device):
            st = self._stream()
            for s in range(0, n_seg, per_call):
                e = min(n_seg, s + per_call)
                mx = int(seg_len[s:e].max())
                if tuning_idx is None:
                    need = lib.ncfa_tuning_workspace_bytes(e - s, mx)
                    ws = self.workspace("chroma", need)
                    check(lib.ncfa_tuning_estimate_batched(_ptr(audio), d_off.data_ptr() + 8 * s, d_len.data_ptr() + 4 * s,
                                                           e - s, mx, sr, tun.data_ptr() + 4 * s, _ptr(ws), ws.numel(), st),
                          "ncfa_tuning_estimate_batched")
                    self.launches += 2
                need = lib.ncfa_chroma_workspace_bytes(e - s, mx)
                ws = self.workspace("chroma", need)
                check(lib.ncfa_chroma_mean_batched(_ptr(audio), d_off.data_ptr() + 8 * s, d_len.data_ptr() + 4 * s, e - s,
                                                   mx, sr, tun.data_ptr() + 4 * s, chroma.data_ptr() + 96 * s, _ptr(ws),
                                                   ws.numel(), st),
                      "ncfa_chroma_mean_batched")
                self.launches += 8
        return chroma[:n_seg], tun[:n_seg]

    def cyclic_xcorr_dev(self, src: torch.Tensor, nc: torch.Tensor) -> torch.Tensor:
        """pitch._cyclic_xcorr_peak for n pairs of float64 vectors [n, n_bins] → int32 lags."""
        n, bins = src.shape
        lag = torch.empty(max(n, 1), dtype=torch.int32, device=self.device)
        if n == 0:
            return lag[:0]
        src, nc = src.contiguous(), nc.contiguous()
        with torch.cuda.device(self.device):
            check(lib.ncfa_cyclic_xcorr_batched(_ptr(src), _ptr(nc), n, bins, _ptr(lag), self._stream()),
                  "ncfa_cyclic_xcorr_batched")
        self.launches += 1
        return lag[:n]

    # ------------------------------------------------------------------ xcorr.py: candidate search
    def xcorr_search_dev(self, a: torch.Tensor, b: torch.Tensor, a_pos: np.ndarray, b_lo: np.ndarray,
                         n_cand: np.ndarray, win: int, stride: int, rms_gate: float):
        """Strided normalised-dot-product search (xcorr.py:113-148) → (best_j int32, best_c float64) on the device."""
        n_w = len(a_pos)
        best_j = torch.empty(max(n_w, 1), dtype=torch.int32, device=self.device)
        best_c = torch.empty(max(n_w, 1), dtype=torch.float64, device=self.device)
        if n_w == 0:
            return best_j[:0], best_c[:0]
        max_cand = max(1, int(n_cand.max()))
        d_pos, d_lo, d_nc = self.to_dev(a_pos.astype(np.int64)), self.to_dev(b_lo.astype(np.int64)), self.to_dev(
            n_cand.astype(np.int32))
        with torch.cuda.device(self.device):
            for s in range(0, n_w, MAX_SEGS_PER_CALL):       # the window index is gridDim.y
                e = min(n_w, s + MAX_SEGS_PER_CALL)
                need = lib.ncfa_xcorr_workspace_bytes(e - s, max_cand)
                ws = self.workspace("xcorr", need)
                check(lib.ncfa_xcorr_search_batched(_ptr(a), _ptr(b), d_pos.data_ptr() + 8 * s, d_lo.data_ptr() + 8 * s,
                                                    d_nc.data_ptr() + 4 * s, e - s, max_cand, int(win), int(stride),
                                                    float(rms_gate), best_j.data_ptr() + 4 * s, best_c.data_ptr() + 8 * s,
                                                    _ptr(ws), ws.numel(), self._stream()),
                      "ncfa_xcorr_search_batched")
                self.launches += 2
        return best_j[:n_w], best_c[:n_w]

    # ------------------------------------------------------------------ xcorr.py: intro alignment
    def align_envelope(self, audio: np.ndarray, sr: int, target_sr: int, hop: int) -> torch.Tensor:
        """librosa.resample(sr → target_sr) then feature.rms(hop)[0].astype(float64), on the device.
        Only power-of-two decimations are supported (the reference calls it with 22050 → 11025)."""
        ratio = sr // target_sr if target_sr > 0 else 0
        if target_sr * ratio != sr or ratio < 1 or (ratio & (ratio - 1)) != 0:
            raise ValueError(f"align_envelope supports sr = target_sr·2^k only (got {sr} → {target_sr})")
        cur = self.to_dev(audio if len(audio) else np.zeros(1, np.float32))
        n = len(audio)
        with torch.cuda.device(self.device):
            st = self._stream()
            while ratio > 1:
                n_out = (n + 1) // 2
                nxt = torch.empty(max(n_out, 1), dtype=torch.float32, device=self.device)
                check(lib.ncfa_decimate2(_ptr(cur), n, _ptr(nxt), st), "ncfa_decimate2")
                self.launches += 1
                cur, n, ratio = nxt, n_out, ratio // 2
            rms = self.rms_frames_dev(cur, n, 2048, hop)
            out = torch.empty(rms.numel(), dtype=torch.float64, device=self.device)
            check(lib.ncfa_f32_to_f64(_ptr(rms), rms.numel(), _ptr(out), st), "ncfa_f32_to_f64")
            self.launches += 1
        return out

    def align_search(self, src_env: torch.Tensor, nc_env: torch.Tensor, n_str: np.ndarray, n_lag: np.ndarray):
        """30-speed envelope correlation of xcorr.find_content_offset → (peak_idx int32, score float64) on the host."""
        n_sp = len(n_str)
        live = n_lag > 0
        max_str = int(n_str[live].max())
        max_lag = int(n_lag[live].max())
        pk = torch.empty(n_sp, dtype=torch.int32, device=self.device)
        sc = torch.empty(n_sp, dtype=torch.float64, device=self.device)
        d_ns, d_nl = self.to_dev(n_str.astype(np.int32)), self.to_dev(n_lag.astype(np.int32))
        with torch.cuda.device(self.device):
            need = lib.ncfa_align_workspace_bytes(n_sp, max_str, max_lag)
            ws = self.workspace("align", need)
            check(lib.ncfa_align_search(_ptr(src_env), int(src_env.numel()), _ptr(nc_env), int(nc_env.numel()), _ptr(d_ns),
                                        _ptr(d_nl), n_sp, max_str, max_lag, _ptr(pk), _ptr(sc), _ptr(ws), ws.numel(),
                                        self._stream()),
                  "ncfa_align_search")
        self.launches += 3
        return self.to_host(pk), self.to_host(sc)

    # ------------------------------------------------------------------ spectral.py: whole-file STFT statistics
    def spectral_stats_dev(self, audio: torch.Tensor, seg_off: np.ndarray, seg_len: np.ndarray, sr: int):
        """→ (stats float64 [n_seg, 16], bin_db_mean float32 [n_seg, 1025]) on the device (layout: include/ncfa.h)."""
        n_seg = len(seg_len)
        stats = torch.zeros((max(n_seg, 1), 16), dtype=torch.float64, device=self.device)
        bins = torch.zeros((max(n_seg, 1), 1025), dtype=torch.float32, device=self.device)
        if n_seg == 0:
            return stats[:0], bins[:0]
        d_off, d_len = self.to_dev(seg_off.astype(np.int64)), self.to_dev(seg_len.astype(np.int32))
        with torch.cuda.device(self.device):
            ws = self.workspace("spectral", lib.ncfa_spectral_workspace_bytes(n_seg))
            check(lib.ncfa_spectral_stats_batched(_ptr(audio), _ptr(d_off), _ptr(d_len), n_seg, int(sr), _ptr(stats),
                                                  _ptr(bins), _ptr(ws), ws.numel(), self._stream()),
                  "ncfa_spectral_stats_batched")
        self.launches += 4
        return stats[:n_seg], bins[:n_seg]

    # ------------------------------------------------------------------ host conveniences
    def onset_strength(self, arrays: Sequence[np.ndarray], hop: int, sr: int) -> List[np.ndarray]:
        audio, off, ln = self.pack(arrays)
        onset, env_off, env_len, _, _ = self.onset_strength_dev(audio, off, ln, hop, sr)
        h = onset.cpu().numpy()
        return [h[o : o + n].copy() for o, n in zip(env_off, env_len)]

    def tempo_lags(self, envelopes: Sequence[np.ndarray], start_bpm: Sequence[float], hop: int, sr: int) -> np.ndarray:
        """feature.tempo's argmax lag for given onset envelopes (kernel-level parity entry)."""
        onset, off, ln = self.pack(envelopes)
        d_off, d_len = self.to_dev(off), self.to_dev(ln)
        d_bpm = self.to_dev(np.asarray(start_bpm, dtype=np.float64))
        return self.tempo_lag_dev(onset, d_off, d_len, ln, hop, sr, d_bpm).cpu().numpy()

    def beat_frames(self, envelopes: Sequence[np.ndarray], lags: Sequence[int], hop: int, sr: int) -> List[np.ndarray]:
        """beat_track's DP for given onset envelopes and lags (kernel-level parity entry)."""
        onset, off, ln = self.pack(envelopes)
        d_off, d_len = self.to_dev(off), self.to_dev(ln)
        d_lag = self.to_dev(np.asarray(lags, dtype=np.int32))
        beats, n_beats = self.beat_track_dev(onset, d_off, d_len, ln, d_lag, hop, sr)
        hb, hn = beats.cpu().numpy(), n_beats.cpu().numpy()
        if (hn < 0).any():
            raise _native.NcfaError("beat buffer overflow")
        return [hb[i, : hn[i]].copy() for i in range(len(envelopes))]

    def tempo_and_beats(self, arrays: Sequence[np.ndarray], start_bpm: Sequence[float], hop: int, sr: int,
                        want_beats: bool = True):
        """onset → tempo → beat DP for each array → (lags int32[n], list of beat-frame arrays | counts)."""
        audio, off, ln = self.pack(arrays)
        _, _, _, lag, beats, n_beats = self.tempo_segments_dev(audio, off, ln, np.asarray(start_bpm, np.float64), hop, sr)
        hl, hn = lag.cpu().numpy(), n_beats.cpu().numpy()
        if (hn < 0).any():
            raise _native.NcfaError("beat buffer overflow")
        if not want_beats:
            return hl, hn
        hb = beats.cpu().numpy()
        return hl, [hb[i, : hn[i]].copy() for i in range(len(arrays))]


_ENGINES: dict = {}          # (device index, thread ident) -> (Engine, weakref to the owning thread)
_ENG_LOCK = threading.Lock()
_RETIRED_LAUNCHES = 0        # launches of engines whose threads have ended (total_launches stays monotonic)


def _drop_dead_engines() -> None:
    """Engines belong to host threads (each pins a parameter ring and owns device workspaces).  A thread that has ended
    must not keep them alive — nor hand them, through a recycled thread ident, to an unrelated new thread."""
    global _RETIRED_LAUNCHES
    for key in [k for k, (_, ref) in _ENGINES.items() if ref() is None or not ref().is_alive()]:
        eng, _ = _ENGINES.pop(key)
        _RETIRED_LAUNCHES += eng.launches


def get_engine(device=None) -> Engine:
    """The calling thread's engine for `device` (workspaces are per engine, so concurrent host threads — each on its own
    CUDA stream — never share scratch buffers).  Engines of threads that have ended are released on the next call."""
    if not torch.cuda.is_available():
        raise _native.NcfaError("nightcore_analyzer needs a CUDA device (sm_100a); there is no CPU fallback")
    idx = torch.cuda.current_device() if device is None else torch.device(device).index or 0
    me = threading.current_thread()
    key = (idx, me.ident)
    with _ENG_LOCK:
        hit = _ENGINES.get(key)
        if hit is not None and hit[1]() is me:
            return hit[0]
        _drop_dead_engines()
        eng = Engine(torch.device("cuda", idx))
        _ENGINES[key] = (eng, weakref.ref(me))
        return eng


def total_launches() -> int:
    """Kernels launched by every engine of this process (bench.py's gpu_launches)."""
    with _ENG_LOCK:
        return _RETIRED_LAUNCHES + sum(e.launches for e, _ in _ENGINES.values())
