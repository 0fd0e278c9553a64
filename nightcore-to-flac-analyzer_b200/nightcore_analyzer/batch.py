"""
Batched analysis of many (nightcore, source) track pairs on one GPU — the data-parallel form of
``pipeline.run`` (pipeline.py:81-216).  Stage order and every per-pair decision follow the
reference; only the loop structure differs: each stage runs once over all pairs of the batch.

  stage 0  upload: all tracks of the batch in one HBM buffer (pinned staging → one H2D copy)
  stage 1  strip_silence bounds          (framed RMS kernel; pipeline.py:91-104)
  stage 2  window energies + gate        (float64 reduction; pipeline.py:127-146)
  stage 3  pitch: chroma shift per chunk (pipeline.py:149-159)            [when compute_pitch]
  stage 4  source windows → tempo        (pipeline.py:169)
  stage 5  prior = median(src)·dur ratio (host scalar per pair; pipeline.py:174-178)
  stage 6  nightcore windows → tempo     (pipeline.py:186)
  stage 7  hop-64 whole-track beat pass  (pipeline.py:204-205)
  stage 8  bootstraps: tempo, pitch, IBI (consensus.py:243-312) — three batched launches
  stage 9  host: AnalysisResult per pair (classification, warnings, rubberband strings)

Pairs are independent; a failing pair (all windows gated away, too few tempo windows) yields its
exception object in the result list and does not disturb the others.
"""
from __future__ import annotations

import os
import queue
import sys
import threading
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import _engine, consensus, tempo as _tempo
from .io import ENERGY_GATE_DB, HOP_SEC, SAMPLE_RATE, SILENCE_STRIP_DB, WINDOW_SEC, _db_from_meansq


@dataclass
class StagedBatch:
    """Tracks of a batch resident in HBM.  Track 2i is pair i's nightcore, 2i+1 its source."""
    audio: torch.Tensor          # float32, all tracks, 4-sample aligned starts
    off: np.ndarray              # int64 [2P] sample offset of each track
    length: np.ndarray           # int64 [2P] samples
    sr: int
    h2d_bytes: int

    @property
    def n_pairs(self) -> int:
        return len(self.off) // 2


@dataclass
class PinnedBatch:
    """Tracks of a batch laid out in pinned host memory, ready for one H2D copy."""
    pinned: torch.Tensor         # float32, pinned
    off: np.ndarray              # int64 [2P]
    length: np.ndarray           # int64 [2P]
    sr: int

    @property
    def n_pairs(self) -> int:
        return len(self.off) // 2


def pin_pairs(pairs: Sequence[Tuple[np.ndarray, np.ndarray]], sr: int = SAMPLE_RATE,
              pinned: Optional[torch.Tensor] = None) -> PinnedBatch:
    """Lay [(nc_audio, src_audio), ...] out in one pinned host buffer (4-sample aligned track starts)."""
    tracks = [np.asarray(t, dtype=np.float32) for p in pairs for t in p]
    length = np.array([len(t) for t in tracks], dtype=np.int64)
    off, total = _engine.aligned_layout(length)
    if pinned is None or pinned.numel() < max(total, 4):
        pinned = torch.empty(max(total, 4), dtype=torch.float32, pin_memory=True)
    dst = pinned.numpy()
    list(_stage_pool().map(lambda a: np.copyto(dst[a[1] : a[1] + len(a[0])], a[0]), zip(tracks, off.tolist())))
    return PinnedBatch(pinned=pinned, off=off, length=length, sr=sr)


def upload(pb: PinnedBatch, n_pairs: Optional[int] = None, out: Optional[torch.Tensor] = None,
           start_pair: int = 0) -> StagedBatch:
    """One asynchronous H2D copy of pairs ``[start_pair, start_pair + n_pairs)`` of a pinned batch (into ``out`` when
    given: a preallocated device buffer avoids allocator traffic — and its implicit synchronisations — in a streaming
    loop).  Offsets of the returned batch are relative to its own buffer."""
    eng = _engine.get_engine()
    s = int(start_pair)
    if s < 0 or s > pb.n_pairs:
        raise ValueError(f"start_pair {s} outside the pinned batch of {pb.n_pairs} pairs")
    k = pb.n_pairs - s if n_pairs is None else int(n_pairs)
    if k < 0 or s + k > pb.n_pairs:
        raise ValueError(f"pairs [{s}, {s + k}) outside the pinned batch of {pb.n_pairs} pairs")
    off, length = pb.off[2 * s : 2 * (s + k)], pb.length[2 * s : 2 * (s + k)]
    base = int(off[0]) if k else 0
    total = _engine.aligned_layout(length)[1]
    n = max(total, 4)
    src = pb.pinned[base : base + n] if base + n <= pb.pinned.numel() else pb.pinned[base:]
    if out is not None and out.numel() >= n:
        audio = out[: src.numel()]
        audio.copy_(src, non_blocking=True)
    else:
        audio = src.to(eng.device, non_blocking=True)
    eng.h2d_bytes += 4 * total
    return StagedBatch(audio=audio, off=off - base, length=length.copy(), sr=pb.sr, h2d_bytes=4 * total)


def stage_pairs(pairs: Sequence[Tuple[np.ndarray, np.ndarray]], sr: int = SAMPLE_RATE,
                pinned: Optional[torch.Tensor] = None) -> StagedBatch:
    """Copy [(nc_audio, src_audio), ...] into one device buffer (through pinned host memory)."""
    return upload(pin_pairs(pairs, sr, pinned))


def _window_starts(n: int, win_n: int, hop_n: int) -> np.ndarray:
    """io.py:94-110: starts while start + win_n <= n."""
    if win_n <= 0 or n < win_n:
        return np.zeros(0, dtype=np.int64)
    return np.arange(0, n - win_n + 1, max(hop_n, 1), dtype=np.int64) if hop_n > 0 else np.zeros(0, dtype=np.int64)


def analyse_staged(batch: StagedBatch, *, window_sec: float = WINDOW_SEC, hop_sec: float = HOP_SEC,
                   energy_gate_db: float = ENERGY_GATE_DB, silence_strip_db: Optional[float] = SILENCE_STRIP_DB,
                   compute_pitch: bool = True, compute_ibi: bool = True, stats: Optional[dict] = None,
                   ) -> List[Union[consensus.AnalysisResult, Exception]]:
    eng = _engine.get_engine()
    d2h0 = eng.d2h_bytes
    sr = batch.sr
    P = batch.n_pairs
    n_tracks = 2 * P
    t_off = batch.off.copy()
    t_len = batch.length.copy()
    failures: List[Optional[Exception]] = [None] * P

    # ---- stage 1: strip_silence (io.py:58-79) — bounds only; the samples never move
    if silence_strip_db is not None and n_tracks:
        bounds = eng.to_host(eng.trim_bounds_dev(batch.audio, t_off, t_len.astype(np.int32), silence_strip_db))
        t_off = t_off + bounds[:, 0]
        t_len = bounds[:, 1] - bounds[:, 0]

    # ---- stage 2: windows, float64 energies, gate (io.py:82-126)
    win_n, hop_n = int(window_sec * sr), int(hop_sec * sr)
    # io.py:94-110 for every track at once: starts 0, hop_n, … while start + win_n <= n  (same values as _window_starts)
    if win_n > 0 and hop_n > 0 and n_tracks:
        tl = t_len.astype(np.int64)
        n_w = np.where(tl >= win_n, (tl - win_n) // hop_n + 1, 0)
        seg_track = np.repeat(np.arange(n_tracks, dtype=np.int64), n_w)
        within = np.arange(int(n_w.sum()), dtype=np.int64) - np.repeat(np.cumsum(n_w) - n_w, n_w)
        seg_off = t_off.astype(np.int64)[seg_track] + within * hop_n
    else:
        seg_track, seg_off = np.zeros(0, np.int64), np.zeros(0, np.int64)
    seg_len = np.full(len(seg_off), win_n, dtype=np.int32)
    if len(seg_off):
        ms = eng.window_energy_dev(batch.audio, eng.to_dev(seg_off), eng.to_dev(seg_len)).cpu().numpy()
        energy_db = 20.0 * np.log10(np.maximum(np.sqrt(ms), 1e-10))        # io.py:38-40, vectorised
    else:
        energy_db = np.zeros(0)
    cnt = np.bincount(seg_track, minlength=n_tracks) if len(seg_track) else np.zeros(n_tracks, np.int64)
    first = np.concatenate([[0], np.cumsum(cnt)[:-1]]) if n_tracks else np.zeros(0, np.int64)
    peak = np.full(n_tracks, -np.inf)
    has = cnt > 0
    if has.any():
        peak[has] = np.maximum.reduceat(energy_db, first[has])
    keep = energy_db >= peak[seg_track] + energy_gate_db if len(seg_track) else np.zeros(0, dtype=bool)
    n_win_kept = np.bincount(seg_track[keep], minlength=n_tracks) if len(seg_track) else np.zeros(n_tracks, np.int64)
    for i in range(P):
        if n_win_kept[2 * i] == 0 or n_win_kept[2 * i + 1] == 0:
            failures[i] = RuntimeError(
                "All windows were discarded by the energy gate.  "
                "Try raising --energy-gate (e.g. --energy-gate -60)."
            )
    alive = np.array([failures[i] is None for i in range(P)], dtype=bool)

    # ---- stage 3: pitch (pitch.py:100-173), one batched pass over all chunk pairs
    src_hz: List[list] = [[] for _ in range(P)]
    nc_hz: List[list] = [[] for _ in range(P)]
    pitch_method: Optional[str] = None
    if compute_pitch:
        from . import pitch as _pitch
        pitch_method = "chroma_xcorr"
        jobs = [(i, t_off[2 * i + 1], t_len[2 * i + 1], t_off[2 * i], t_len[2 * i]) for i in range(P) if alive[i]]
        shifts = _pitch.chroma_shifts_staged(batch.audio, jobs, sr)
        for (i, *_), st in zip(jobs, shifts):
            src_hz[i], nc_hz[i] = _pitch.hz_lists(st)

    # ---- stage 4: source windows (120 BPM prior)
    def run_tempo(sel: np.ndarray, bpm: np.ndarray):
        if len(sel) == 0:
            return np.zeros(0, np.int32), np.zeros(0, np.int32)
        _, _, _, lag, _, n_beats = eng.tempo_segments_dev(batch.audio, seg_off[sel], seg_len[sel], bpm,
                                                          _tempo.HOP_LENGTH, sr)
        return eng.to_host(lag), _engine.check_beat_counts(eng.to_host(n_beats))

    is_src = (seg_track % 2) == 1
    pair_of = seg_track // 2
    sel_src = np.flatnonzero(keep & is_src & alive[pair_of])
    lag_s, nb_s = run_tempo(sel_src, np.full(len(sel_src), 120.0))
    def per_pair_tempos(sel, lag, nb):
        """tempo.py:51-77 for every window at once: both estimators equal bpms[lag] ⇒ that value when the window has
        >= MIN_BEATS beats and a positive lag, else None; split into one list per pair (window order preserved)."""
        out: List[list] = [[] for _ in range(P)]
        if len(sel) == 0:
            return out
        ok = (nb >= _tempo.MIN_BEATS) & (lag > 0)
        bpm = 60.0 * sr / (_tempo.HOP_LENGTH * np.where(ok, lag, 1).astype(np.float64))
        vals = [float(b) if o else None for b, o in zip(bpm.tolist(), ok.tolist())]
        owners = pair_of[sel]
        cuts = np.flatnonzero(np.diff(owners)) + 1
        starts = np.concatenate([[0], cuts])
        ends = np.concatenate([cuts, [len(sel)]])
        for a, b in zip(starts, ends):
            out[int(owners[a])] = vals[a:b]
        return out

    src_tempos = per_pair_tempos(sel_src, lag_s, nb_s)

    # ---- stage 5: per-pair prior (pipeline.py:171-178)
    nc_dur = t_len[0::2] / sr
    src_dur = t_len[1::2] / sr
    prior = np.full(P, 120.0)
    for i in range(P):
        valid = [t for t in src_tempos[i] if t is not None]
        if valid and nc_dur[i] > 0 and src_dur[i] > 0:
            prior[i] = consensus._median_small(valid) * (src_dur[i] / nc_dur[i])

    # ---- stage 6: nightcore windows with the pair's prior
    sel_nc = np.flatnonzero(keep & ~is_src & alive[pair_of])
    lag_n, nb_n = run_tempo(sel_nc, prior[pair_of[sel_nc]] if len(sel_nc) else np.zeros(0))
    nc_tempos = per_pair_tempos(sel_nc, lag_n, nb_n)

    # ---- stage 7: hop-64 whole-track pass (tempo.py:120-173) for every live pair
    ibis: List[Optional[Tuple[np.ndarray, np.ndarray]]] = [None] * P
    if compute_ibi and alive.any():
        tr = np.array([k for i in range(P) if alive[i] for k in (2 * i, 2 * i + 1)], dtype=np.int64)
        bpm = np.array([prior[k // 2] if k % 2 == 0 else 120.0 for k in tr])
        _, _, _, lag64, beats64, nb64 = eng.tempo_segments_dev(batch.audio, t_off[tr], t_len[tr].astype(np.int32), bpm,
                                                               _tempo.IBI_HOP_LENGTH, sr)
        hn = _engine.check_beat_counts(eng.to_host(nb64))
        mb = int(hn.max()) if len(hn) else 0
        hb = eng.to_host(beats64[:, : max(mb, 1)])
        per_track = {}
        for j, k in enumerate(tr):
            per_track[int(k)] = _tempo._ibis_from_beats(hb[j, : hn[j]], sr, _tempo.IBI_HOP_LENGTH, _tempo.IBI_MIN_IBIS)
        for i in range(P):
            if alive[i]:
                n_i, s_i = per_track[2 * i], per_track[2 * i + 1]
                if n_i is not None and len(n_i) >= 4 and s_i is not None and len(s_i) >= 4:
                    ibis[i] = (n_i, s_i)

    # ---- stage 8: bootstraps, batched per kind
    q_lo, q_hi = consensus._percentile_args(consensus.CI_LEVEL)
    valid_t = [(consensus._valid(src_tempos[i]), consensus._valid(nc_tempos[i])) for i in range(P)]
    valid_p = [(consensus._valid(src_hz[i]), consensus._valid(nc_hz[i])) for i in range(P)]
    for i in range(P):
        if alive[i] and (len(valid_t[i][0]) < consensus.MIN_VALID or len(valid_t[i][1]) < consensus.MIN_VALID):
            failures[i] = consensus._insufficient(*valid_t[i])
            alive[i] = False

    def boot(jobs):
        if not jobs:
            return np.zeros((0, 3))
        out, _, _ = eng.bootstrap(jobs, consensus.BOOTSTRAP_SEED, consensus.N_BOOTSTRAP, q_lo, q_hi)
        return out

    t_idx = [i for i in range(P) if alive[i]]
    t_out = boot([(valid_t[i][1], valid_t[i][0]) for i in t_idx])                 # nc first
    p_idx = [i for i in t_idx if len(valid_p[i][0]) >= consensus.MIN_VALID and len(valid_p[i][1]) >= consensus.MIN_VALID]
    p_out = boot([(valid_p[i][1], valid_p[i][0]) for i in p_idx])                 # nc first
    i_idx = [i for i in t_idx if ibis[i] is not None]
    i_out = boot([(ibis[i][1], ibis[i][0]) for i in i_idx])                       # src first

    # ---- stage 9: host assembly
    results: List[Union[consensus.AnalysisResult, Exception]] = [None] * P  # type: ignore[list-item]
    tmap = {i: t_out[j] for j, i in enumerate(t_idx)}
    pmap = {i: p_out[j] for j, i in enumerate(p_idx)}
    imap = {i: i_out[j] for j, i in enumerate(i_idx)}
    for i in range(P):
        if failures[i] is not None:
            results[i] = failures[i]
            continue
        ts = (float(tmap[i][0]), (float(tmap[i][1]), float(tmap[i][2])))
        if i in pmap:
            ps = (float(pmap[i][0]), (float(pmap[i][1]), float(pmap[i][2])))
            n_pitch = (len(valid_p[i][0]), len(valid_p[i][1]))
        else:
            ps, n_pitch = (1.0, (1.0, 1.0)), (0, 0)
        res = consensus._assemble(src_hz[i], nc_hz[i], src_tempos[i], nc_tempos[i], valid_t[i][0], valid_t[i][1], ps,
                                  ts, n_pitch, float(nc_dur[i]), float(src_dur[i]))
        res.intro_offset_sec = None
        res.pitch_method = pitch_method
        if i in imap:
            res.ibi_ratio = float(imap[i][0])
            res.ibi_ci = (float(imap[i][1]), float(imap[i][2]))
        results[i] = res
    if stats is not None:
        stats["windows"] = int(len(sel_src) + len(sel_nc))
        stats["windows_sliced"] = int(len(seg_off))
        stats["tracks"] = int(n_tracks)
        stats["d2h_bytes"] = int(eng.d2h_bytes - d2h0)
        stats["hop64_frames"] = int(sum(1 + int(t_len[k]) // 64 for k in range(n_tracks))) if compute_ibi else 0
    return results


def plan_subbatches(n_pairs: int, sub: int, workers: int = 2, first: int = 8, growth: float = 1.5) -> List[int]:
    """Sub-batch sizes for ``n_pairs`` pairs, at most ``sub`` each.  A job can start only when its upload is complete,
    and the upload of the next job runs while the current ones compute; the copy engine moves a pair about twice
    as fast as the kernels analyse one, so sizes grow geometrically (``first``, x ``growth``) until they reach
    ``sub``: every upload hides behind the compute of the jobs before it and only the first few pairs' copy is
    exposed.  The rest is split evenly (no short tail job); a remainder smaller than the job before it is folded into
    that job (a batch of 125 pairs becomes 8, 12, 18, 27, 60 — not one unstreamed pass)."""
    sizes: List[int] = []
    left = int(n_pairs)
    sub = max(1, int(sub))
    if 5 * first <= left <= 2 * sub and growth == 1.5:
        # A batch of one or two jobs' worth (a rank's share of a 1000-pair batch on 8 GPUs): when several ranks upload at
        # once the host feeds each GPU at ~37 GB/s instead of 55 and the call becomes upload bound — it then ends one job
        # after the last byte arrives, so the LAST job must be short as well as the first.  Up, then down
        # (measured on one GPU, 125 pairs: 12/24/40/29/20 → 878 pairs/s, 8/12/18/27/60 → 886, i.e. free when compute bound).
        shape = (0.10, 0.19, 0.32, 0.23, 0.16)
        sizes = [max(1, int(round(f * left))) for f in shape]
        sizes[2] += left - sum(sizes)
        if all(0 < k <= sub for k in sizes):
            return sizes
        sizes = []
    s = float(max(1, first))
    while left > 0 and int(s) < sub:
        k = min(int(s), left)
        if left - k < k:
            k = left
        sizes.append(k)
        left -= k
        s *= growth
    if left > 0:
        k = -(-left // sub)
        base, r = divmod(left, k)
        sizes += [base + 1] * r + [base] * (k - r)
    return sizes


# Size of the first streamed job.  Its upload is the only one nothing hides, so it should be small; but jobs of a few
# pairs are latency bound on the device (one CTA per envelope in the beat tracker, short grids), so it should not be tiny
# either.  Measured on B200, 1000 pairs (profiles/r2l): first = 8 → 1107 pairs/s end to end, 24 → 913, 48 → 891, 83 → 890.
FIRST_JOB_PAIRS = 8
JOB_GROWTH = 1.5             # growth factor of the streamed job sizes


# ------------------------------------------------------------------------------------------------ the batch scheduler
# One stager thread walks the jobs (consecutive, disjoint slices of the batch) in order: it lays a slice out in pinned
# memory when the caller's arrays are pageable, queues its host→HBM copy on a copy stream into one of `workers + 2`
# preallocated device slots and hands (StagedBatch, copy-done event) to whichever of the `workers` analysis threads is
# free.  Each analysis thread has its own CUDA stream and Engine (workspaces, pinned parameter ring), so while one waits
# for a small device→host read or assembles results the other keeps the GPU fed, and copies never sit in front of kernels.
SUB_BATCH_PAIRS = 125        # pairs analysed per device pass (3.6 GB of audio at 180 s + 144 s per pair)
INLINE_PAIRS = 8             # batches up to this size are analysed in the calling thread, in one pass


class _Slot:
    def __init__(self, device, n_floats: int, want_pinned: bool):
        self.dev = torch.empty(max(n_floats, 4), dtype=torch.float32, device=device)
        self.pinned = torch.empty(max(n_floats, 4), dtype=torch.float32, pin_memory=True) if want_pinned else None
        self.free = torch.cuda.Event()       # recorded by the analysis stream that last read `dev`


_SLOTS: dict = {}
_SCHED_LOCK = threading.Lock()
_STAGE_POOL = None


def _stage_pool():
    """Threads that copy pageable tracks into the pinned staging slot (np.copyto releases the GIL).  Unlike torch's
    copy_, whose parallelism follows OMP_NUM_THREADS (torchrun sets it to 1), the pool is ours.  Measured on the 16-core
    B200 box, 1000 pairs from pageable numpy arrays: 4 threads 751 pairs/s, 12 threads 858, torch copy_ with 16 OpenMP
    threads 842 (profiles/r2z_*)."""
    global _STAGE_POOL
    if _STAGE_POOL is None:
        import concurrent.futures as cf
        n = max(2, min(12, len(os.sched_getaffinity(0)) * 3 // 4))
        _STAGE_POOL = cf.ThreadPoolExecutor(max_workers=max(1, n), thread_name_prefix="ncfa-stage")
    return _STAGE_POOL


def _slots_for(device, n_slots: int, n_floats: int, want_pinned: bool) -> List[_Slot]:
    """Device (and, for pageable input, pinned staging) slots, cached across calls and grown on demand."""
    key = torch.device(device).index
    cur = _SLOTS.get(key, [])
    ok = (len(cur) >= n_slots and all(s.dev.numel() >= n_floats for s in cur[:n_slots]) and
          (not want_pinned or all(s.pinned is not None and s.pinned.numel() >= n_floats for s in cur[:n_slots])))
    if not ok:
        keep_pinned = want_pinned or any(s.pinned is not None for s in cur)
        size = max([n_floats] + [s.dev.numel() for s in cur])
        _SLOTS[key] = cur = []          # drop the old buffers before allocating the new ones
        cur += [_Slot(device, size, keep_pinned) for _ in range(n_slots)]
        _SLOTS[key] = cur
    return cur[:n_slots]


def release_buffers() -> None:
    """Free the cached device / pinned staging slots of the scheduler."""
    with _SCHED_LOCK:
        _SLOTS.clear()


def analyse_batch(source, sr: int = SAMPLE_RATE, *, sub_batch: int = SUB_BATCH_PAIRS, workers: int = 2,
                  sizes: Optional[Sequence[int]] = None, stats: Optional[dict] = None, **kwargs):
    """Analyse every pair of ``source`` — a ``PinnedBatch`` (pin_pairs) or a sequence of ``(nc_audio, src_audio)``
    numpy arrays — and return one AnalysisResult (or exception object) per pair, in order.  The batch is cut into
    consecutive sub-batches (``sizes``, default ``plan_subbatches``) that stream through HBM: staging (pageable →
    pinned, multi-threaded), host→device copy and analysis of different sub-batches overlap."""
    pinned_in = isinstance(source, PinnedBatch)
    if pinned_in:
        sr = source.sr
        P = source.n_pairs
        lengths = source.length
    else:
        tracks = [np.ascontiguousarray(t, dtype=np.float32) for p in source for t in p]
        P = len(tracks) // 2
        lengths = np.array([len(t) for t in tracks], dtype=np.int64)
    if P == 0:
        return []
    if sizes is None:
        sizes = [P] if P <= INLINE_PAIRS else plan_subbatches(P, sub_batch, workers, first=FIRST_JOB_PAIRS,
                                                              growth=JOB_GROWTH)
    sizes = [int(k) for k in sizes]
    if any(k <= 0 for k in sizes) or sum(sizes) != P:
        raise ValueError(f"sub-batch sizes {sizes} do not cover the {P} pairs of the batch exactly once")
    starts = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(int)

    if stats is not None:
        stats["sub_batches"] = list(sizes)
    if len(sizes) == 1:      # one pass in the calling thread
        st = upload(source) if pinned_in else stage_pairs(list(source), sr)
        s1: dict = {}
        res = analyse_staged(st, stats=s1, **kwargs)
        if stats is not None:
            s1["h2d_bytes"] = st.h2d_bytes
            for key, v in s1.items():
                stats[key] = stats.get(key, 0) + v
        return res

    eng = _engine.get_engine()
    device = eng.device
    main = torch.cuda.current_stream(device)
    nw = max(1, min(int(workers), len(sizes)))
    need = max(_engine.aligned_layout(lengths[2 * s : 2 * (s + k)])[1] for s, k in zip(starts, sizes))
    with _SCHED_LOCK:       # one scheduled batch per process at a time (the slots are shared)
        # device slots: one per worker + TWO ahead.  With one ahead the copy of job j+3 cannot start before job j ends, and
        # a worker that finishes early finds nothing uploaded: measured 1036 pairs/s with 3 slots, 1218 with 4, 1227 with 6
        # (profiles/r3a_e2e_slots.log; 3.6 GB of HBM per slot at 125 pairs)
        n_slots = nw + 2
        slots = _slots_for(device, n_slots, need, want_pinned=not pinned_in)
        free_q: "queue.Queue[_Slot]" = queue.Queue()
        for sl in slots:
            sl.free.record(main)
            free_q.put(sl)
        ready_q: "queue.Queue" = queue.Queue()
        copy_stream = _worker_stream(device, 100)
        copy_stream.wait_stream(main)
        out: list = [None] * len(sizes)
        errors: list = []
        copy_events: list = []   # (start, end, bytes) of every host→HBM copy, on the copy stream's clock

        def stager():
            try:
                torch.cuda.set_device(device)
                for j, (s, k) in enumerate(zip(starts, sizes)):
                    sl = free_q.get()
                    if errors:
                        break
                    ln = lengths[2 * s : 2 * (s + k)]
                    if pinned_in:
                        base = int(source.off[2 * s])
                        off = source.off[2 * s : 2 * (s + k)] - base
                        total = _engine.aligned_layout(ln)[1]
                        src = source.pinned[base : base + total]
                    else:
                        off, total = _engine.aligned_layout(ln)
                        dst = sl.pinned.numpy()       # pageable → pinned: one memcpy per track on a small thread pool
                        list(_stage_pool().map(lambda a: np.copyto(dst[a[1] : a[1] + len(a[0])], a[0]),
                                               zip(tracks[2 * s : 2 * (s + k)], off.tolist())))
                        src = sl.pinned[:total]
                    with torch.cuda.stream(copy_stream):
                        copy_stream.wait_event(sl.free)
                        ev0 = torch.cuda.Event(enable_timing=True)
                        ev0.record(copy_stream)
                        sl.dev[:total].copy_(src, non_blocking=True)
                        ev = torch.cuda.Event(enable_timing=True)
                        ev.record(copy_stream)
                    copy_events.append((ev0, ev, 4 * total))
                    ready_q.put((j, StagedBatch(audio=sl.dev[: max(total, 4)], off=off.copy(), length=ln.copy(), sr=sr,
                                                h2d_bytes=4 * total), ev, sl))
            except BaseException as e:  # noqa: BLE001
                errors.append(e)
            finally:
                for _ in range(nw):
                    ready_q.put(None)

        def worker(w: int):
            torch.cuda.set_device(device)
            stream = _worker_stream(device, w)
            stream.wait_stream(main)
            with torch.cuda.stream(stream):
                while True:
                    item = ready_q.get()
                    if item is None:
                        break
                    j, st, ev, sl = item
                    try:
                        stream.wait_event(ev)
                        s1: dict = {}
                        res = analyse_staged(st, stats=s1, **kwargs)
                        s1["h2d_bytes"] = st.h2d_bytes
                        out[j] = (res, s1)
                    except BaseException as e:  # noqa: BLE001
                        errors.append(e)
                    finally:
                        sl.free.record(stream)
                        free_q.put(sl)
                stream.synchronize()

        with _fast_gil_handoff():
            futs = [_worker_thread(device, 100).submit(stager)] + [_worker_thread(device, w).submit(worker, w) for w in range(nw)]
            for f in futs:
                f.result()
        for w in range(nw):
            main.wait_stream(_worker_stream(device, w))
    if errors:
        raise errors[0]
    if stats is not None and copy_events:
        copy_events[-1][1].synchronize()
        ms = sum(a.elapsed_time(b) for a, b, _ in copy_events)
        stats["h2d_copy_ms"] = stats.get("h2d_copy_ms", 0.0) + ms          # time the copy engine spent on the uploads
        stats["h2d_copy_gbs"] = sum(n for _, _, n in copy_events) / max(ms, 1e-9) / 1e6
    results: list = []
    for res, s1 in out:
        results += res
        if stats is not None:
            for key, v in s1.items():
                stats[key] = stats.get(key, 0) + v
    return results


class _fast_gil_handoff:
    """While several host threads feed one GPU, a thread that returns from a device wait must get the interpreter back
    quickly: with CPython's default 5 ms switch interval it can sit behind another worker's pure-Python loop for the
    whole interval while BOTH streams run dry (measured: 4-6 ms holes, 13 % of the step — profiles/micro/timeline.py).
    0.2 ms keeps the hand-off an order of magnitude shorter than the kernels it schedules."""

    def __enter__(self):
        self.old = sys.getswitchinterval()
        sys.setswitchinterval(min(self.old, 2e-4))

    def __exit__(self, *a):
        sys.setswitchinterval(self.old)


def stagger_sizes(n_pairs: int, sub: int, workers: int = 2) -> List[int]:
    """Sub-batch sizes for a batch that is already resident in HBM: ``sub`` pairs each, but the first job is a fraction
    of one so that the workers run out of phase — equal jobs started together reach their host-side phases (result
    read-back, bootstrap staging, assembly) at the same moment and leave the device idle."""
    n_pairs, sub, workers = int(n_pairs), max(1, int(sub)), max(1, int(workers))
    if workers < 2 or n_pairs <= sub:
        return [min(sub, n_pairs - s) for s in range(0, n_pairs, sub)]
    first = max(1, sub // workers)
    sizes = [first]
    left = n_pairs - first
    k = -(-left // sub)
    base, r = divmod(left, k)
    return sizes + [base + 1] * r + [base] * (k - r)


def run_batch_arrays(pairs, sr: int = SAMPLE_RATE, **kwargs):
    """[(nc_audio, src_audio), ...] or a PinnedBatch → [AnalysisResult | Exception, ...] (kwargs of analyse_batch)."""
    return analyse_batch(pairs, sr, **kwargs)


def run_subbatches(jobs: Sequence, fn, workers: int = 2) -> list:
    """Run ``fn(x)`` for every job on ``workers`` host threads, each with its own CUDA stream and engine, and return
    the results in job order (sub-batches that already live in HBM)."""
    eng = _engine.get_engine()
    device = eng.device
    main = torch.cuda.current_stream(device)
    workers = max(1, min(workers, len(jobs)))
    streams = [_worker_stream(device, w) for w in range(workers)]
    for st in streams:
        st.wait_stream(main)
    out: list = [None] * len(jobs)
    nxt = iter(range(len(jobs)))
    lock = threading.Lock()

    def work(w: int):
        torch.cuda.set_device(device)
        with torch.cuda.stream(streams[w]):
            while True:
                with lock:
                    i = next(nxt, None)
                if i is None:
                    break
                out[i] = fn(jobs[i])
            streams[w].synchronize()

    if workers == 1:
        work(0)
    else:
        # one persistent host thread per worker index: its engine (workspaces, pinned parameter ring) is built once
        with _fast_gil_handoff():
            for f in [_worker_thread(device, w).submit(work, w) for w in range(workers)]:
                f.result()
    for st in streams:
        main.wait_stream(st)
    return out


def analyse_resident(batches: Sequence[StagedBatch], stats: Optional[dict] = None, workers: int = 2, **kwargs):
    """Same analysis threads for sub-batches that already live in HBM."""
    def one(st):
        s1: dict = {}
        return analyse_staged(st, stats=s1, **kwargs), s1

    results: list = []
    for res, s1 in run_subbatches(list(batches), one, workers):
        results += res
        if stats is not None:
            for key, v in s1.items():
                stats[key] = stats.get(key, 0) + v
    return results


_WORKER_STREAMS: dict = {}
_WORKER_THREADS: dict = {}


def _worker_thread(device, w: int):
    import concurrent.futures as cf
    key = (torch.device(device).index, w)
    if key not in _WORKER_THREADS:
        _WORKER_THREADS[key] = cf.ThreadPoolExecutor(max_workers=1, thread_name_prefix=f"ncfa-worker{w}")
    return _WORKER_THREADS[key]


def _worker_stream(device, w: int) -> "torch.cuda.Stream":
    key = (torch.device(device).index, w)
    if key not in _WORKER_STREAMS:
        _WORKER_STREAMS[key] = torch.cuda.Stream(device=device)
    return _WORKER_STREAMS[key]
