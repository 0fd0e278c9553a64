"""numpy restatement of the two searches of xcorr.cu as include/ncfa.h states them: ncfa_xcorr_search_batched (the
waveform speed search) and ncfa_align_search (the intro alignment).

Every dtype is named: no value here goes through numpy's scalar-promotion rules, which changed in numpy 2 (NEP 50).
That is why the speed search is not `pipeline_port.speed_xcorr_arrays`: there `np.dot(wa, wb) / (norm_a * norm_b)` is
a float32 divided by a Python float, which numpy 2 rounds to float32 and numpy 1 (the reference's pin) computes in
float64.  The kernel and `search` below follow the float64 form.  The two can pick different candidates only when two
candidates tie in float32.

Sums are float64.  On integer-valued inputs whose sums stay below 2**24 every partial sum is exact, in float32 and in
float64, in any order, so the GPU must then match these functions bit for bit, ties included."""
from __future__ import annotations

import numpy as np

NORM_GATE = np.float64(1e-10)       # the ‖wa‖ and ‖wb‖ gates (xcorr.py:127, 135)
SCORE_GATE = np.float64(1e-12)      # the alignment score's denominator (xcorr.py:250)
_CHUNK = 1 << 23                    # samples gathered at once


def candidate_c(a, b, a_pos, b_lo, n_cand, win: int, stride: int, rms_gate: float) -> np.ndarray:
    """c of every candidate → float64 [n_windows, max(n_cand)], −inf where the RMS gate or the ‖wa‖ gate drops the
    window, where the ‖wb‖ gate drops the candidate, and for j >= n_cand[w].

    Window w is a[a_pos[w] : a_pos[w] + win]; its candidate j is b[b_lo[w] + j·stride : … + win].
      na2, nb2, dot   float64 sums
      rms_a           float32(sqrt(na2 / win))
      norm_a, norm_b  float32(sqrt(na2)), float32(sqrt(nb2))
      c               float64(float32(dot)) / (float64(norm_a) · float64(norm_b))
    The window is kept unless float64(rms_a) < rms_gate or float64(norm_a) < 1e-10; the candidate unless
    float64(norm_b) < 1e-10."""
    a64 = np.asarray(a, dtype=np.float32).astype(np.float64)
    b64 = np.asarray(b, dtype=np.float32).astype(np.float64)
    a_pos = np.asarray(a_pos, dtype=np.int64)
    b_lo = np.asarray(b_lo, dtype=np.int64)
    n_cand = np.asarray(n_cand, dtype=np.int64)
    n_w = len(a_pos)
    max_cand = int(n_cand.max(initial=0))
    out = np.full((n_w, max_cand), -np.inf, dtype=np.float64)
    if n_w == 0 or max_cand == 0:
        return out
    av = np.lib.stride_tricks.sliding_window_view(a64, win)
    bv = np.lib.stride_tricks.sliding_window_view(b64, win)
    j = np.arange(max_cand, dtype=np.int64)
    step = max(1, _CHUNK // (win * (max_cand + 1)))
    for s in range(0, n_w, step):
        e = min(n_w, s + step)
        live = j[None, :] < n_cand[s:e, None]
        rows = np.where(live, b_lo[s:e, None] + j[None, :] * np.int64(stride), np.int64(0))
        rows = np.clip(rows, 0, len(bv) - 1)           # the rows of dead candidates are never used
        wa = av[a_pos[s:e]]                             # [k, win]
        wb = bv[rows]                                   # [k, max_cand, win]
        na2 = np.sum(wa * wa, axis=1, dtype=np.float64)
        nb2 = np.sum(wb * wb, axis=2, dtype=np.float64)
        dot = np.sum(wa[:, None, :] * wb, axis=2, dtype=np.float64)
        rms_a = np.sqrt(na2 / np.float64(win)).astype(np.float32)
        norm_a = np.sqrt(na2).astype(np.float32).astype(np.float64)
        norm_b = np.sqrt(nb2).astype(np.float32).astype(np.float64)
        keep_w = ~(rms_a.astype(np.float64) < np.float64(rms_gate)) & ~(norm_a < NORM_GATE)
        keep = live & keep_w[:, None] & ~(norm_b < NORM_GATE)
        with np.errstate(divide="ignore", invalid="ignore"):
            c = dot.astype(np.float32).astype(np.float64) / (norm_a[:, None] * norm_b)
        out[s:e] = np.where(keep & ~np.isnan(c), c, np.float64(-np.inf))
    return out


def first_max(c: np.ndarray):
    """The first strict maximum of each row, kept when it is > 0 → (best_j int32, best_c float64); (−1, 0.0)
    otherwise."""
    n_w = c.shape[0]
    if c.shape[1] == 0:
        return np.full(n_w, -1, dtype=np.int32), np.zeros(n_w, dtype=np.float64)
    j = np.argmax(c, axis=1)
    best = c[np.arange(n_w), j]
    keep = best > np.float64(0.0)
    return np.where(keep, j, -1).astype(np.int32), np.where(keep, best, np.float64(0.0)).astype(np.float64)


def search(a, b, a_pos, b_lo, n_cand, win: int, stride: int, rms_gate: float):
    """ncfa_xcorr_search_batched → (best_j int32 [n_windows], best_c float64 [n_windows])."""
    return first_max(candidate_c(a, b, a_pos, b_lo, n_cand, win, stride, rms_gate))


def stretch(nc_env, n_stretched: int) -> np.ndarray:
    """np.interp(np.linspace(0, 1, n_stretched), np.linspace(0, 1, len(nc_env)), nc_env) (xcorr.py:228)."""
    nc = np.asarray(nc_env, dtype=np.float64)
    return np.interp(np.linspace(np.float64(0.0), np.float64(1.0), int(n_stretched), dtype=np.float64),
                     np.linspace(np.float64(0.0), np.float64(1.0), len(nc), dtype=np.float64), nc)


def align(src_env, nc_env, n_stretched, n_lags):
    """ncfa_align_search → (peak_idx int32 [n_speeds], score float64 [n_speeds], stretched: list of float64 arrays,
    None for a skipped speed).

    Per speed s with n_lags[s] > 0: stretched = stretch(nc_env, n_stretched[s]);
    corr = np.correlate(src_env, stretched, 'valid')[:n_lags[s]]; peak = the first argmax;
    score = corr[peak] / sqrt(Σ src_env[peak : peak + n]² · Σ stretched²), 0 when that denominator is <= 1e-12.
    A speed with n_lags[s] <= 0 gives (−1, 0.0) whatever its n_stretched."""
    src = np.asarray(src_env, dtype=np.float64)
    n_sp = len(n_lags)
    peak = np.full(n_sp, -1, dtype=np.int32)
    score = np.zeros(n_sp, dtype=np.float64)
    rows = []
    for s in range(n_sp):
        n_lag = int(n_lags[s])
        if n_lag <= 0:
            rows.append(None)
            continue
        st = stretch(nc_env, int(n_stretched[s]))
        n = len(st)
        corr = np.correlate(src[: n_lag + n - 1], st, mode="valid")     # = np.correlate(src, st, 'valid')[:n_lag]
        pk = int(np.argmax(corr))
        denom = np.sqrt(np.float64(np.sum(src[pk : pk + n] ** 2, dtype=np.float64)) *
                        np.float64(np.sum(st ** 2, dtype=np.float64)))
        peak[s] = pk
        score[s] = corr[pk] / denom if denom > SCORE_GATE else np.float64(0.0)
        rows.append(st)
    return peak, score, rows
