"""numpy float64 restatement of ncfa_render_batched (include/ncfa.h): the band-limited speed change of one segment.

The table comes from the library (ncfa_host_render_table) and is passed in.  Every operation below is the one the
kernel performs, in the same order, with one vectorised pass per tap k, so the result must match the GPU bit for bit.
"""
from __future__ import annotations

import math

import numpy as np

ZEROS = 32
PHASES = 512
BETA = 10.0
ROLLOFF = 0.95


def out_len(n: int, ratio: float) -> int:
    return math.floor((n - 1) / ratio) + 1 if n > 0 else 0


def table_formula() -> np.ndarray:
    """T[j] = sinc(j/L)·I0(β·sqrt(1 − (j/(Z·L))²))/I0(β), j < Z·L, and T[Z·L] = 0 (numpy's sinc and i0)."""
    zl = ZEROS * PHASES
    j = np.arange(zl, dtype=np.float64)
    t = np.sinc(j / PHASES) * np.i0(BETA * np.sqrt(1.0 - (j / zl) ** 2)) / np.i0(BETA)
    return np.append(t, 0.0)


def render(x: np.ndarray, ratio: float, table: np.ndarray, m=None) -> np.ndarray:
    """Outputs m (default: all floor((n − 1)/ratio) + 1 of them) of segment x played `ratio` times faster."""
    x = np.asarray(x, dtype=np.float32).astype(np.float64)
    n = len(x)
    R = float(ratio)
    c = ROLLOFF / max(1.0, R)
    half = ZEROS / c
    m = np.arange(out_len(n, R), dtype=np.int64) if m is None else np.asarray(m, dtype=np.int64)
    t = m.astype(np.float64) * R
    n0 = np.floor(t - half) + 1.0
    acc = np.zeros(len(m))
    zl = ZEROS * PHASES
    for k in range(math.ceil(2.0 * half) + 1):
        nk = n0 + k
        d = (np.abs(t - nk) * c) * PHASES
        i = np.floor(d)
        f = d - i
        ok = (i < zl) & (nk >= 0) & (nk < n)
        ii = np.where(ok, i, 0).astype(np.int64)
        xv = x[np.where(ok, nk, 0).astype(np.int64)]
        term = (table[ii] + f * (table[ii + 1] - table[ii])) * xv
        acc = np.where(ok, acc + term, acc)
    return (acc * c).astype(np.float32)
