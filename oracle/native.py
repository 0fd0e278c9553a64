"""ctypes loader for oracle/csrc/oracle_native.c (TEST INFRASTRUCTURE — see oracle/__init__.py)."""
from __future__ import annotations

import ctypes
import os
import subprocess
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "csrc", "oracle_native.c")
_OUT_DIR = os.path.join(_HERE, "_build")
_SO = os.path.join(_OUT_DIR, "liboracle_native.so")
_lib = None


def build(force: bool = False) -> str:
    os.makedirs(_OUT_DIR, exist_ok=True)
    if force or not os.path.exists(_SO) or (
        os.path.exists(_SRC) and os.path.getmtime(_SO) < os.path.getmtime(_SRC)
    ):
        tmp = _SO + f".tmp{os.getpid()}"
        subprocess.check_call(
            ["gcc", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-o", tmp, _SRC, "-lm"]
        )
        os.replace(tmp, _SO)
    return _SO


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
        dp = ctypes.POINTER(ctypes.c_double)
        ip = ctypes.POINTER(ctypes.c_int64)
        _lib.orc_local_score.argtypes = [dp, ctypes.c_int64, dp, ctypes.c_int64, dp]
        _lib.orc_beat_dp.argtypes = [dp, ctypes.c_int64, ctypes.c_double, ctypes.c_double, ip, dp]
        _lib.orc_beat_dp_pen.argtypes = [dp, ctypes.c_int64, ctypes.c_double, ctypes.c_double, dp, ip, dp, dp]
        _lib.orc_bootstrap.argtypes = [dp, ctypes.c_int, dp, ctypes.c_int, ctypes.c_int] + [ctypes.c_uint64] * 4 + [
            dp, ctypes.POINTER(ctypes.c_int32)]
        _lib.orc_pcg64_raw.argtypes = [ctypes.c_uint64] * 4 + [ctypes.c_int, ctypes.POINTER(ctypes.c_uint64)]
        for f in (_lib.orc_local_score, _lib.orc_beat_dp, _lib.orc_beat_dp_pen, _lib.orc_bootstrap, _lib.orc_pcg64_raw):
            f.restype = None
    return _lib


def _dp(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))


def local_score(onset_norm: np.ndarray, window: np.ndarray, K: int) -> np.ndarray:
    onset_norm = np.ascontiguousarray(onset_norm, dtype=np.float64)
    window = np.ascontiguousarray(window, dtype=np.float64)
    out = np.empty(len(onset_norm), dtype=np.float64)
    lib().orc_local_score(_dp(onset_norm), len(onset_norm), _dp(window), int(K), _dp(out))
    return out


def beat_dp(localscore: np.ndarray, fpb: float, tightness: float):
    localscore = np.ascontiguousarray(localscore, dtype=np.float64)
    n = len(localscore)
    backlink = np.empty(n, dtype=np.int64)
    cumscore = np.empty(n, dtype=np.float64)
    lib().orc_beat_dp(_dp(localscore), n, float(fpb), float(tightness),
                      backlink.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), _dp(cumscore))
    return backlink, cumscore


def beat_dp_pen(localscore: np.ndarray, fpb: float, tightness: float, pen=None):
    """beat_dp with the transition penalty read from pen[d − near], d = near .. far (None: librosa's log form)
    → (backlink, cumscore, margin): margin[i] = (best − second best) / max(|best|, |second|) over frame i's candidate
    predecessors, +inf with fewer than two, 0 on an exact tie."""
    localscore = np.ascontiguousarray(localscore, dtype=np.float64)
    n = len(localscore)
    backlink = np.empty(n, dtype=np.int64)
    cumscore = np.empty(n, dtype=np.float64)
    margin = np.empty(n, dtype=np.float64)
    if pen is not None:
        near, far = int(np.round(fpb / 2.0)), int(2.0 * fpb)
        pen = np.ascontiguousarray(pen, dtype=np.float64)
        assert len(pen) == far - near + 1, (len(pen), near, far)
    lib().orc_beat_dp_pen(_dp(localscore), n, float(fpb), float(tightness), None if pen is None else _dp(pen),
                          backlink.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), _dp(cumscore), _dp(margin))
    return backlink, cumscore, margin


def pcg64_state(seed: int):
    """(state_hi, state_lo, inc_hi, inc_lo) of numpy's PCG64(seed) (SeedSequence hashing is numpy's)."""
    st = np.random.PCG64(seed).state["state"]
    s, i = int(st["state"]), int(st["inc"])
    m = (1 << 64) - 1
    return (s >> 64) & m, s & m, (i >> 64) & m, i & m


def bootstrap(a: np.ndarray, b, n_boot: int, seed: int, return_indices: bool = False):
    """boot[i] = median(choice(a)) / median(choice(b)), a drawn first — PCG64(seed)-exact."""
    a = np.ascontiguousarray(a, dtype=np.float64)
    nb = 0 if b is None else len(b)
    bb = np.zeros(1) if b is None else np.ascontiguousarray(b, dtype=np.float64)
    boot = np.empty(n_boot, dtype=np.float64)
    idx = np.empty(n_boot * (len(a) + nb), dtype=np.int32) if return_indices else None
    lib().orc_bootstrap(_dp(a), len(a), _dp(bb), nb, int(n_boot), *pcg64_state(seed), _dp(boot),
                        idx.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)) if idx is not None else None)
    return (boot, idx) if return_indices else boot


def pcg64_raw(seed: int, n: int) -> np.ndarray:
    out = np.empty(n, dtype=np.uint64)
    lib().orc_pcg64_raw(*pcg64_state(seed), n, out.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)))
    return out
