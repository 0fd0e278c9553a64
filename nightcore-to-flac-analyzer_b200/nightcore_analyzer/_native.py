"""ctypes binding of libncfa.so — the C ABI declared in include/ncfa.h.

There is no CPU fallback: if the library is missing, importing this module raises.  Every call
returns an int status; ``check()`` turns a negative status into ``NcfaError`` with the
library's thread-local message.
"""
from __future__ import annotations

import ctypes
import os
import re
from ctypes import c_double, c_int, c_int32, c_int64, c_size_t, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libncfa.so")
HEADER_PATH = os.path.normpath(os.path.join(_HERE, "..", "..", "include", "ncfa.h"))


class NcfaError(RuntimeError):
    pass


if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python __graft_entry__.py` (nvcc, sm_100a). "
        "nightcore_analyzer has no CPU fallback."
    )

lib = ctypes.CDLL(LIB_PATH)

_P = c_void_p  # every device/host pointer is passed as an integer address

_SIGNATURES = {
    "ncfa_version": (c_int, []),
    "ncfa_last_error": (ctypes.c_char_p, []),
    "ncfa_init_tables": (c_int, [c_int]),
    "ncfa_param_upload": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p]),
    "ncfa_profile_enable": (None, [c_int]),
    "ncfa_profile_report": (c_int, [ctypes.c_char_p, c_size_t]),
    "ncfa_profile_timeline": (c_int, [ctypes.c_char_p, c_size_t]),
    "ncfa_window_energy": (c_int, [_P, _P, _P, c_int, _P, _P]),
    "ncfa_rms_frames": (c_int, [_P, c_int64, c_int, c_int, _P, _P]),
    "ncfa_trim_workspace_bytes": (c_size_t, [c_int, c_int]),
    "ncfa_trim_bounds_batched": (c_int, [_P, _P, _P, c_int, c_int, c_double, _P, _P, c_size_t, _P]),
    "ncfa_onset_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "ncfa_onset_strength_batched": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, _P, _P, _P, c_size_t, _P]),
    "ncfa_tempo_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "ncfa_tempo_lag_batched": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, _P, _P, _P, c_size_t, _P]),
    "ncfa_beat_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "ncfa_beat_track_batched": (c_int, [_P, _P, _P, c_int, c_int, _P, c_int, _P, c_int, _P, _P, c_size_t, _P]),
    "ncfa_bootstrap_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "ncfa_bootstrap_ratio_batched": (
        c_int,
        [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, ctypes.POINTER(c_uint64), c_double, c_double, _P, _P,
         _P, _P, c_size_t, _P],
    ),
    "ncfa_tuning_workspace_bytes": (c_size_t, [c_int, c_int]),
    "ncfa_tuning_estimate_batched": (c_int, [_P, _P, _P, c_int, c_int, c_int, _P, _P, c_size_t, _P]),
    "ncfa_chroma_workspace_bytes": (c_size_t, [c_int, c_int]),
    "ncfa_chroma_mean_batched": (c_int, [_P, _P, _P, c_int, c_int, c_int, _P, _P, _P, c_size_t, _P]),
    "ncfa_cyclic_xcorr_batched": (c_int, [_P, _P, c_int, c_int, _P, _P]),
    "ncfa_xcorr_workspace_bytes": (c_size_t, [c_int, c_int]),
    "ncfa_xcorr_search_batched": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_double, _P, _P, _P,
                                          c_size_t, _P]),
    "ncfa_decimate2": (c_int, [_P, c_int64, _P, _P]),
    "ncfa_f32_to_f64": (c_int, [_P, c_int64, _P, _P]),
    "ncfa_align_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "ncfa_align_search": (c_int, [_P, c_int, _P, c_int, _P, _P, c_int, c_int, c_int, _P, _P, _P, c_size_t, _P]),
    "ncfa_spectral_workspace_bytes": (c_size_t, [c_int]),
    "ncfa_spectral_stats_batched": (c_int, [_P, _P, _P, c_int, c_int, _P, _P, _P, c_size_t, _P]),
    "ncfa_render_out_len": (c_int64, [c_int32, c_double]),
    "ncfa_render_batched": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, _P, _P, _P]),
    "ncfa_host_render_table": (c_int, [_P]),
    "ncfa_host_cqt_matrix": (c_int, [c_int, c_int, _P]),
    "ncfa_host_halfband_taps": (c_int, [_P]),
    "ncfa_host_mel_lanes": (c_int, [c_int, _P, _P, _P]),
}


def declared_symbols() -> list[str]:
    """Function names declared in include/ncfa.h."""
    with open(HEADER_PATH) as f:
        text = f.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ncfa_[a-z0-9_]+)\s*\(", text)))


def check_symbols() -> list[str]:
    """Every symbol the header declares must be exported by the library."""
    names = declared_symbols()
    missing = [n for n in names if not hasattr(lib, n)]
    if missing:
        raise NcfaError(f"libncfa.so does not export: {missing}")
    return names


for _name, (_res, _args) in _SIGNATURES.items():
    if hasattr(lib, _name):
        _fn = getattr(lib, _name)
        _fn.restype = _res
        _fn.argtypes = _args


def profile_report() -> dict:
    """{kernel name: (launches, total_ms)} since profiling was enabled; clears the records."""
    buf = ctypes.create_string_buffer(1 << 16)
    check(lib.ncfa_profile_report(buf, len(buf)), "ncfa_profile_report")
    out = {}
    for line in buf.value.decode().splitlines():
        name, n, ms = line.split(",")
        out[name] = (int(n), float(ms))
    return out


def profile_timeline() -> list:
    """[(kernel name, stream, t0_ms, t1_ms)] of every launch since profiling was enabled; clears the records."""
    buf = ctypes.create_string_buffer(1 << 22)
    check(lib.ncfa_profile_timeline(buf, len(buf)), "ncfa_profile_timeline")
    out = []
    for line in buf.value.decode().splitlines():
        name, st, t0, t1 = line.split(",")
        out.append((name, st, float(t0), float(t1)))
    return out


def last_error() -> str:
    return (lib.ncfa_last_error() or b"").decode("utf-8", "replace")


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise NcfaError(f"{what} failed with status {rc}: {last_error()}")
