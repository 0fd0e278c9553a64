"""CPU: oracle/xcorr_restated.py, the restatement the GPU search tests compare against, agrees with the port of the
reference (oracle/pipeline_port.py).

The speed search is not compared value for value: the port's c is `np.float32 / float`, which numpy 2 rounds to float32
(NEP 50), while the reference pins numpy < 2, where it is float64, and the kernel and the restatement follow the float64
form.  The two can pick differently only where two candidates tie in float32, which these pairs never do, so the picks
must be identical and the values agree to float32 rounding."""
import numpy as np
import pytest

from oracle import librosa_restated as lr
from oracle import pipeline_port as port
from oracle import synth
from oracle import xcorr_restated as xr
from test_gpu_xcorr import SR, make_pair


def port_grid(ya, yb, sr, stride):
    """The windows and candidate grid of port.speed_xcorr_arrays → (s, win, a_pos, b_lo, n_cand)."""
    min_len = min(len(ya), len(yb))
    s, e = int(min_len * 0.10), int(min_len * 0.90)
    la, lb = len(ya[s:e]), len(yb[s:e])
    win = int(3.0 * sr)
    search = int(0.05 * lb)
    a_pos = np.linspace(0, la - win, 20).astype(int).astype(np.int64)
    b_lo = np.zeros(len(a_pos), dtype=np.int64)
    n_cand = np.zeros(len(a_pos), dtype=np.int32)
    for i, pa in enumerate(a_pos):
        expected = int(pa * lb / la)
        lo_b, hi_b = max(0, expected - search), min(lb - win, expected + search)
        b_lo[i] = lo_b
        n_cand[i] = 0 if lo_b >= hi_b else len(range(lo_b, hi_b, stride))
    return s, win, a_pos, b_lo, n_cand


@pytest.mark.parametrize("div", [4, 8])
@pytest.mark.parametrize("seed,dur,sr", [(4000, 120.0, SR), (4001, 40.0, 44100), (4002, 60.0, SR), (4003, 60.0, SR)])
def test_search_picks_match_port(seed, dur, sr, div):
    a, b = make_pair(seed, dur, sr)
    win = int(3.0 * sr)
    stride = win // div
    (_, w_quality), (w_pos, w_pb) = port.speed_xcorr_arrays(a, b, sr, return_indices=True, stride=stride)
    s, win, a_pos, b_lo, n_cand = port_grid(a, b, sr, stride)
    assert a_pos.tolist() == w_pos.tolist()
    bj, bc = xr.search(a, b, s + a_pos, s + b_lo, n_cand, win, stride, port.XCORR_RMS_GATE)
    assert bj.dtype == np.int32 and bc.dtype == np.float64
    got_pb = np.where(bj >= 0, b_lo + bj.astype(np.int64) * stride, -1)
    assert got_pb.tolist() == w_pb.tolist()
    assert int((bj >= 0).sum()) >= 3
    keep = bj >= 0
    assert abs(float(np.median(bc[keep])) - w_quality) <= 1e-6


def test_search_gates_and_ties():
    """Exact integer data: the RMS gate at the window's float32 RMS, a zero A window, a zero B candidate, periodic B."""
    rng = np.random.default_rng(3)
    win, stride = 12, 4
    a = rng.integers(-4, 5, 3 * win).astype(np.float32)
    a[win : 2 * win] = 0.0
    b = np.tile(rng.integers(-4, 5, stride), 12).astype(np.float32)     # period of one block: every candidate ties
    b[-win:] = 0.0
    a_pos = np.array([0, win, 2 * win])
    b_lo = np.array([0, 0, len(b) - win])
    n_cand = np.array([6, 6, 1])
    c = xr.candidate_c(a, b, a_pos, b_lo, n_cand, win, stride, 0.0)
    assert np.all(c[0, :6] == c[0, 0]) and np.all(c[1] == -np.inf) and c[2, 0] == -np.inf
    bj, bc = xr.search(a, b, a_pos, b_lo, n_cand, win, stride, 0.0)
    want0 = (0, float(c[0, 0])) if c[0, 0] > 0 else (-1, 0.0)
    assert (int(bj[0]), float(bc[0])) == want0 and bj[1:].tolist() == [-1, -1] and bc[1:].tolist() == [0.0, 0.0]
    rms = np.float32(np.sqrt(np.sum(a[:win].astype(np.float64) ** 2) / np.float64(win)))
    assert xr.search(a, b, a_pos[:1], b_lo[:1], n_cand[:1], win, stride, np.float64(rms))[0][0] == want0[0]
    assert xr.search(a, b, a_pos[:1], b_lo[:1], n_cand[:1], win, stride, np.nextafter(np.float64(rms), np.inf))[0][0] == -1


def align_case(seed_body, seed_intro):
    body = synth.synth(seed_body, 60.0, SR, bpm=110.0)
    intro = synth.synth(seed_intro, 12.0, SR, bpm=90.0) * 0.3
    src = np.concatenate([intro, body]).astype(np.float32)
    import scipy.signal
    nc = scipy.signal.resample_poly(body, 4, 5).astype(np.float32)
    return src, nc


@pytest.mark.parametrize("seeds", [(77, 78), (79, 80)])
def test_align_matches_port_debug(seeds):
    """The geometry of port.content_offset (xcorr.py:221-240) fed to xr.align gives the port's (peak, score) per speed,
    bit for bit: both are the same numpy operations."""
    src, nc = align_case(*seeds)
    _, dbg = port.content_offset(src, nc, SR, return_debug=True)
    src_env = lr.rms(lr.resample(src, SR, port.ALIGN_SR), 2048, port.ALIGN_HOP).astype(np.float64)
    nc_env = lr.rms(lr.resample(nc, SR, port.ALIGN_SR), 2048, port.ALIGN_HOP).astype(np.float64)
    max_frames = int(120.0 / (port.ALIGN_HOP / port.ALIGN_SR))
    n_str, n_lag = [], []
    for speed in np.linspace(1.03, 1.50, 30):
        ns = int(len(nc_env) / speed)
        search_len = min(max_frames, len(src_env) - ns)
        live = 4 <= ns < len(src_env) and search_len > 0
        n_str.append(ns if live else 0)
        n_lag.append(search_len + 1 if live else -1)
    peak, score, rows = xr.align(src_env, nc_env, np.array(n_str), np.array(n_lag))
    assert len(dbg) == 30 and any(d is not None for d in dbg)
    for s, d in enumerate(dbg):
        if d is None:
            assert (int(peak[s]), float(score[s]), rows[s]) == (-1, 0.0, None)
        else:
            assert (int(peak[s]), float(score[s])) == d, s
            assert len(rows[s]) == n_str[s]


def test_stretch_is_np_interp_of_linspace():
    """n_stretched = 1 is np.linspace(0, 1, 1) = [0]: the first envelope value, not the last."""
    nc = np.array([-2.0, 1.0, 3.0])
    assert xr.stretch(nc, 1).tolist() == [-2.0]
    assert xr.stretch(nc, 2).tolist() == [-2.0, 3.0]
    assert xr.stretch(nc, 5).tolist() == [-2.0, -0.5, 1.0, 2.0, 3.0]
    peak, score, rows = xr.align(np.array([1.0, 5.0, 2.0]), nc, np.array([1, 3]), np.array([3, 0]))
    assert peak.tolist() == [0, -1] and score.tolist() == [-1.0, 0.0] and rows[1] is None
