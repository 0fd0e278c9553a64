"""GPU: waveform cross-correlation speed search and intro alignment vs the CPU restatement
(oracle/pipeline_port.py: speed_xcorr_arrays / content_offset).

best_pb per window and the alignment peak index are integers and must be identical; slope is a
polyfit of identical integer tables (exact); quality is a float32-rounded cosine: abs 1e-5."""
import numpy as np
import pytest
import scipy.signal

from oracle import pipeline_port as port
from oracle import synth

pytestmark = pytest.mark.gpu
SR = 22050


def make_pair(seed, dur, sr=SR, up=1000, down=1003):
    a = synth.synth(seed, dur, sr, bpm=124.0)
    b = scipy.signal.resample_poly(a, up, down).astype(np.float32)
    b = (b + np.random.default_rng(seed).standard_normal(len(b)).astype(np.float32) * 0.01).astype(np.float32)
    return a, b


def test_speed_xcorr_matches_port(engine):
    from nightcore_analyzer import xcorr as nx
    a, b = make_pair(4000, 120.0)
    (slope, quality), (a_pos, best_pb) = nx.estimate_speed_xcorr_batch([(a, b)], SR, return_indices=True)[0]
    (w_slope, w_quality), (w_pos, w_pb) = port.speed_xcorr_arrays(a, b, SR, return_indices=True)
    assert a_pos.tolist() == w_pos.tolist()
    assert best_pb.tolist() == w_pb.tolist()
    assert slope == w_slope
    assert abs(quality - w_quality) <= 1e-5
    assert nx.estimate_speed_xcorr_arrays(a, b, SR) == (slope, quality)


def test_speed_xcorr_44k_and_batch(engine):
    from nightcore_analyzer import xcorr as nx
    a, b = make_pair(4001, 40.0, sr=44100)
    c, d = make_pair(4002, 60.0)
    res = nx.estimate_speed_xcorr_batch([(a, b)], 44100, return_indices=True)[0]
    want = port.speed_xcorr_arrays(a, b, 44100, return_indices=True)
    assert res[1][1].tolist() == want[1][1].tolist() and res[0][0] == want[0][0]
    both = nx.estimate_speed_xcorr_batch([(c, d), (c, c)], SR)
    assert both[0] == nx.estimate_speed_xcorr_arrays(c, d, SR)
    w_same = port.speed_xcorr_arrays(c, c, SR)     # identical files: the strided grid need not contain the true offset
    assert both[1][0] == w_same[0] and abs(both[1][1] - w_same[1]) <= 1e-5


def test_xcorr_direct_path_matches_port(engine):
    """stride = win // 8: a window spans 8 blocks, more than the block form takes, so the search runs the direct kernels
    (one CTA per (window, candidate)) — the path of any (win, stride) outside the block form."""
    from nightcore_analyzer import xcorr as nx
    a, b = make_pair(4003, 60.0)
    s, la, lb, win, _, a_pos, lo, _ = nx._search_tables(len(a), len(b), SR, nx.XCORR_N_WINDOWS, nx.XCORR_WINDOW_SEC,
                                                         nx.XCORR_SEARCH_RANGE, nx.XCORR_SKIP_EDGES)
    stride = win // 8
    search = int(nx.XCORR_SEARCH_RANGE * lb)
    n_cand = np.zeros(len(a_pos), dtype=np.int32)
    for i, (pa, lo_b) in enumerate(zip(a_pos, lo)):
        hi_b = min(lb - win, int(pa * lb / la) + search)
        n_cand[i] = 0 if lo_b >= hi_b else len(range(lo_b, hi_b, stride))
    audio, off, _ = engine.pack([a, b])
    bj, bc = engine.xcorr_search_dev(audio, audio, off[0] + s + a_pos, off[1] + s + lo, n_cand, win, stride,
                                     nx.XCORR_RMS_GATE)
    bj, bc = engine.to_host(bj), engine.to_host(bc)
    (w_slope, w_quality), (w_pos, w_pb) = port.speed_xcorr_arrays(a, b, SR, return_indices=True, stride=stride)
    assert a_pos.tolist() == w_pos.tolist()
    assert bj.tolist() == np.where(w_pb >= 0, (w_pb - lo) // stride, -1).tolist()
    assert int((bj >= 0).sum()) >= 3
    ya, yb = a[s:], b[s:]
    for pa, lo_b, j, c in zip(a_pos, lo, bj, bc):
        if j >= 0:
            wa = ya[pa : pa + win].astype(np.float64)
            wb = yb[lo_b + j * stride : lo_b + j * stride + win].astype(np.float64)
            assert abs(c - float(np.dot(wa, wb) / (np.linalg.norm(wa) * np.linalg.norm(wb)))) <= 1e-5
    slope, quality = nx._fit(a_pos, lo, stride, bj, bc)
    assert slope == w_slope
    assert abs(quality - w_quality) <= 1e-5


def test_xcorr_direct_form_stays_inside_its_workspace(engine):
    """One window with one candidate in the direct form (win / stride = 8), given exactly ncfa_xcorr_workspace_bytes at
    the start of a larger buffer: the bytes after it keep their pattern, and the pick is the cosine of the two
    windows."""
    import torch
    from nightcore_analyzer._native import check, lib
    win, stride = 4096, 512
    rng = np.random.default_rng(21)
    a = rng.standard_normal(win).astype(np.float32)
    b = (a + 0.1 * rng.standard_normal(win)).astype(np.float32)
    audio, off, _ = engine.pack([a, b])
    d_pos, d_lo = engine.to_dev(off[:1]), engine.to_dev(off[1:])
    d_n = engine.to_dev(np.array([1], np.int32))
    need = lib.ncfa_xcorr_workspace_bytes(1, 1)
    ws = torch.full((need + 4096,), 0xA5, dtype=torch.uint8, device=engine.device)
    best_j = torch.empty(1, dtype=torch.int32, device=engine.device)
    best_c = torch.empty(1, dtype=torch.float64, device=engine.device)
    check(lib.ncfa_xcorr_search_batched(audio.data_ptr(), audio.data_ptr(), d_pos.data_ptr(), d_lo.data_ptr(),
                                        d_n.data_ptr(), 1, 1, win, stride, 0.0, best_j.data_ptr(), best_c.data_ptr(),
                                        ws.data_ptr(), need, torch.cuda.current_stream().cuda_stream),
          "ncfa_xcorr_search_batched")
    torch.cuda.synchronize()
    assert bool((ws[need:] == 0xA5).all())
    a64, b64 = a.astype(np.float64), b.astype(np.float64)
    want = float(np.dot(a64, b64) / (np.linalg.norm(a64) * np.linalg.norm(b64)))
    assert best_j.item() == 0
    assert abs(best_c.item() - want) <= 1e-5

def test_speed_xcorr_sentinels(engine):
    from nightcore_analyzer import xcorr as nx
    short = synth.synth(1, 3.0, SR, bpm=120.0)
    assert nx.estimate_speed_xcorr_arrays(short, short, SR) == (1.0, 0.0)            # shorter than one window
    z = np.zeros(SR * 30, np.float32)
    assert nx.estimate_speed_xcorr_arrays(z, z, SR) == (1.0, 0.0)                    # RMS gate drops every window
    assert nx.quality_label(0.8) == "good match" and nx.quality_label(0.5) == "moderate match"
    assert nx.quality_label(0.1).startswith("poor match")


def test_find_content_offset_matches_port(engine):
    from nightcore_analyzer import xcorr as nx
    body = synth.synth(77, 60.0, SR, bpm=110.0)
    intro = synth.synth(78, 12.0, SR, bpm=90.0) * 0.3
    src = np.concatenate([intro, body]).astype(np.float32)
    nc = scipy.signal.resample_poly(body, 4, 5).astype(np.float32)
    got = nx.find_content_offset(src, nc, SR)
    want, dbg = port.content_offset(src, nc, SR, return_debug=True)
    assert got == want
    assert got[0] > 1.0
