"""The reference's own control flow (its io/tempo/pitch/xcorr/consensus/pipeline modules run UNMODIFIED over the
librosa shim, tests/golden/make_pipeline_golden.py → tests/golden/pipeline_golden.json) against
  * the CPU oracle port (oracle/pipeline_port.py)            — CPU tests, pin the port to the reference's flow;
  * the CUDA product (nightcore_analyzer)                    — GPU tests, through the drop-in API.
Integer-derived outputs (quantised BPMs, chunk Hz, bootstrap ratios/CIs, IBI ratio) are compared bit-exact via
float.hex; the xcorr quality (float32 cosine) within 1e-5."""
import json
import os

import numpy as np
import pytest
import scipy.signal

from conftest import fromhex
from oracle import pipeline_port as port
from oracle import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SR = 22050


@pytest.fixture(scope="module")
def g():
    with open(os.path.join(ROOT, "tests", "golden", "pipeline_golden.json")) as f:
        return json.load(f)


def unhex(v):
    return None if v is None else fromhex(v)


def pair_A():
    src, nc = synth.make_pair(1000, 45.0, SR)
    return nc, src


def pair_C():
    a = synth.synth(4000, 120.0, SR, bpm=124.0)
    b = scipy.signal.resample_poly(a, 1000, 1003).astype(np.float32)
    b = (b + np.random.default_rng(4000).standard_normal(len(b)).astype(np.float32) * 0.01).astype(np.float32)
    return a, b


def pair_D():
    body = synth.synth(77, 60.0, SR, bpm=110.0)
    intro = synth.synth(78, 12.0, SR, bpm=90.0) * 0.3
    return np.concatenate([intro, body]).astype(np.float32), scipy.signal.resample_poly(body, 4, 5).astype(np.float32)


# ------------------------------------------------------------------------------------------- CPU: port vs golden
def test_port_pipeline_matches_reference_flow(g):
    nc, src = pair_A()
    w = port.run_arrays(nc, src, SR)
    A = g["pipeline_A"]
    assert w["src_tempos"] == [unhex(v) for v in A["src_tempos"]]
    assert w["nc_tempos"] == [unhex(v) for v in A["nc_tempos"]]
    assert w["nc_hz"] == [unhex(v) for v in A["nc_hz"]] and w["src_hz"] == [unhex(v) for v in A["src_hz"]]
    assert w["tempo"] == (unhex(A["tempo_ratio"]), tuple(unhex(v) for v in A["tempo_ci"]))
    assert w["ibi"] == (unhex(A["ibi_ratio"]), tuple(unhex(v) for v in A["ibi_ci"]))


def test_port_xcorr_and_align_match_reference_flow(g):
    a, b = pair_C()
    ratio, quality = port.speed_xcorr_arrays(a, b, SR)
    assert ratio == unhex(g["xcorr_C"]["ratio"]) and quality == unhex(g["xcorr_C"]["quality"])
    s, n = pair_D()
    off, speed = port.content_offset(s, n, SR)
    assert off == unhex(g["align_D"]["offset_sec"]) and float(speed) == unhex(g["align_D"]["speed"])


def test_port_pitch_chroma_matches_reference_flow(g):
    """The reference's estimate_pitch_chroma, as stored in the golden file, against the port's chunk-wise chroma lags
    and shift bootstrap on the same inputs."""
    src3 = synth.synth(3000, 75.0, SR, bpm=112.0)
    nc3 = synth.synth(3000, 60.0, SR, bpm=112.0, speed=1.25, pitch_mult=1.25 * 2.0 ** (1.5 / 12))
    s_hz, n_hz, point, ci, n_chunks, _ = port.estimate_pitch_chroma(src3, nc3, SR)
    B = g["pitch_B"]
    assert n_hz == [unhex(v) for v in B["nc_hz"]] and point == unhex(B["point_st"]) and n_chunks == B["n_chunks"]
    assert s_hz == [unhex(v) for v in B["src_hz"]]
    assert tuple(ci) == tuple(unhex(v) for v in B["ci_st"])


# ------------------------------------------------------------------------------------------- GPU: product vs golden
@pytest.mark.gpu
def test_gpu_pipeline_matches_reference_flow(engine, g):
    import nightcore_analyzer as na
    nc, src = pair_A()
    logs = []
    res = na.run_arrays(nc, src, SR, log=logs.append)
    A = g["pipeline_A"]
    assert res.src_tempos_raw == [unhex(v) for v in A["src_tempos"]]
    assert res.nc_tempos_raw == [unhex(v) for v in A["nc_tempos"]]
    assert res.nc_pitches_raw == [unhex(v) for v in A["nc_hz"]]
    assert res.tempo_ratio == unhex(A["tempo_ratio"]) and list(res.tempo_ci) == [unhex(v) for v in A["tempo_ci"]]
    assert res.pitch_ratio == unhex(A["pitch_ratio"]) and list(res.pitch_ci) == [unhex(v) for v in A["pitch_ci"]]
    assert res.ibi_ratio == unhex(A["ibi_ratio"]) and list(res.ibi_ci) == [unhex(v) for v in A["ibi_ci"]]
    assert res.classification == A["classification"] and res.pitch_method == A["pitch_method"]
    assert res.warnings == A["warnings"] and res.rubberband == A["rubberband"]
    assert str(res) == A["str"]
    assert [res.n_source_pitch_windows, res.n_nc_pitch_windows, res.n_source_tempo_windows,
            res.n_nc_tempo_windows] == A["n"]
    # log lines of pipeline.run after the two "Loading…" stanzas (run_arrays starts at "Stripping silence")
    ref_logs = A["logs"][A["logs"].index(next(m for m in A["logs"] if m.startswith("Stripping silence"))):]
    assert logs == ref_logs


@pytest.mark.gpu
def test_gpu_pitch_chroma_matches_reference_flow(engine, g):
    from nightcore_analyzer import pitch as npitch
    src3 = synth.synth(3000, 75.0, SR, bpm=112.0)
    nc3 = synth.synth(3000, 60.0, SR, bpm=112.0, speed=1.25, pitch_mult=1.25 * 2.0 ** (1.5 / 12))
    logs = []
    s_hz, n_hz, point, ci, n_chunks = npitch.estimate_pitch_chroma(src3, nc3, SR, log=logs.append)
    B = g["pitch_B"]
    assert n_hz == [unhex(v) for v in B["nc_hz"]] and s_hz == [unhex(v) for v in B["src_hz"]]
    assert point == unhex(B["point_st"]) and tuple(ci) == tuple(unhex(v) for v in B["ci_st"]) and n_chunks == B["n_chunks"]
    assert logs == B["logs"]


@pytest.mark.gpu
def test_gpu_xcorr_and_align_match_reference_flow(engine, g, tmp_path):
    from nightcore_analyzer import xcorr as nx
    a, b = pair_C()
    np.save(tmp_path / "a.npy", a)
    np.save(tmp_path / "b.npy", b)
    ratio, quality = nx.estimate_speed_xcorr(str(tmp_path / "a.npy"), str(tmp_path / "b.npy"))
    assert ratio == unhex(g["xcorr_C"]["ratio"])
    assert abs(quality - unhex(g["xcorr_C"]["quality"])) <= 1e-5
    assert nx.quality_label(quality) == g["xcorr_C"]["label"]
    s, n = pair_D()
    off, speed = nx.find_content_offset(s, n, SR)
    assert off == unhex(g["align_D"]["offset_sec"]) and float(speed) == unhex(g["align_D"]["speed"])
