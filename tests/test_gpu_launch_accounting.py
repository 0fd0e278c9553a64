"""GPU: Engine.launches (bench.py's gpu_launches) counts exactly the kernels the library launches.  Every launch in
libncfa is profiled under its kernel name, so with ncfa_profile_enable(1) the launch counts of profile_report() must
add up to the increment of Engine.launches, call by call."""
import numpy as np
import pytest
import torch

from oracle import synth

pytestmark = pytest.mark.gpu
SR = 22050


@pytest.fixture
def profiled(engine):
    from nightcore_analyzer import _native
    torch.cuda.synchronize()
    _native.lib.ncfa_profile_enable(1)
    _native.profile_report()
    try:
        yield _native
    finally:
        torch.cuda.synchronize()
        _native.profile_report()
        _native.lib.ncfa_profile_enable(0)


def test_engine_launch_count_matches_the_profiler(engine, profiled):
    y = synth.synth(11, 12.0, SR, bpm=124.0)
    z = synth.synth(12, 5.0, SR, bpm=131.0)
    audio, off, ln = engine.pack([y, z])
    d_off, d_len = engine.to_dev(off), engine.to_dev(ln)
    bpm = np.array([120.0, 130.0])
    d_bpm = engine.to_dev(bpm)
    rng = np.random.default_rng(5)
    a_len, b_len = np.array([35, 30], np.int32), np.array([27, 20], np.int32)
    a_off = np.array([0, 35], np.int64)
    b_off = np.array([0, 27], np.int64)
    d_a = engine.to_dev(100.0 + rng.random(65))
    d_b = engine.to_dev(120.0 + rng.random(47))
    chroma = torch.from_numpy(rng.random((3, 12))).to(engine.device)
    torch.cuda.synchronize()
    profiled.profile_report()

    rows = []

    def count(name, fn):
        l0 = engine.launches
        out = fn()
        torch.cuda.synchronize()
        prof = profiled.profile_report()
        rows.append((name, engine.launches - l0, sum(n for n, _ in prof.values()), sorted(prof)))
        return out

    count("to_dev", lambda: engine.to_dev(np.arange(10, dtype=np.int64)))
    count("window_energy_dev", lambda: engine.window_energy_dev(audio, d_off, d_len))
    count("rms_frames_dev", lambda: engine.rms_frames_dev(audio, int(ln[0]), 2048, 512))
    count("trim_bounds_dev", lambda: engine.trim_bounds_dev(audio, off, ln, 60.0))
    onset, _, env_len, d_env_off, d_env_len = count("onset_strength_dev",
                                                    lambda: engine.onset_strength_dev(audio, off, ln, 512, SR))
    lag = count("tempo_lag_dev", lambda: engine.tempo_lag_dev(onset, d_env_off, d_env_len, env_len, 512, SR, d_bpm))
    count("beat_track_dev", lambda: engine.beat_track_dev(onset, d_env_off, d_env_len, env_len, lag, 512, SR))
    count("tempo_segments_dev", lambda: engine.tempo_segments_dev(audio, off, ln, bpm, 64, SR))
    count("bootstrap_dev", lambda: engine.bootstrap_dev(d_a, a_off, a_len, d_b, b_off, b_len, 7, 500, 2.5, 97.5))
    count("chroma_mean_dev", lambda: engine.chroma_mean_dev(audio, off, ln, SR))
    count("cyclic_xcorr_dev", lambda: engine.cyclic_xcorr_dev(chroma, chroma.roll(2, dims=1)))
    for stride in (1024, 512):       # block form (win / stride = 4) and direct form (8)
        count(f"xcorr_search_dev[stride={stride}]",
              lambda: engine.xcorr_search_dev(audio, audio, off[:1] + 1000, off[1:] + 100, np.array([10]), 4096,
                                              stride, 0.0))
    count("spectral_stats_dev", lambda: engine.spectral_stats_dev(audio, off, ln, SR))
    src_env = count("align_envelope", lambda: engine.align_envelope(y, SR, SR // 2, 512))
    nc_env = engine.align_envelope(z, SR, SR // 2, 512)
    torch.cuda.synchronize()
    profiled.profile_report()
    n_str = np.array([100, 120], np.int32)
    count("align_search", lambda: engine.align_search(src_env, nc_env, n_str, src_env.numel() - n_str + 1))

    assert all(n > 0 for _, n, _, _ in rows)
    bad = [r for r in rows if r[1] != r[2]]
    assert not bad, "\n".join(f"{name}: Engine.launches +{n}, profiler {p} {names}" for name, n, p, names in bad)
