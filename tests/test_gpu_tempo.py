"""GPU: onset strength / tempo lag / beat DP kernels vs the CPU restatement (oracle/librosa_restated.py).

Tolerances: onset envelope float32, max abs error <= 1e-4 of the envelope's maximum (the FFT
runs in float32 on the device, in float64 on the oracle); tempo lags and beat frames are
integers and must be identical when both sides are given the same envelope."""
import numpy as np
import pytest

from oracle import librosa_restated as lr
from oracle import synth

pytestmark = pytest.mark.gpu
SR = 22050


def rel_err(a, b):
    return float(np.max(np.abs(a - b)) / max(1e-12, float(np.max(np.abs(b)))))


@pytest.fixture(scope="module")
def windows():
    out = []
    for seed, bpm in ((1, 96.0), (2, 120.0), (3, 139.0)):
        y = synth.synth(seed, 20.0, SR, bpm=bpm)
        out += [y[:220500], y[110250:330750]]
    return out


def test_onset_strength_hop512(engine, windows):
    got = engine.onset_strength(windows, hop=512, sr=SR)
    for y, g in zip(windows, got):
        want = lr.onset_strength(y, SR, 512)
        assert g.shape == want.shape == (431,)
        assert np.all(g[:3] == 0)
        assert rel_err(g, want) < 1e-4


def test_onset_strength_hop64_and_ragged(engine):
    ys = [synth.synth(4, 6.0, SR, bpm=110.0), synth.synth(5, 3.3, SR, bpm=128.0)[:70001], np.zeros(5000, np.float32)]
    got = engine.onset_strength(ys, hop=64, sr=SR)
    for y, g in zip(ys, got):
        want = lr.onset_strength(y, SR, 64)
        assert g.shape == want.shape
        assert rel_err(g, want) < 1e-4 or float(np.max(np.abs(want))) == 0.0
    assert np.all(got[2] == 0)


@pytest.mark.parametrize("hop", [64, 512, 96])
def test_onset_kernel_matches_oracle_at_each_hop_form(engine, hop):
    """The STFT kernel has one instantiation per hop class: hop 64 and hop 512 (the two frames of a warp share register
    loads) and any other even hop (two independent loads; hop 96 here).  Each matches the oracle — ragged tails, odd
    frame counts and short segments included; an all-zero envelope must come out all zero."""
    ys = [synth.synth(7, 4.0, SR, bpm=101.0), synth.synth(8, 2.0, SR, bpm=133.0)[:40001], synth.synth(9, 1.0, SR)[:1500],
          synth.synth(10, 3.0, SR)[:64 * 700]]
    got = engine.onset_strength(ys, hop=hop, sr=SR)
    for i, (y, g) in enumerate(zip(ys, got)):
        want = lr.onset_strength(y, SR, hop)
        assert g.shape == want.shape, (i, g.shape, want.shape)
        if float(np.max(np.abs(want))) == 0.0:
            assert np.all(g == 0), i
        else:
            assert rel_err(g, want) < 1e-4, (i, rel_err(g, want))


def test_onset_top_db_clamp_active(engine):
    """A window that is silent for its first half exercises the per-segment max − 80 dB floor."""
    y = synth.synth(6, 10.0, SR, bpm=120.0).copy()
    y[:110250] *= 1e-6
    g = engine.onset_strength([y], hop=512, sr=SR)[0]
    want = lr.onset_strength(y, SR, 512)
    assert rel_err(g, want) < 1e-4


def test_short_segments(engine):
    for n in (1, 511, 512, 2047, 2049):
        y = np.random.default_rng(n).standard_normal(n).astype(np.float32)
        g = engine.onset_strength([y], hop=512, sr=SR)[0]
        want = lr.onset_strength(y, SR, 512)
        assert g.shape == want.shape
        assert np.max(np.abs(g - want)) <= 1e-4 * max(1.0, float(np.max(np.abs(want))))


def test_tempo_lag_matches_oracle_on_same_envelope(engine, windows):
    envs = [lr.onset_strength(y, SR, 512) for y in windows]
    priors = [120.0, 120.0, 90.0, 150.0, 200.0, 60.0]
    got = engine.tempo_lags(envs, priors, hop=512, sr=SR)
    want = [lr.tempo_lag(e, SR, 512, p) for e, p in zip(envs, priors)]
    assert got.tolist() == want


def test_tempo_lag_hop64(engine):
    y = synth.synth(8, 30.0, SR, bpm=126.0)
    env = lr.onset_strength(y, SR, 64)
    got = engine.tempo_lags([env], [120.0], hop=64, sr=SR)
    assert got.tolist() == [lr.tempo_lag(env, SR, 64, 120.0)]


def test_tempo_lag_weak_periodicity_and_off_centre_priors(engine):
    """Noise envelopes have a flat tempogram, so the branch-and-bound cannot prune: phase 2 has to evaluate the lags on
    BOTH sides of the phase-1 interval (exact, not block-aligned, intervals; ragged envelope lengths; priors far from
    the data).  The argmax must still be the oracle's."""
    rng = np.random.default_rng(77)
    envs, priors = [], []
    for n, p in ((431, 60.0), (431, 240.0), (300, 120.0), (97, 120.0), (431, 31.0), (1000, 300.0)):
        e = rng.exponential(1.0, n).astype(np.float32)
        e[:3] = 0.0
        envs.append(e)
        priors.append(p)
    got = engine.tempo_lags(envs, priors, hop=512, sr=SR)
    want = [lr.tempo_lag(e, SR, 512, p) for e, p in zip(envs, priors)]
    assert got.tolist() == want
    # hop 64: several 4096-frame chunks (ragged last chunk), weak periodicity, prior an octave off
    e = (rng.exponential(1.0, 9000) * (1.0 + 0.3 * np.sin(np.arange(9000) * 2 * np.pi / 171.0))).astype(np.float32)
    for p in (120.0, 55.0, 250.0):
        assert engine.tempo_lags([e], [p], hop=64, sr=SR).tolist() == [lr.tempo_lag(e, SR, 64, p)]


def test_tempo_lag_envelope_with_silent_stretches(engine):
    """Frames whose energy collapses force the running sums to be rebuilt (sign flag of the stored reciprocal) and
    all-zero stretches take the 'unscaled' branch of normalize(): the scores must survive both."""
    y = synth.synth(21, 40.0, SR, bpm=117.0).copy()
    y[5 * SR:12 * SR] = 0.0
    y[20 * SR:21 * SR] *= 1e-4
    env = lr.onset_strength(y, SR, 64)
    assert engine.tempo_lags([env], [120.0], hop=64, sr=SR).tolist() == [lr.tempo_lag(env, SR, 64, 120.0)]
    env512 = lr.onset_strength(y[: 10 * SR], SR, 512)
    assert engine.tempo_lags([env512], [120.0], hop=512, sr=SR).tolist() == [lr.tempo_lag(env512, SR, 512, 120.0)]


def test_tempo_lag_all_zero_envelope(engine):
    got = engine.tempo_lags([np.zeros(431, np.float32)], [120.0], hop=512, sr=SR)
    assert got.tolist() == [0]


def test_beat_frames_match_oracle_on_same_envelope(engine, windows):
    envs = [lr.onset_strength(y, SR, 512) for y in windows]
    lags = [lr.tempo_lag(e, SR, 512, 120.0) for e in envs]
    got = engine.beat_frames(envs, lags, hop=512, sr=SR)
    for e, lag, g in zip(envs, lags, got):
        bpm = 60.0 * SR / (512 * float(lag))
        want = lr.beat_track_frames(e, bpm, SR, 512)
        assert g.tolist() == want.tolist()


def test_beat_frames_hop64(engine):
    y = synth.synth(9, 30.0, SR, bpm=104.0)
    env = lr.onset_strength(y, SR, 64)
    lag = lr.tempo_lag(env, SR, 64, 120.0)
    got = engine.beat_frames([env], [lag], hop=64, sr=SR)[0]
    want = lr.beat_track_frames(env, 60.0 * SR / (64 * float(lag)), SR, 64)
    assert got.tolist() == want.tolist()


def test_beat_frames_ragged_batch_and_slow_tempo(engine):
    """One launch with envelopes of very different lengths and frames-per-beat (the local-score kernel's sliding
    window needs full-width interiors; short envelopes and the ends take the one-frame path; a slow tempo makes the
    DP ring wrap many times)."""
    rng = np.random.default_rng(5)
    envs, lags = [], []
    for seed, dur, bpm in ((31, 12.0, 72.0), (32, 3.0, 160.0), (33, 25.0, 95.0)):
        y = synth.synth(seed, dur, SR, bpm=bpm)
        envs.append(lr.onset_strength(y, SR, 64))
        lags.append(lr.tempo_lag(envs[-1], SR, 64, 120.0))
    envs.append(rng.exponential(1.0, 700).astype(np.float32))
    lags.append(400)   # window wider than the envelope: every frame is an edge frame
    got = engine.beat_frames(envs, lags, hop=64, sr=SR)
    for e, lag, g in zip(envs, lags, got):
        want = lr.beat_track_frames(e, 60.0 * SR / (64 * float(lag)), SR, 64)
        assert g.tolist() == want.tolist()


def test_end_to_end_tempo_api(engine, windows):
    """tempo.batch_estimate_tempo through the drop-in API: the BPM grid value must match the
    oracle run end-to-end (onset envelopes differ in the last float32 bits, the argmax must not)."""
    from nightcore_analyzer import io as nio, tempo as ntempo
    y = synth.synth(12, 40.0, SR, bpm=118.0)
    wins = nio.slice_windows(y, SR)
    assert len(wins) == 7
    lines = []
    got = ntempo.batch_estimate_tempo(wins, log=lines.append, start_bpm=120.0)
    assert lines[0] == "    tempo window 1/7  [0.0–10.0 s]" and lines[-1].endswith("windows yielded a confident tempo estimate")
    for w, g in zip(wins, got):
        env = lr.onset_strength(w.audio, SR, 512)
        bpm, beats = lr.beat_track(env, SR, 512, 120.0)
        want = float(np.atleast_1d(bpm)[0]) if len(beats) >= 4 else None
        assert g == want
    assert ntempo.estimate_tempo(wins[2], start_bpm=100.0) is not None


def test_estimate_ibis_global(engine):
    from nightcore_analyzer import tempo as ntempo
    y = synth.synth(13, 45.0, SR, bpm=125.0)
    got = ntempo.estimate_ibis_global(y, SR)
    env = lr.onset_strength(y, SR, 64)
    _, beats = lr.beat_track(env, SR, 64, 120.0)
    t = lr.frames_to_time(beats, SR, 64)
    want = np.diff(t)
    want = want[want > 0.05]
    assert got is not None and np.array_equal(got, want)
    assert ntempo.estimate_ibis_global(np.zeros(22050, np.float32), SR) is None
