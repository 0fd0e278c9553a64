"""GPU: the band-limited speed change (ncfa_render_batched, the HQNC render of workflow.py:117) against its numpy
restatement bit for bit — at every ratio kind, short and odd lengths, mono and stereo, in mixed batches and at every
sample placement — its launch accounting, and the render → verify → re-render loop end to end."""
import numpy as np
import pytest
import torch

from oracle import render_restated as rr, synth

pytestmark = pytest.mark.gpu
RATIOS = (0.8, 1.0, 1.2315, 1.25, 1.5, 1.25 * 44100 / 48000)
LENGTHS = (1, 2, 3, 511, 4097, 88200)
CANARY = 1.0e3


@pytest.fixture(scope="module")
def table():
    from nightcore_analyzer import _native
    t = np.zeros(rr.ZEROS * rr.PHASES + 1)
    _native.check(_native.lib.ncfa_host_render_table(t.ctypes.data), "ncfa_host_render_table")
    return t


def noise(n, seed):
    return (np.random.default_rng(seed).standard_normal(n) * 0.3).astype(np.float32)


def same_bits(a, b):
    return a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()


@pytest.mark.parametrize("ratio", RATIOS)
def test_matches_oracle_bit_for_bit(engine, table, ratio):
    from nightcore_analyzer import render
    tracks = [noise(n, n) for n in LENGTHS] + [np.stack([noise(88200, 1), noise(88200, 2)], axis=1)]
    got = render.speed_arrays(tracks, ratio)
    for t, g in zip(tracks, got):
        if t.ndim == 1:
            assert same_bits(g, rr.render(t, ratio, table)), (len(t), ratio)
        else:
            assert g.shape == (rr.out_len(len(t), ratio), 2)
            for j in range(2):
                assert same_bits(np.ascontiguousarray(g[:, j]), rr.render(t[:, j], ratio, table)), (j, ratio)


def test_mixed_launch_equals_segments_alone(engine):
    segs = [noise(n, 100 + n) for n in (4097, 1, 88200, 511, 2, 30000)]
    ratios = np.array([1.5, 0.8, 1.2315, 1.0, 1.25, 1.25 * 44100 / 48000])
    audio, off, ln = engine.pack(segs)
    out, out_off = engine.render_dev(audio, off, ln, ratios)
    out_len = engine.render_layout(ln, ratios)[0]
    h = out.cpu().numpy()
    for i, (s, r) in enumerate(zip(segs, ratios)):
        a1, o1, l1 = engine.pack([s])
        alone, _ = engine.render_dev(a1, o1, l1, [r])
        assert same_bits(h[out_off[i] : out_off[i] + out_len[i]], alone.cpu().numpy()[: out_len[i]]), (i, r)


def place(engine, arrays, phases, canary=CANARY, margin=4096, seed=1234):
    """Device buffer with array i at an offset ≡ phases[i] (mod 4) and at least `margin` samples of loud seeded noise
    before and after every array → (audio, seg_off int64, seg_len int32)."""
    lens = np.array([len(a) for a in arrays], dtype=np.int32)
    starts = np.zeros(len(arrays), dtype=np.int64)
    pos = margin
    for i, (n, ph) in enumerate(zip(lens, phases)):
        pos += (int(ph) - pos) % 4
        starts[i] = pos
        pos += int(n) + margin
    host = (np.random.default_rng(seed).standard_normal(pos) * canary).astype(np.float32)
    for a, s, n in zip(arrays, starts, lens):
        host[s : s + n] = np.asarray(a, dtype=np.float32)
    return torch.from_numpy(host).to(engine.device), starts, lens


def test_placement_invariance(engine):
    segs = [noise(n, 7 + n) for n in (1, 3, 511, 4097, 20001)]
    ratios = np.array([1.25, 0.8, 1.5, 1.2315, 1.25 * 44100 / 48000])
    out_len = engine.render_layout(np.array([len(s) for s in segs]), ratios)[0]

    def run(audio, off, ln):
        out, out_off = engine.render_dev(audio, off, ln, ratios)
        h = out.cpu().numpy()
        return [h[o : o + n].copy() for o, n in zip(out_off, out_len)]

    want = run(*engine.pack(segs))
    for phase in range(4):
        got = run(*place(engine, segs, [(phase + i) % 4 for i in range(len(segs))]))
        for i, (g, w) in enumerate(zip(got, want)):
            assert same_bits(g, w), (phase, i)


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


def test_launch_count_matches_the_profiler(engine, profiled):
    audio, off, ln = engine.pack([noise(5000, 1), noise(300, 2), noise(0, 3)])
    torch.cuda.synchronize()
    profiled.profile_report()
    l0 = engine.launches
    engine.render_dev(audio, off, ln, [1.25, 0.8, 1.5])
    torch.cuda.synchronize()
    prof = profiled.profile_report()
    assert "render_kernel" in prof and prof["render_kernel"][0] == 1
    assert engine.launches - l0 == sum(n for n, _ in prof.values()), prof


def _stereo_source(sr, seconds=60.0):
    left = synth.synth(2100, seconds, sr, bpm=128.0)
    right = 0.8 * left + 0.05 * np.random.default_rng(9).standard_normal(len(left))
    st = np.stack([left, right], axis=1)
    return (0.5 * st / np.max(np.abs(st))).astype(np.float32)


def _write_pair(tmp_path, sr, width):
    import scipy.signal
    from nightcore_analyzer.io import write_wav
    src = _stereo_source(sr)
    ncog = np.stack([scipy.signal.resample_poly(src[:, j], 4, 5) for j in range(2)], axis=1)   # speed 1.25
    write_wav(tmp_path / "src.wav", src, sr, width)
    write_wav(tmp_path / "ncog.wav", ncog, sr, 2)
    return str(tmp_path / "src.wav"), str(tmp_path / "ncog.wav"), str(tmp_path / "hqnc.wav")


def test_render_and_verify_corrects_the_speed(engine, tmp_path):
    import scipy.signal
    from nightcore_analyzer import render, verify
    from nightcore_analyzer.io import load_audio, read_wav
    src, ncog, out = _write_pair(tmp_path, 22050, 2)
    hist = render.render_and_verify(src, ncog, out, speed=1.2315)
    assert len(hist) == 2 and not hist[0][1].tempo_ok and hist[1][1].tempo_ok, [(s, v.best_ratio) for s, v in hist]
    speed, v = hist[-1]
    assert abs(speed / 1.25 - 1.0) < 0.005, speed
    frames, rate, width = read_wav(out)
    assert (rate, width, frames.shape[1]) == (22050, 2, 2) and len(frames) == rr.out_len(60 * 22050, speed)
    first = render.render_and_verify(src, ncog, out, speed=None)
    assert abs(first[0][0] / 1.25 - 1.0) < 0.02, first[0][0]
    # The waveform cross-correlation steps its candidates a quarter window (0.75 s) apart, so its quality is the
    # correlation at up to 0.375 s of misalignment: on this synthetic beat track it is low for any resampler (about
    # 0.1).  The HQNC must score at least what an independent resampler's copy of the nightcore scores.
    src_mono = read_wav(src)[0].mean(axis=1)
    ref = scipy.signal.resample_poly(src_mono.astype(np.float64), 4, 5).astype(np.float32)
    q_ref = verify.verify_arrays(ref, load_audio(ncog)[0], 22050, log=None).result.xcorr_quality
    assert v.result.xcorr_quality >= q_ref - 0.02, (v.result.xcorr_quality, q_ref)


def test_render_and_verify_from_a_24_bit_44k_source(engine, tmp_path):
    from nightcore_analyzer import render
    from nightcore_analyzer.io import read_wav
    src, ncog, out = _write_pair(tmp_path, 44100, 3)
    hist = render.render_and_verify(src, ncog, out)
    speed, v = hist[-1]
    assert v.tempo_ok and abs(speed / 1.25 - 1.0) < 0.005, [(s, w.best_ratio) for s, w in hist]
    frames, rate, width = read_wav(out)
    assert (rate, width, frames.shape[1]) == (44100, 3, 2)


def test_render_cli_speed_mode(engine, tmp_path):
    from nightcore_analyzer import render
    from nightcore_analyzer.io import read_wav, write_wav
    x = np.stack([noise(10000, 1), noise(10000, 2)], axis=1)
    write_wav(tmp_path / "s.wav", x, 44100, 3)
    assert render.main(["--source", str(tmp_path / "s.wav"), "--output", str(tmp_path / "o.wav"), "--speed", "1.25"]) == 0
    frames, rate, width = read_wav(tmp_path / "o.wav")
    src, _, _ = read_wav(tmp_path / "s.wav")
    want = np.stack([render.speed_arrays([src], 1.25)[0][:, j] for j in range(2)], axis=1)
    assert (rate, width) == (44100, 3) and frames.shape == want.shape
    full = float(1 << 23)
    assert np.array_equal(frames * full, np.clip(np.rint(want.astype(np.float64) * full), -full, full - 1))
