"""GPU: every segment kernel at every sample placement the C ABI allows (include/ncfa.h: a segment may start at any
int64 sample offset), against the zero-padded 4-aligned layout of Engine.pack and against the oracle.

Several kernels pick their load path from the alignment of the segment start:
  * the STFT of the onset front-end (stft_logmel2_kernel), of the tuning estimator (tuning_peaks_kernel) and of both
    spectral passes loads a frame with float2 loads when its first sample is 8-byte aligned and one sample at a time
    otherwise (load_frame_guarded / the scalar loop) — phases 1 and 3 put EVERY frame on the guarded path;
  * cqt_tc_kernel stages octave 0 with cp.async when the segment start is 16-byte aligned (phase 0: the clamp-free fast
    path inside the segment, the zero-fill form at its edges) and with plain loads otherwise (phases 1, 2, 3);
  * decimate2_kernel reads level 1 with float2 loads when the segment start is 8-byte aligned (phases 0, 2) and
    de-interleaves it one sample at a time otherwise (phases 1, 3);
  * the waveform xcorr block form copies the 16-byte-aligned superset of every tile (up to three samples before and
    after a window land in shared memory and must not be used).
`place` lays the segments out at chosen residues mod 4 with `margin` samples of loud noise (the canary) before and after
every segment, the buffer's own ends included, so a read outside [0, len) changes the result instead of reading the
zeros that `pack` puts between arrays.  The canary is finite on purpose: the dB steps clamp with fmaxf(1e-10, ·), which
would swallow a NaN.

Integer and float outputs must be bit-identical across placements: the fast and the fallback paths load the same
values and do the same arithmetic, and every reduction runs in an order fixed by the segment length alone.  One
exception, the per-bin mean dB of the spectral statistics, is explained at `assert_spectral_equal`.  Parity with the
oracle uses the tolerances of the family's own test file."""
import numpy as np
import pytest

from oracle import librosa_restated as lr
from oracle import pipeline_port as port
from oracle import synth

pytestmark = pytest.mark.gpu
SR = 22050
PHASES = (0, 1, 2, 3)
CANARY = 1e3


def place(engine, arrays, phases, canary=CANARY, margin=4096, base=0, seed=1234):
    """Device buffer with array i at an offset ≡ phases[i] (mod 4), at least `margin` samples of seeded noise of
    amplitude `canary` before and after every array, the layout starting at sample `base` (samples below `base` are
    left uninitialised and never read) → (audio, seg_off int64, seg_len int32)."""
    import torch
    lens = np.array([len(a) for a in arrays], dtype=np.int32)
    starts = np.zeros(len(arrays), dtype=np.int64)
    pos = base + margin
    for i, (n, ph) in enumerate(zip(lens, phases)):
        pos += (int(ph) - pos) % 4
        starts[i] = pos
        pos += int(n) + margin
    host = (np.random.default_rng(seed).standard_normal(pos - base) * canary).astype(np.float32)
    for a, s, n in zip(arrays, starts, lens):
        host[s - base : s - base + n] = np.asarray(a, dtype=np.float32)
    if base == 0:
        audio = torch.from_numpy(host).to(engine.device)
    else:
        audio = torch.empty(pos, dtype=torch.float32, device=engine.device)
        audio[base:].copy_(torch.from_numpy(host))
    return audio, starts, lens


def rel_err(a, b):
    return float(np.max(np.abs(a - b)) / max(1e-12, float(np.max(np.abs(b)))))


def tuning_index(t):
    return int(round((t + 0.5) * 100))


# ------------------------------------------------------------------------------------------------ runners (→ numpy)
def run_onset(engine, layout, hop):
    audio, off, ln = layout
    onset, env_off, env_len, _, _ = engine.onset_strength_dev(audio, off, ln, hop, SR)
    h = onset.cpu().numpy()
    return [h[o : o + n].copy() for o, n in zip(env_off, env_len)]


def run_chroma(engine, layout, tuning_idx=None):
    audio, off, ln = layout
    chroma, tun = engine.chroma_mean_dev(audio, off, ln, SR, tuning_idx=tuning_idx)
    return chroma.cpu().numpy(), tun.cpu().numpy()


def run_spectral(engine, layout, sr):
    audio, off, ln = layout
    stats, bins = engine.spectral_stats_dev(audio, off, ln, sr)
    return stats.cpu().numpy(), bins.cpu().numpy()


def run_trim(engine, layout, top_db):
    audio, off, ln = layout
    return engine.trim_bounds_dev(audio, off, ln, top_db).cpu().numpy()


def run_energy(engine, layout):
    audio, off, ln = layout
    return engine.window_energy_dev(audio, engine.to_dev(off), engine.to_dev(ln)).cpu().numpy()


def assert_lists_equal(got, want):
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert g.dtype == w.dtype and g.shape == w.shape, i
        assert np.array_equal(g, w), (i, float(np.max(np.abs(g.astype(np.float64) - w))))


def assert_spectral_equal(got, want):
    """stats: bit-identical.  Per-bin mean dB: spectral_pass2_kernel adds every frame's dB into a float64 shared-memory
    accumulator per bin with atomicAdd from 16 warps, so the order of those additions is not fixed — not even between
    two runs of the same layout.  A reordered float64 sum moves by far less than half a float32 ulp of the mean, so the
    float32 result may differ by at most one ulp; a load from outside the segment moves it by orders of magnitude more."""
    (gs, gb), (ws, wb) = got, want
    assert np.array_equal(gs, ws), np.argwhere(gs != ws).tolist()
    assert np.all(np.abs(gb - wb) <= np.spacing(np.abs(wb))), float(np.max(np.abs(gb - wb)))


# ------------------------------------------------------------------------------------------------ signals
def onset_arrays():
    """The ragged set of test_gpu_tempo's per-hop test, plus 1, 2047, 2049 and odd lengths, plus silence."""
    return [synth.synth(7, 4.0, SR, bpm=101.0), synth.synth(8, 2.0, SR, bpm=133.0)[:40001],
            synth.synth(9, 1.0, SR)[:1500], synth.synth(10, 3.0, SR)[:64 * 700],
            synth.synth(11, 0.1, SR)[:1], synth.synth(12, 0.2, SR)[:2047], synth.synth(13, 0.2, SR)[:2049],
            synth.synth(14, 1.5, SR, bpm=117.0)[:33333], np.zeros(3001, np.float32)]


def chroma_arrays():
    """A 20 s pitch chunk, a ragged odd-length chunk, short segments around the CQT frame (1024 at octave 0) and the STFT
    frame (2048), a chunk of 441 000 + 63 samples (ragged tails at every pyramid level, octave-6 frames at the edge of
    the clamp-free fast path), and silence."""
    short = [synth.synth(60 + k, 0.5, SR, bpm=120.0)[:n] for k, n in enumerate((1, 511, 1023, 1024, 2047, 4097))]
    return ([synth.synth(31, 20.0, SR, bpm=118.0), synth.synth(34, 5.0, SR, bpm=100.0)[:100001]] + short +
            [synth.synth(35, 20.01, SR, bpm=110.0, pitch_mult=2.0 ** (0.3 / 12))[:441063], np.zeros(30001, np.float32)])


# the 20 s chunk (index 0) is compared with the oracle in test_gpu_pitch.py; every other chunk here
CHROMA_ORACLE = (1, 2, 3, 4, 5, 6, 7, 8, 9)


def spectral_arrays(sr):
    import scipy.signal
    y = synth.synth(20 + sr // 22050, 4.0, sr, bpm=120.0)
    if sr == 44100:     # band-limited like a lossy transcode, as in test_gpu_spectral
        y = scipy.signal.sosfilt(scipy.signal.butter(12, 15000, btype="low", fs=sr, output="sos"), y).astype(np.float32)
    return [y, synth.synth(22, 2.5, sr, bpm=140.0)[:50001], synth.synth(23, 0.1, sr)[:1999],
            np.zeros(4097, np.float32)]


def trim_arrays():
    """(signal, name) pairs for librosa.effects.trim.  Leading / trailing silences end in the middle of a 512-sample
    block; frame dB values stay clear of every tested −top_db threshold (asserted in test_trim_thresholds_are_clear)."""
    rng = np.random.default_rng(99)
    out = [(synth.synth(70 + k, 0.2, SR)[:n], f"len{n}") for k, n in enumerate((1, 511, 512, 513, 2047, 2048, 2049))]
    y = np.zeros(100003, np.float32)
    y[30257:81111] = synth.synth(80, 3.0, SR, bpm=125.0)[: 81111 - 30257]
    out.append((y, "silence_both_ends"))
    spike = np.zeros(20001, np.float32)
    spike[7777] = 0.9
    out.append((spike, "spike"))
    quiet = synth.synth(81, 2.0, SR, bpm=95.0).copy()
    quiet[: 20000 + 300] *= 1e-6
    out.append((quiet, "quiet_start_1e-6"))
    tail = synth.synth(82, 1.5, SR, bpm=130.0).copy()
    tail[-12345:] = 0.0
    tail[-12345:-9000] = (rng.standard_normal(3345) * 1e-5).astype(np.float32)
    out.append((tail, "quiet_then_silent_tail"))
    # a 100 dB fade-in and fade-out: every top_db cuts at a different frame
    t = np.arange(60001) / 60001.0
    fade = (rng.standard_normal(60001) * 10.0 ** (-5.0 * np.abs(2.0 * t - 1.0))).astype(np.float32)
    out.append((fade, "fades"))
    out.append((np.zeros(7001, np.float32), "zeros"))
    return out


TRIM_DB = (30.0, 60.0, 80.0)


def oracle_trim_db(y):
    """The frame dB values librosa.effects.trim compares with −top_db (oracle/librosa_restated.trim)."""
    mag = np.abs(lr.rms(y, 2048, 512))
    ref = np.max(mag)
    return 10.0 * np.log10(np.maximum(1e-5 ** 2, mag ** 2)) - 10.0 * np.log10(np.maximum(1e-5 ** 2, ref ** 2))


def energy_arrays():
    rng = np.random.default_rng(7)
    return [(rng.standard_normal(n) * s).astype(np.float32)
            for n, s in ((1, 0.5), (255, 1.0), (256, 0.1), (257, 2.0), (767, 1.0), (768, 1e-3), (769, 1.0), (1023, 1.0),
                         (1025, 3.0), (100003, 0.25))]


# ------------------------------------------------------------------------------------------------ fixtures (pack reference)
@pytest.fixture(scope="module")
def onset_ref(engine):
    ys = onset_arrays()
    return ys, {hop: run_onset(engine, engine.pack(ys), hop) for hop in (64, 512, 96)}


@pytest.fixture(scope="module")
def chroma_ref(engine):
    import torch
    ys = chroma_arrays()
    layout = engine.pack(ys)
    chroma, tun = run_chroma(engine, layout)
    tun_t = torch.tensor(tun, dtype=torch.int32)
    return ys, tun_t, (chroma, tun), run_chroma(engine, layout, tun_t)


@pytest.fixture(scope="module")
def spectral_ref(engine):
    return {sr: (spectral_arrays(sr), run_spectral(engine, engine.pack(spectral_arrays(sr)), sr)) for sr in (22050, 44100)}


@pytest.fixture(scope="module")
def trim_ref(engine):
    ys = [y for y, _ in trim_arrays()]
    layout = engine.pack(ys)
    return ys, {db: run_trim(engine, layout, db) for db in TRIM_DB}


# ------------------------------------------------------------------------------------------------ 2. placement invariance
@pytest.mark.parametrize("phase", PHASES)
@pytest.mark.parametrize("hop", [64, 512, 96])
def test_onset_placement_invariant(engine, onset_ref, hop, phase):
    """stft_logmel2_kernel<1> (hop 64), <8> (hop 512), <0> (hop 96): phases 0 and 2 run the float2 fast path inside the
    segment and load_frame_guarded at its edges, phases 1 and 3 run load_frame_guarded for every frame."""
    ys, ref = onset_ref
    assert_lists_equal(run_onset(engine, place(engine, ys, [phase] * len(ys)), hop), ref[hop])


def test_onset_mixed_phases_one_launch(engine, onset_ref):
    ys, ref = onset_ref
    phases = [i % 4 for i in range(len(ys))]
    assert_lists_equal(run_onset(engine, place(engine, ys, phases, margin=4099, seed=5), 64), ref[64])


@pytest.mark.parametrize("phase", PHASES)
def test_tuning_and_chroma_placement_invariant(engine, chroma_ref, phase):
    """Phase 0: cp.async octave 0 (clamp-free inside, zero-fill at the edges) and float2 decimation; phase 2: plain-load
    octave 0 and float2 decimation; phases 1, 3: plain-load octave 0 and the scalar decimation.  The tuning STFT takes
    the float2 path at phases 0, 2 and the scalar loop at phases 1, 3."""
    ys, tun_t, (w_chroma, w_tun), (w_chroma_given, _) = chroma_ref
    layout = place(engine, ys, [phase] * len(ys))
    chroma, tun = run_chroma(engine, layout)
    assert np.array_equal(tun, w_tun), (tun.tolist(), w_tun.tolist())
    assert np.array_equal(chroma, w_chroma), float(np.max(np.abs(chroma - w_chroma)))
    chroma_given, tun_given = run_chroma(engine, layout, tun_t)
    assert np.array_equal(tun_given, w_tun)
    assert np.array_equal(chroma_given, w_chroma_given), float(np.max(np.abs(chroma_given - w_chroma_given)))


@pytest.mark.parametrize("phase", PHASES)
@pytest.mark.parametrize("sr", [22050, 44100])
def test_spectral_placement_invariant(engine, spectral_ref, sr, phase):
    ys, ref = spectral_ref[sr]
    assert_spectral_equal(run_spectral(engine, place(engine, ys, [phase] * len(ys)), sr), ref)


@pytest.mark.parametrize("phase", PHASES)
def test_trim_placement_invariant(engine, trim_ref, phase):
    ys, ref = trim_ref
    layout = place(engine, ys, [(phase + i) % 4 for i in range(len(ys))])
    for db in TRIM_DB:
        got = run_trim(engine, layout, db)
        assert np.array_equal(got, ref[db]), (db, got.tolist(), ref[db].tolist())


@pytest.mark.parametrize("phase", PHASES)
def test_window_energy_placement_invariant(engine, phase):
    ys = energy_arrays()
    want = run_energy(engine, engine.pack(ys))
    got = run_energy(engine, place(engine, ys, [(phase + 3 * i) % 4 for i in range(len(ys))]))
    assert np.array_equal(got, want)


def xcorr_case(win, stride, n_cand, n_windows=8):
    """Windows of A and the B spans of their candidates as separate arrays (A exactly `win` samples, B exactly the
    samples the last candidate reaches), so the canary sits right next to the first A and the last B sample.  Each B
    span holds a noisy copy of its A window at candidate `truth`."""
    a_list, b_list, truth = [], [], []
    for w in range(n_windows):
        rng = np.random.default_rng(300 + w)
        a = synth.synth(310 + w, win / SR + 0.01, SR, bpm=120.0)[:win]
        b = (rng.standard_normal((n_cand - 1) * stride + win) * 0.3).astype(np.float32)
        j = int(rng.integers(0, n_cand))
        b[j * stride : j * stride + win] += a
        a_list.append(a)
        b_list.append(b)
        truth.append(j)
    return a_list, b_list, truth


@pytest.mark.parametrize("form", ["block", "direct"])
def test_xcorr_search_placement_invariant(engine, form):
    """Block form (win = 4·stride + 3: the ring kernel with 16-byte superset bulk copies) and direct form (stride =
    win // 8: one CTA per candidate).  a_pos and b_lo run through all four residues mod 4 independently."""
    from nightcore_analyzer import xcorr as nx
    win = 4015
    stride = 1003 if form == "block" else win // 8
    n_cand = 40
    a_list, b_list, truth = xcorr_case(win, stride, n_cand)
    arrays = [x for ab in zip(a_list, b_list) for x in ab]
    nc = np.full(len(a_list), n_cand, dtype=np.int32)

    def search(layout):
        audio, off, _ = layout
        bj, bc = engine.xcorr_search_dev(audio, audio, off[0::2], off[1::2], nc, win, stride, nx.XCORR_RMS_GATE)
        return engine.to_host(bj), engine.to_host(bc)

    want_j, want_c = search(engine.pack(arrays))
    assert want_j.tolist() == truth
    for w, (a, b, j) in enumerate(zip(a_list, b_list, want_j)):
        wa, wb = a.astype(np.float64), b[j * stride : j * stride + win].astype(np.float64)
        assert abs(want_c[w] - float(np.dot(wa, wb) / (np.linalg.norm(wa) * np.linalg.norm(wb)))) <= 1e-5
    for shift in PHASES:
        phases = [(w + shift) % 4 if k == 0 else (w // 4 + 3 * w + shift) % 4 for w in range(len(a_list)) for k in (0, 1)]
        got_j, got_c = search(place(engine, arrays, phases))
        assert np.array_equal(got_j, want_j) and np.array_equal(got_c, want_c), shift


# ------------------------------------------------------------------------------------------------ intro alignment
ALIGN_LENGTHS = (1, 2, 3, 4097, 100001)


@pytest.mark.parametrize("phase", PHASES)
def test_decimate2_and_rms_frames_any_base_pointer(engine, phase):
    """ncfa_decimate2 and ncfa_rms_frames take one base pointer: odd and even ones, odd and even n.  Bit-identical to
    the same data at a 256-byte aligned allocation; decimate2 within one float32 ulp of lr.decimate2(scale=False)
    (float64 sums rounded once on both sides), rms within test_gpu_io's 2e-6 of the maximum."""
    import torch
    from nightcore_analyzer._native import check, lib
    ys = [synth.synth(90 + k, n / SR + 0.01, SR, bpm=120.0)[:n] for k, n in enumerate(ALIGN_LENGTHS)]
    audio, off, ln = place(engine, ys, [(phase + i) % 4 for i in range(len(ys))])

    def dec(ptr, n):
        out = torch.empty((n + 1) // 2, dtype=torch.float32, device=engine.device)
        with torch.cuda.device(engine.device):
            check(lib.ncfa_decimate2(ptr, n, out.data_ptr(), engine._stream()), "ncfa_decimate2")
        return out.cpu().numpy()

    for y, o, n in zip(ys, off, ln):
        n = int(n)
        aligned = engine.to_dev(y)
        got = dec(audio.data_ptr() + 4 * int(o), n)
        assert np.array_equal(got, dec(aligned.data_ptr(), n)), n
        want = lr.decimate2(y, scale=False)
        assert got.shape == want.shape and np.all(np.abs(got - want) <= np.spacing(np.abs(want))), n
        rms = engine.rms_frames_dev(audio[int(o) : int(o) + n], n, 2048, 512).cpu().numpy()
        assert np.array_equal(rms, engine.rms_frames_dev(aligned, n, 2048, 512).cpu().numpy()), n
        want = lr.rms(y, 2048, 512)
        assert np.max(np.abs(rms - want)) <= 2e-6 * float(np.max(want)) + 1e-12, n


# ------------------------------------------------------------------------------------------------ 3. oracle parity at the edges
@pytest.mark.parametrize("phase", [0, 3])
@pytest.mark.parametrize("hop", [64, 512, 96])
def test_onset_oracle_at_edges(engine, onset_ref, hop, phase):
    ys, _ = onset_ref
    got = run_onset(engine, place(engine, ys, [phase] * len(ys)), hop)
    for i, (y, g) in enumerate(zip(ys, got)):
        want = lr.onset_strength(y, SR, hop)
        assert g.shape == want.shape, i
        if float(np.max(np.abs(want))) == 0.0:
            assert np.all(g == 0), i
        else:
            assert rel_err(g, want) < 1e-4, (i, rel_err(g, want))
    assert np.all(got[-1] == 0)


@pytest.mark.parametrize("phase", [0, 1])
def test_tuning_and_chroma_oracle_at_edges(engine, phase):
    import torch
    ys = chroma_arrays()
    sel = [ys[i] for i in CHROMA_ORACLE]
    layout = place(engine, sel, [phase] * len(sel))
    _, tun = run_chroma(engine, layout)
    want_t = [lr.estimate_tuning(y, SR, bins_per_octave=36) for y in sel]
    assert tun.tolist() == [tuning_index(t) for t in want_t]
    chroma, _ = run_chroma(engine, layout, torch.tensor(tun, dtype=torch.int32))
    for i, (y, t, g) in enumerate(zip(sel, want_t, chroma)):
        want = lr.chroma_cqt(y, SR, 512, 36, tuning=t).mean(axis=1)
        if float(np.max(want)) == 0.0:
            assert np.all(g == 0.0), i
        else:
            assert np.max(np.abs(g - want)) <= 1e-4 * np.max(want), (i, len(y))
    assert tun[-1] == 50 and np.all(chroma[-1] == 0.0)


def rel(a, b):
    return abs(a - b) / max(abs(b), 1e-30)


@pytest.mark.parametrize("phase", [0, 1])
@pytest.mark.parametrize("sr", [22050, 44100])
def test_spectral_oracle_at_edges(engine, sr, phase):
    """The statistics spectral.analyze_arrays derives from the kernel outputs, at the tolerances of test_gpu_spectral:
    centroid, roll-off and band means 1e-5 relative, per-bin mean dB 2e-3 dB, the effective-bandwidth bin exact."""
    from nightcore_analyzer.spectral import _BANDS
    ys = spectral_arrays(sr)
    stats, bins = run_spectral(engine, place(engine, ys, [phase] * len(ys)), sr)
    freqs = np.fft.rfftfreq(n=2048, d=1.0 / sr)
    for i, y in enumerate(ys[:-1]):
        want = port.spectral_stats(y, sr)
        n_frames = stats[i, 7]
        assert n_frames == 1 + len(y) // 512
        assert rel(stats[i, 0] / n_frames, want["centroid"]) < 1e-5, i
        assert rel(stats[i, 1] / n_frames, want["rolloff"]) < 1e-5, i
        for b, (name, (lo, hi)) in enumerate(zip(("sub_bass", "bass", "midrange", "presence", "brilliance"), _BANDS)):
            n_bins = int(np.count_nonzero((freqs >= lo) & (freqs < hi)))
            got = float(np.float32(stats[i, 2 + b] / (n_bins * n_frames))) if n_bins else 0.0
            assert rel(got, want[name]) < 1e-5, (i, name)
        assert np.max(np.abs(bins[i] - want["freq_avg_db"])) < 2e-3, i
        significant = bins[i] > (np.max(bins[i]) - 60.0)
        assert float(freqs[np.where(significant)[0][-1]]) == want["effective_bandwidth_hz"], i
    assert stats[-1, 0] == 0.0 and stats[-1, 1] == 0.0 and np.all(bins[-1] == 0.0)


def test_trim_thresholds_are_clear():
    """The kernel sums the frame energies in float64, the oracle takes a float32 mean: a frame within rounding of the
    threshold could legitimately fall on either side.  The signals keep every frame 1e-3 dB away from it."""
    for y, name in trim_arrays():
        db = oracle_trim_db(y)
        for top_db in TRIM_DB:
            assert np.min(np.abs(db + top_db)) > 1e-3, (name, top_db)


@pytest.mark.parametrize("phase", [0, 2])
def test_trim_bounds_match_oracle_batched(engine, phase):
    """Every segment in one trim_bounds_dev call per top_db: lengths around the 512-sample block and the 2048-sample
    frame, silences ending mid-block, a single spike, a 1e-6 quiet section, all zeros (the reference's quirk: (0, n))."""
    cases = trim_arrays()
    ys = [y for y, _ in cases]
    layout = place(engine, ys, [(phase + i) % 4 for i in range(len(ys))])
    for db in TRIM_DB:
        got = run_trim(engine, layout, db)
        for (y, name), g in zip(cases, got):
            _, (s, e) = lr.trim(y, db)
            assert (int(g[0]), int(g[1])) == (int(s), int(e)), (name, db, g.tolist(), (s, e))
    zeros = run_trim(engine, layout, 60.0)[-1]
    assert zeros.tolist() == [0, len(ys[-1])]


@pytest.mark.parametrize("phase", [0, 1])
def test_window_energy_matches_float64_mean(engine, phase):
    ys = energy_arrays()
    got = run_energy(engine, place(engine, ys, [(phase + i) % 4 for i in range(len(ys))]))
    for g, y in zip(got, ys):
        want = float(np.mean(y.astype(np.float64) ** 2))
        assert abs(g - want) <= 1e-12 * want, (len(y), g, want)


# ------------------------------------------------------------------------------------------------ 4. offsets above 2^31
def test_segments_above_2_31_samples(engine):
    """A batch resident in HBM puts segments past sample 2^31 (a 1000-pair batch holds ~7·10^9 samples).  The same
    segments placed after sample 2^31 + 2^20 and placed low give bit-identical results (spectral bins: one ulp, see
    assert_spectral_equal)."""
    import torch
    free, _ = torch.cuda.mem_get_info(engine.device)
    if free < 12e9:
        pytest.skip(f"needs ~9 GB of free device memory for a 2^31-sample buffer; {free / 1e9:.1f} GB free")
    ys = chroma_arrays()[6:9] + onset_arrays()[1:3] + [y for y, _ in trim_arrays()[7:9]]
    phases = [i % 4 for i in range(len(ys))]
    low = place(engine, ys, phases)
    want = (run_onset(engine, low, 512), run_chroma(engine, low), run_spectral(engine, low, SR),
            [run_trim(engine, low, db) for db in TRIM_DB], run_energy(engine, low))
    del low
    high = place(engine, ys, phases, base=2 ** 31 + 2 ** 20)
    try:
        assert int(high[1][0]) > 2 ** 31 and high[0].numel() > 2 ** 31 + 2 ** 20
        assert_lists_equal(run_onset(engine, high, 512), want[0])
        chroma, tun = run_chroma(engine, high)
        assert np.array_equal(tun, want[1][1]) and np.array_equal(chroma, want[1][0])
        assert_spectral_equal(run_spectral(engine, high, SR), want[2])
        for db, w in zip(TRIM_DB, want[3]):
            assert np.array_equal(run_trim(engine, high, db), w), db
        assert np.array_equal(run_energy(engine, high), want[4])
    finally:
        del high
        torch.cuda.synchronize(engine.device)
        torch.cuda.empty_cache()
