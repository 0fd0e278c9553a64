"""The beat tracker (beat.cu, ncfa_beat_track_batched) bit for bit against the oracle at every lag, wavefront shape,
thread form, tie and trim edge.

beat.cu runs three kernels per envelope: the float64 normalisation onset / (std(ddof=1) + tiny) with the Gaussian
window, the local score (a 4-frame register sliding window over 1024-frame shared-memory tiles, a one-frame loop at
the ends), and the DP.  The DP takes near = round(fpb / 2) frames at a time as one wavefront: every 8th frame of it
(and its last) is an anchor that scans all its predecessors with one warp, and the frames between anchors only scan
the interval the anchors leave (the monotone argmax).  Then come the radix-select median of the local maxima of the
cumulative score, the last beat, the backtrack and librosa's trim.  It runs in 64 threads when max_env_len <= 2048 and
in 512 threads otherwise.

White box.  Every call gets exactly the workspace its size query asks for, followed by a byte pattern, and a beat
buffer whose unused slots hold a pattern; the per-segment workspace is then read back.  The oracle chain
(librosa_restated.beat_track_from_norm) is run on the kernel's own normalised onsets, window and transition penalties
(the DP copies its shared-memory table into the workspace: torch cannot recompute it, because this file is built
without FMA contraction, which changes the instructions of the device log against torch's).  The local score, cumulative score,
backlinks, the backtracked path (tail first) and the beats must then be identical: ties between predecessors, which
silent frames make common, are decided by the tie rules alone (strict > inside a lane, the larger frame on equal scores
across lanes), and any other arithmetic difference shows too.

End to end.  On cases where every frame's best predecessor beats the second by at least 1e-9 relative in the
unmodified oracle (asserted on the CPU), the beats also equal beat_track_frames on the float32 envelope.

The CPU-only preconditions (each case reaches the path it is built for, decisiveness, trim thresholds clear of every
local score) are tests of their own and run without a GPU."""
import functools

import numpy as np
import pytest
import torch

from oracle import librosa_restated as lr

gpu = pytest.mark.gpu
SR = 22050
FENCE = 8192            # bytes of pattern after the workspace
PAT = 0xA5
ROW_PAT = -7            # unused beat slots, and OUT_FENCE elements after the beat and count buffers
OUT_FENCE = 16
TINY = np.finfo(np.float64).tiny
W512, W96, W64 = 344, 1837, 2756     # floor(8·sr / hop): the largest lag the tempogram returns at hop 512, 96, 64


def near_of(lag):
    return int(np.round(lag / 2.0))


def expo(seed, n):
    return np.random.default_rng(seed).exponential(1.0, n).astype(np.float32)


def backtrack(backlink, tail):
    out, n = [], int(tail)
    while n >= 0:
        out.append(n)
        n = int(backlink[n])
    return out                     # tail first, as the kernel keeps it


# ------------------------------------------------------------------------------------------------ cases
class Case:
    def __init__(self, name, env, lag, expect, e2e=False):
        self.name, self.env, self.lag, self.expect, self.e2e = name, np.asarray(env, np.float32), int(lag), expect, e2e

    def __repr__(self):
        return self.name


def has_beats(k):
    return lambda d, b: len(b) >= k and bool(np.all(np.diff(b) >= near_of(d["fpb"])))


def no_predecessor(d, b):
    return bool(np.all(d["backlink"] == -1))


SWEEP_LAGS = list(range(2, 81))
BIG_LAGS = [127, 128, 129, W512, W96, W64 - 1, W64]


def sweep_len(lag):
    return 5 * lag + lag % 11 + 2


def sweep_cases(lags):
    # random envelopes with a non-zero first frame: librosa's local score leaves onset[0] out for i <= fpb
    out = []
    for lag in lags:
        seed = 1000 + lag if lag != W96 else 7919 + W96
        out.append(Case(f"sweep-lag{lag}", expo(seed, sweep_len(lag)), lag, has_beats(3), e2e=lag < W64 - 1))
    return out


def length_cases():
    out = []
    for lag in (7, 20, 64):
        nr = near_of(lag)
        for n in sorted({2, 3, nr - 1, nr, nr + 1, lag, 2 * lag, 2 * lag + 1}):
            if n >= 2:
                out.append(Case(f"len{n}-lag{lag}", expo(10 * lag + n, n), lag,
                                no_predecessor if n <= nr else has_beats(1), e2e=True))
    for lag in (5, 600):                 # at fpb >= 512 the window is wider than the 1024-frame score tile
        for k in (1, 2, 4):
            for dn in (-1, 0, 1, 2, 3):
                n = 1024 * k + dn
                out.append(Case(f"len{n}-lag{lag}", expo(lag + n, n), lag, has_beats(2 if lag == 600 else 3),
                                e2e=True))
    return out


def leading_silence():
    e = expo(11, 2000)
    e[:300] = 0.0
    return e


def trailing_silence():
    e = expo(2, 2000)
    e[-400:] = 0.0
    return e


def silent_middle(seed):
    e = expo(40 + seed, 1500)
    e[400 + 50 * seed : 900 + 50 * seed] = 0.0
    return e


def clicks():
    return (np.random.default_rng(3).random(3000) < 0.05).astype(np.float32)


def rounded():
    return np.round(expo(4, 3000))


def spike():
    e = np.zeros(1500, np.float32)
    e[517] = 3.0
    return e


def spike_at_frame_0():
    e = np.zeros(500, np.float32)
    e[0] = 2.0
    return e


def local_max_values(d):
    return d["cumscore"][lr.localmax(d["cumscore"])]


def first_scored(d):
    return int(np.argmax(d["localscore"] >= 0.01 * d["localscore"].max()))


def ties_on_path(d, b):
    path = backtrack(d["backlink"], d["tail"])
    return bool(np.any(d["margin"][path] == 0.0))


def anchor_lane_tie_changed(d, b=None):
    """Replay of the DP's phase A on the debug output: True when an anchor at or after `first` has its best score at
    two predecessors of one lane (32·k frames apart), so that a lane keeping its farthest maximum instead of its nearest
    would change the anchor's backlink.  Only such a case tests the strict > of the lane scan."""
    cum, pen, n, fpb = d["cumscore"], d["pen"], len(d["cumscore"]), int(d["fpb"])
    near, far, first = near_of(fpb), 2 * fpb, first_scored(d)
    for base in range(0, n, near):
        nf = min(near, n - base)
        for j in sorted(set(range(0, nf, 8)) | {nf - 1}):
            i = base + j
            lo, hi = max(0, i - far), i - near
            if i < first or hi - lo < 32:
                continue
            locs = np.arange(hi, lo - 1, -1)
            sc = cum[locs] - pen[i - locs - near]
            t = locs[sc == sc.max()]
            lanes = (i - near - t) % 32
            if max(t[lanes == l].min() for l in set(lanes.tolist())) != t.max():
                return True
    return False


def same_lane_tie():
    # spikes at q, q + 98 and q + 162 at fpb = 126: pen(98) = pen(162) (98·162 = 126²), so frames q + 98 and q + 162
    # get the same cumulative score from q, and the anchor 512 = q + 260 finds both, 64 frames apart, as its best
    e = np.zeros(3000, np.float32)
    e[[252, 350, 414]] = 1.0
    return e


def upper_median_moves_tail(d, b=None):
    """An even number of local maxima, and the threshold half the UPPER middle value (instead of half the mean of the
    two middle values) would pick another last beat."""
    c = d["cumscore"]
    m = lr.localmax(c)
    v = np.sort(c[m])
    if len(v) == 0 or len(v) % 2:
        return False
    late = np.flatnonzero(m & (c >= 0.5 * v[len(v) // 2]))
    return (late[-1] if len(late) else len(c) - 1) != d["tail"]


def short_burst():
    # two local maxima: the burst (cum ≈ 10.2) and the last frame (≈ 4.2, compared with itself), which clears half the
    # median (3.6) but not half the upper value (5.1)
    e = np.zeros(57, np.float32)
    e[2:4] = 1.0
    return e


SHAPE_CASES = [
    # first > 0: the frames before the first one whose local score reaches 1 % of the maximum get no backlink
    ("leading-silence", leading_silence, 20,
     lambda d, b: first_scored(d) > 250 and bool(np.all(d["backlink"][: first_scored(d)] == -1))
     and d["backlink"][first_scored(d)] >= 0 and b[0] >= first_scored(d)),
    # the path runs on through the silence and the trim cuts it back
    ("trailing-silence", trailing_silence, 20,
     lambda d, b: backtrack(d["backlink"], d["tail"])[0] >= 1600 and b[-1] < 1600),
    # duplicate local-maximum values, an even and an odd number of local maxima
    ("silent-middle-even", lambda: silent_middle(0), 20,
     lambda d, b: len(np.unique(local_max_values(d))) < len(local_max_values(d)) and len(local_max_values(d)) % 2 == 0),
    ("silent-middle-odd", lambda: silent_middle(3), 20,
     lambda d, b: len(np.unique(local_max_values(d))) < len(local_max_values(d)) and len(local_max_values(d)) % 2 == 1),
    # exact ties between predecessors on the beat path
    ("clicks-lag20", clicks, 20, ties_on_path),
    ("clicks-lag7", clicks, 7, ties_on_path),
    ("rounded-lag2", rounded, 2, ties_on_path),
    ("rounded-lag5", rounded, 5, ties_on_path),
    ("rounded-lag7", rounded, 7, ties_on_path),
    ("spike", spike, 30, lambda d, b: len(b) == 1 and b[0] == 517),
    # librosa's loop bound leaves onset[0] out of every frame's local score (frame fpb is the first whose window reaches
    # it, and the tap is excluded there): ls is all zero.  At fpb = 20 frame 20 starts a 4-frame group of the kernel's
    # sliding window, so the fast path must not begin there.
    ("spike-at-frame-0", spike_at_frame_0, 20, lambda d, b: d["localscore"].max() == 0.0 and len(b) == 0),
    ("same-lane-tie-lag126", same_lane_tie, 126, anchor_lane_tie_changed),
    ("last-frame-median-lag69", short_burst, 69, upper_median_moves_tail),
    # max(ls) = 0: score and trim thresholds are 0, the local maxima of cum are <= 0, no beats
    ("all-zero", lambda: np.zeros(500, np.float32), 20,
     lambda d, b: d["localscore"].max() == 0.0 and d["threshold"] == 0.0 and local_max_values(d).max() <= 0.0
     and len(b) == 0),
]


def shape_cases():
    return [Case(name, make(), lag, expect) for name, make, lag, expect in SHAPE_CASES]


def long_case():
    # the one hop-64-sized envelope: 100 000 frames at the hop-64 tempogram's largest lag
    return Case("len100000-lag2756", expo(64, 100000), W64, has_beats(10))


def all_cases():
    return sweep_cases(SWEEP_LAGS) + sweep_cases(BIG_LAGS) + length_cases() + shape_cases() + [long_case()]


@functools.lru_cache(maxsize=None)
def case_by_name():
    return {c.name: c for c in all_cases()}


@functools.lru_cache(maxsize=None)
def oracle_run(name):
    """beat_track_frames (unmodified oracle, CPU float64 exp / log) on the case's float32 envelope → (beats, debug)."""
    c = case_by_name()[name]
    return lr.beat_track_frames(c.env, 60.0 * SR / (512 * float(c.lag)), SR, 512, return_debug=True)


# ------------------------------------------------------------------------------------------------ CPU preconditions
def test_sweep_covers_wavefront_shapes():
    """near < 8, = 8, = 9 and multiples of 8; fpb = 1 and 3 mod 4 (np.round's half to even); ragged last wavefronts."""
    nears = {near_of(l) for l in SWEEP_LAGS + BIG_LAGS}
    assert {1, 2, 3, 7, 8, 9, 16, 24, 32, 40} <= nears
    assert {l % 4 for l in SWEEP_LAGS} == {0, 1, 2, 3}
    assert near_of(5) == 2 and near_of(7) == 4 and near_of(9) == 4 and near_of(11) == 6     # half to even
    assert len({sweep_len(l) % near_of(l) for l in SWEEP_LAGS if near_of(l) > 4}) >= 6
    assert max(BIG_LAGS) == W64 and sweep_len(W64) > 4096


@pytest.mark.parametrize("case", all_cases(), ids=repr)
def test_case_reaches_its_path(case):
    beats, d = oracle_run(case.name)
    assert case.expect(d, beats), (case.name, beats[:20])


def test_end_to_end_cases_are_decisive():
    """Where the kernel and the oracle may differ in the last bits of exp, log and the std, an end-to-end comparison is
    only meaningful if no decision is within rounding: every predecessor choice wins by 1e-9 relative, no local score
    is within 1e-12 of the 1 % score threshold, no two neighbouring cumulative scores (is_localmax) and no local maximum
    and half the median (the last beat) are within 1e-9 of the largest |cum|."""
    for c in all_cases():
        if not c.e2e:
            continue
        d = oracle_run(c.name)[1]
        assert float(d["margin"].min()) >= 1e-9, (c.name, float(d["margin"].min()))
        ls, cum = d["localscore"], d["cumscore"]
        assert float(np.min(np.abs(ls - 0.01 * ls.max()))) > 1e-12 * ls.max(), c.name
        scale = float(np.max(np.abs(cum)))
        if len(cum) > 1:
            assert float(np.min(np.abs(np.diff(cum)))) > 1e-9 * scale, c.name
        v = local_max_values(d)
        if len(v):
            assert float(np.min(np.abs(v - 0.5 * d["median"]))) > 1e-9 * scale, c.name


def test_trim_thresholds_are_clear():
    """numpy sums the trim threshold's mean pairwise, the device sequentially: no local score may lie within 1e-12
    relative of the threshold (unless it is exactly 0, where both sides compute 0)."""
    for c in all_cases():
        d = oracle_run(c.name)[1]
        thr = float(d["threshold"])
        if thr != 0.0:
            assert float(np.min(np.abs(d["localscore"] - thr))) > 1e-12 * thr, c.name


def test_beat_count_check_raises_on_overflow(monkeypatch):
    """A count of −1 (more beats than max_beats) raises at every host reader instead of reading as "too few beats"."""
    from fake_engine import FakeEngine
    from nightcore_analyzer import _engine, _native, io as nio, tempo as ntempo

    class Overflowing(FakeEngine):
        """The oracle's results, except that the last segment of every call at `hop` reports −1 beats."""
        def __init__(self, hop):
            super().__init__()
            self.hop, self.calls = hop, 0

        def tempo_segments_dev(self, audio, seg_off, seg_len, start_bpm, hop, sr):
            out = list(super().tempo_segments_dev(audio, seg_off, seg_len, start_bpm, hop, sr))
            if hop == self.hop:
                self.calls += 1
                out[5] = out[5].clone()
                out[5][-1] = -1
            return tuple(out)

    assert _engine.check_beat_counts(np.array([0, 4, 7], np.int32)).tolist() == [0, 4, 7]
    with pytest.raises(_native.NcfaError, match="beat buffer overflow"):
        _engine.check_beat_counts(np.array([3, -1], np.int32))
    from nightcore_analyzer import batch
    from oracle import synth
    src, nc = synth.make_pair(1000, 45.0, SR)
    for hop in (512, 64):        # batch.py: the window pass (source windows first), then the hop-64 whole-track pass
        eng = Overflowing(hop)
        monkeypatch.setattr(_engine, "get_engine", lambda device=None: eng)
        if hop == 512:
            with pytest.raises(_native.NcfaError, match="beat buffer overflow"):
                ntempo.batch_estimate_tempo(nio.slice_windows(src, SR))
            assert eng.calls == 1
        audio, off, ln = eng.pack([nc, src])
        st = batch.StagedBatch(audio=audio, off=off, length=ln.astype(np.int64), sr=SR, h2d_bytes=0)
        eng.calls = 0
        with pytest.raises(_native.NcfaError, match="beat buffer overflow"):
            batch.analyse_staged(st, compute_pitch=False)
        assert eng.calls == 1


# ------------------------------------------------------------------------------------------------ ABI helper
def align256(n):
    return (n + 255) // 256 * 256


def run_beats(engine, envs, lags, max_env_len=None, max_lag=None, max_beats=None):
    """One ncfa_beat_track_batched call with explicit maxima, exactly the workspace its size query gives (then a
    pattern) and a pattern-filled beat buffer → (n_beats, list of per-segment dicts read back from the workspace)."""
    from nightcore_analyzer._native import check, lib
    n = len(envs)
    lens = np.array([len(e) for e in envs], np.int32)
    S = int(max_env_len if max_env_len is not None else max(1, lens.max()))
    L = int(max_lag if max_lag is not None else max(lags))
    MB = int(max_beats if max_beats is not None else S // 2 + 2)
    off = np.zeros(n, np.int64)
    off[1:] = np.cumsum(lens[:-1] + 3)          # a few frames of padding between envelopes
    host = np.full(int(off[-1]) + int(lens[-1]) + 3, 1e30, np.float32)
    for e, o in zip(envs, off):
        host[o : o + len(e)] = e
    dev = engine.device
    onset = torch.from_numpy(host).to(dev)
    d_off, d_len = torch.from_numpy(off).to(dev), torch.from_numpy(lens).to(dev)
    d_lag = torch.from_numpy(np.asarray(lags, np.int32)).to(dev)
    need = lib.ncfa_beat_workspace_bytes(n, S, L)
    K = 2 * L + 1
    F = 3 * S + 2 * K + 8                       # float64 per segment: onorm | ls | cum | window[K] | pen[K] | 8 spare
    f64_bytes = align256(n * F * 8)
    assert f64_bytes + align256(n * 2 * S * 4) == need, "the test's workspace layout has drifted from beat_ws"
    ws = torch.full((need + FENCE,), PAT, dtype=torch.uint8, device=dev)
    beats = torch.full((n * MB + OUT_FENCE,), ROW_PAT, dtype=torch.int32, device=dev)
    n_beats = torch.full((n + OUT_FENCE,), ROW_PAT, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    with torch.cuda.device(dev):
        check(lib.ncfa_beat_track_batched(onset.data_ptr(), d_off.data_ptr(), d_len.data_ptr(), n, S, d_lag.data_ptr(),
                                          L, beats.data_ptr(), MB, n_beats.data_ptr(), ws.data_ptr(), need,
                                          torch.cuda.current_stream().cuda_stream), "ncfa_beat_track_batched")
    torch.cuda.synchronize()
    assert bool((ws[need:] == PAT).all()), "the beat tracker wrote past ncfa_beat_workspace_bytes"
    assert bool((beats[n * MB :] == ROW_PAT).all()) and bool((n_beats[n:] == ROW_PAT).all())
    nb = n_beats[:n].cpu().numpy()
    rows = beats[: n * MB].view(n, MB).cpu().numpy()
    f64 = ws[:f64_bytes].view(torch.float64).cpu().numpy()
    i32 = ws[f64_bytes:need].view(torch.int32).cpu().numpy()
    segs = []
    for s in range(n):
        N, b = int(lens[s]), nb[s]
        row = rows[s]
        assert b >= -1
        written = MB if b < 0 else b
        assert np.all(row[written:] == ROW_PAT), f"segment {s} wrote past its beats"
        base = s * F
        segs.append(dict(n_beats=int(b), beats=row[:written].copy(), onorm=f64[base : base + N],
                         ls=f64[base + S : base + S + N], cum=f64[base + 2 * S : base + 2 * S + N],
                         window=f64[base + 3 * S : base + 3 * S + 2 * int(lags[s]) + 1],
                         pen=f64[base + 3 * S + K : base + 3 * S + K + 2 * int(lags[s]) - near_of(lags[s]) + 1],
                         backlink=i32[s * 2 * S : s * 2 * S + N], path=i32[s * 2 * S + S : s * 2 * S + S + N]))
    return nb, segs


def device_window(engine, lag):
    """The Gaussian window in float64 by torch on the device, in beat.cu's operation order.  The divisor is a device
    tensor: torch multiplies by the reciprocal when it divides by a Python scalar."""
    dev = engine.device
    k = torch.arange(2 * lag + 1, dtype=torch.float64, device=dev)
    a = ((k - float(lag)) * 32.0) / torch.tensor(float(lag), dtype=torch.float64, device=dev)
    return torch.exp(-0.5 * (a * a)).cpu().numpy()


def check_white_box(engine, case, seg):
    """The kernel's workspace and beats against the oracle chain run on the kernel's own onorm, window and penalty."""
    env64 = case.env.astype(np.float64)
    want_norm = env64 / (env64.std(ddof=1) + TINY)
    scale = float(np.max(np.abs(want_norm)))
    assert float(np.max(np.abs(seg["onorm"] - want_norm))) <= 1e-14 * scale, case.name
    assert np.array_equal(device_window(engine, case.lag), seg["window"]), (case.name, "torch's exp differs")
    dd = np.arange(near_of(case.lag), 2 * case.lag + 1, dtype=np.float64)
    want_pen = 100.0 * (np.log(dd) - np.log(float(case.lag))) ** 2
    assert np.all(np.abs(seg["pen"] - want_pen) <= 1e-12 * (1.0 + want_pen)), (case.name, "penalty table")
    beats, d = lr.beat_track_from_norm(seg["onorm"].copy(), case.lag, window=seg["window"].copy(),
                                       pen=seg["pen"].copy())
    assert np.array_equal(seg["ls"], d["localscore"]), (case.name, np.flatnonzero(seg["ls"] != d["localscore"])[:8])
    assert np.array_equal(seg["cum"], d["cumscore"]), (case.name, np.flatnonzero(seg["cum"] != d["cumscore"])[:8])
    assert np.array_equal(seg["backlink"], d["backlink"]), (case.name,
                                                             np.flatnonzero(seg["backlink"] != d["backlink"])[:8])
    path = backtrack(d["backlink"], d["tail"])
    assert seg["path"][: len(path)].tolist() == path, (case.name, "tail / backtrack")
    assert seg["n_beats"] == len(beats) and seg["beats"].tolist() == beats.tolist(), case.name
    assert case.expect(d, beats), (case.name, "the kernel's own arithmetic leaves the intended path")
    return d


def check_end_to_end(case, seg):
    if case.e2e:
        assert seg["beats"].tolist() == oracle_run(case.name)[0].tolist(), case.name


def run_cases(engine, cases, **abi):
    nb, segs = run_beats(engine, [c.env for c in cases], [c.lag for c in cases], **abi)
    out = []
    for c, seg in zip(cases, segs):
        out.append(check_white_box(engine, c, seg))
        check_end_to_end(c, seg)
    return segs, out


# ------------------------------------------------------------------------------------------------ GPU tests
@gpu
def test_lag_sweep_64_threads(engine):
    """Every lag 2..80 in one launch of the 64-thread form (max_env_len <= 2048)."""
    cases = sweep_cases(SWEEP_LAGS)
    assert max(len(c.env) for c in cases) <= 2048
    run_cases(engine, cases, max_lag=80)


@gpu
def test_lag_sweep_large_lags(engine):
    """Lags around 128, the tempogram maxima at hop 512, 96 and 64 (ring and shared-memory sizing at max_lag = 2756)."""
    run_cases(engine, sweep_cases(BIG_LAGS), max_lag=W64)


@gpu
def test_lengths(engine):
    """N = 2, 3, near ± 1, fpb, 2·fpb, 2·fpb + 1, and N = 1024·k − 1 .. 1024·k + 3 around the score tiles, at a small
    fpb and at fpb = 600 (window wider than a tile)."""
    cases = length_cases()
    run_cases(engine, [c for c in cases if len(c.env) <= 2048], max_lag=W64)       # 64 threads
    run_cases(engine, [c for c in cases if len(c.env) > 2048], max_lag=W64)


@gpu
def test_shapes(engine):
    """Leading and trailing silence, silent middles, clicks and rounded envelopes with ties on the path, one spike,
    the all-zero envelope: all in the 512-thread form, those of up to 2048 frames in the 64-thread form too."""
    cases = shape_cases()
    segs, _ = run_cases(engine, cases, max_lag=W512, max_env_len=4096)
    short = [k for k, c in enumerate(cases) if len(c.env) <= 2048]
    assert len(short) >= 6
    segs64, _ = run_cases(engine, [cases[k] for k in short], max_lag=W512, max_env_len=2048)
    for k, s in zip(short, segs64):
        same(segs[k], s, cases[k].name)


@gpu
def test_hop64_sized_envelope(engine):
    run_cases(engine, [long_case()], max_lag=W64)


# ---- invariance, bitwise and independent of the oracle
FIELDS = ("onorm", "ls", "cum", "backlink", "beats")


def same(a, b, what):
    assert a["n_beats"] == b["n_beats"], what
    for f in FIELDS:
        assert np.array_equal(a[f], b[f]), (what, f)


def invariance_set():
    return [Case("inv-a", expo(501, 1500), 23, None), Case("inv-b", expo(502, 333), 8, None),
            Case("inv-c", clicks()[:2000], 20, None), Case("inv-d", expo(504, 1999), 64, None),
            Case("inv-e", rounded()[:900], 5, None)]


@gpu
def test_alone_and_at_every_batch_position(engine):
    cases = invariance_set()
    alone = [run_beats(engine, [c.env], [c.lag], max_env_len=2000, max_lag=W512)[1][0] for c in cases]
    for r in range(len(cases)):
        order = cases[r:] + cases[:r]
        _, segs = run_beats(engine, [c.env for c in order], [c.lag for c in order], max_env_len=2000, max_lag=W512)
        for c, s in zip(order, segs):
            same(alone[cases.index(c)], s, (c.name, r))


@gpu
def test_thread_form_and_max_lag_do_not_change_results(engine):
    cases = invariance_set()
    envs, lags = [c.env for c in cases], [c.lag for c in cases]
    _, ref = run_beats(engine, envs, lags, max_env_len=2048, max_lag=max(lags))        # 64 threads
    for S, L in ((2049, max(lags)), (2048, W512), (4096, W64), (2048, W64)):
        _, segs = run_beats(engine, envs, lags, max_env_len=S, max_lag=L)
        for c, a, b in zip(cases, ref, segs):
            same(a, b, (c.name, S, L))
    for c in cases:                                                                  # max_lag = lag exactly
        _, segs = run_beats(engine, [c.env], [c.lag], max_env_len=2048, max_lag=c.lag)
        same(ref[cases.index(c)], segs[0], (c.name, "max_lag = lag"))


@gpu
def test_scaling_by_powers_of_two(engine):
    """x·2^k gives the same onorm bit for bit, hence the same ls, cum, backlinks and beats."""
    cases = invariance_set()
    envs, lags = [c.env for c in cases], [c.lag for c in cases]
    _, ref = run_beats(engine, envs, lags, max_lag=W512)
    for k in (-20, 7):
        scaled = [(e.astype(np.float64) * 2.0 ** k).astype(np.float32) for e in envs]
        assert all(np.array_equal(s.astype(np.float64) / 2.0 ** k, e) for s, e in zip(scaled, envs))
        _, segs = run_beats(engine, scaled, lags, max_lag=W512)
        for c, a, b in zip(cases, ref, segs):
            same(a, b, (c.name, k))


# ---- contract
@gpu
def test_inadmissible_segments_give_zero_beats(engine):
    """lag < 2, lag > max_lag, N < 2: n_beats = 0 and the row is not written; the neighbours are unaffected."""
    good = expo(600, 700)
    envs = [good, good, good, good, expo(601, 1), np.zeros(0, np.float32), good]
    lags = [20, 0, 1, 41, 20, 20, 20]
    nb, segs = run_beats(engine, envs, lags, max_env_len=700, max_lag=40)
    assert nb.tolist()[1:6] == [0, 0, 0, 0, 0]
    for s in segs[1:6]:
        assert len(s["beats"]) == 0            # and run_beats checked the row still holds its pattern
    assert nb[0] > 3 and segs[0]["beats"].tolist() == segs[6]["beats"].tolist()


@gpu
def test_beat_count_at_and_past_max_beats(engine):
    """A count equal to max_beats comes back as is; one more is flagged −1 with the first max_beats beats in the row
    and the next row untouched."""
    c = sweep_cases([9])[0]
    env, lag = c.env, c.lag
    want = oracle_run(c.name)[0]
    n = len(want)
    assert n >= 4
    nb, segs = run_beats(engine, [env, env], [lag, 0], max_lag=lag, max_beats=n)
    assert nb.tolist() == [n, 0] and segs[0]["beats"].tolist() == want.tolist()
    nb, segs = run_beats(engine, [env, env], [lag, 0], max_lag=lag, max_beats=n - 1)
    assert nb.tolist() == [-1, 0] and segs[0]["beats"].tolist() == want[: n - 1].tolist()


@gpu
def test_engine_raises_on_beat_overflow(engine):
    """Engine.beat_frames at hop 512 sizes its rows with max_beats_for (502 for 2000 frames): lag 2 (996 beats) and
    lag 3 (663) overflow and raise, lag 4 (499) fits."""
    from nightcore_analyzer import _native
    env = np.random.default_rng(1).exponential(1.0, 2000).astype(np.float32)
    assert engine.max_beats_for(2000, 512, SR) == 502
    for lag in (2, 3):
        with pytest.raises(_native.NcfaError, match="beat buffer overflow"):
            engine.beat_frames([env], [lag], hop=512, sr=SR)
    got = engine.beat_frames([env], [4], hop=512, sr=SR)[0]
    assert len(got) == 499
    assert got.tolist() == lr.beat_track_frames(env, 60.0 * SR / (512 * 4.0), SR, 512).tolist()
