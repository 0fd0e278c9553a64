"""CPU: the algebraic identities the CUDA kernels are built on, checked in numpy against the plain definitions
(the kernels themselves are compared with the oracle on the GPU; these pin the mathematics they restate)."""
import numpy as np


def test_real_fft_unpack_identity():
    """stft_core.cuh PostStage: a 2048-point real FFT as a packed 1024-point complex FFT.  With z[n] = x[2n] + i x[2n+1],
    Z = FFT_1024(z), E = (Z[k] + conj Z[N-k]) / 2, O = (Z[k] - conj Z[N-k]) / (2i), W = exp(-2 pi i k / 2048):
    X[k] = E + W O and X[1024-k] = conj(E - W O) for k = 0..511, X[512] = conj(Z[512])."""
    rng = np.random.default_rng(1)
    x = rng.standard_normal(2048)
    X = np.fft.rfft(x)
    Z = np.fft.fft(x[0::2] + 1j * x[1::2])
    k = np.arange(512)
    Zc = np.conj(Z[(1024 - k) % 1024])
    E = 0.5 * (Z[k] + Zc)
    O = (Z[k] - Zc) / 2j
    W = np.exp(-2j * np.pi * k / 2048)
    assert np.max(np.abs(E + W * O - X[k])) < 1e-10
    assert np.max(np.abs(np.conj(E - W * O) - X[1024 - k])) < 1e-10
    assert abs(np.conj(Z[512]) - X[512]) < 1e-10
    # the kernel stores |.|^2 only, so conj / no conj is immaterial there
    assert abs(abs(Z[512]) ** 2 - abs(X[512]) ** 2) < 1e-9


def test_four_step_fft_identity():
    """stft_core.cuh: 1024 = 32 x 32.  Lane n2 holds z[32 n1 + n2]; FFT_32 over n1, multiply by W_1024^(k1 n2),
    transpose, FFT_32 over n2 gives Z[k1 + 32 k2]."""
    rng = np.random.default_rng(2)
    z = rng.standard_normal(1024) + 1j * rng.standard_normal(1024)
    a = z.reshape(32, 32)                       # a[n1, n2]
    b = np.fft.fft(a, axis=0)                   # b[k1, n2]
    b = b * np.exp(-2j * np.pi * np.outer(np.arange(32), np.arange(32)) / 1024)
    c = np.fft.fft(b, axis=1)                   # c[k1, k2]
    Z = np.fft.fft(z)
    k1, k2 = np.meshgrid(np.arange(32), np.arange(32), indexing="ij")
    assert np.max(np.abs(c - Z[k1 + 32 * k2])) < 1e-9


def test_block_partial_initial_sums_identity():
    """tempo.cu tg_r0_kernel: S(f) = sum_{J<W} z[f+J] e^{i theta J} assembled from 32-sample block partials
    P[b] = sum_{j<32} z[32 b + j] e^{i theta j}:  S(32 t) = sum_{m < W//32} e^{i theta 32 m} P[t + m] + tail."""
    rng = np.random.default_rng(3)
    W = 2756
    z = rng.exponential(1.0, 32 * 40 + W + 64)
    theta = 2 * np.pi / W
    nb = len(z) // 32
    j = np.arange(32)
    for harm in (1, 2):
        P = np.array([np.sum(z[32 * b : 32 * b + 32] * np.exp(1j * harm * theta * j)) for b in range(nb)])
        for t in (0, 3, 39):
            f = 32 * t
            direct = np.sum(z[f : f + W] * np.exp(1j * harm * theta * np.arange(W)))
            M = W // 32
            s = sum(np.exp(1j * harm * theta * 32 * m) * P[t + m] for m in range(M))
            J = np.arange(32 * M, W)
            s += np.sum(z[f + J] * np.exp(1j * harm * theta * J))
            assert abs(s - direct) < 1e-9 * abs(direct)


def test_halfband_even_taps_hit_odd_samples():
    """chroma.cu decimate2_kernel: a 127-tap half-band FIR has zeros at every even offset from the centre (index 63),
    i.e. only h[63] and the even indices h[0], h[2], ... are non-zero; out[t] = sum_i h[i] x[2t + 63 - i] then reads
    the even input sample 2t once (centre tap) and odd input samples otherwise."""
    from oracle import librosa_restated as lr
    h = lr.halfband_fir()
    assert len(h) == 127
    odd_idx = np.arange(1, 127, 2)
    odd_idx = odd_idx[odd_idx != 63]
    assert np.max(np.abs(h[odd_idx])) < 1e-15 * np.max(np.abs(h)) + 1e-17
    x = np.random.default_rng(4).standard_normal(4000)
    full = np.convolve(x, h)[63::2][:1900]                 # centred 2:1 decimation
    t = np.arange(200, 1700)
    he = h[0::2]                                            # 64 even-index taps
    mine = h[63] * x[2 * t] + np.array([np.sum(he * x[2 * tt + 63 - 2 * np.arange(64)]) for tt in t])
    assert np.max(np.abs(mine - full[t])) < 1e-12


def _beat_dp_full_scan(ls, fpb):
    """librosa's numba DP loop (nearest predecessor first, strict >) as beat.cu's <MONO = false> runs it."""
    n = len(ls)
    near, far = int(np.rint(fpb / 2.0)), 2 * fpb
    logf = np.log(float(fpb))
    pen = np.array([100.0 * (np.log(float(d)) - logf) ** 2 for d in range(near, far + 1)])
    cum, back = np.zeros(n), np.full(n, -1, np.int64)
    for i in range(n):
        best, bl = -np.inf, -1
        for loc in range(i - near, i - far - 1, -1):
            if loc < 0:
                break
            sc = cum[loc] - pen[i - loc - near]
            if sc > best:
                best, bl = sc, loc
        cum[i] = ls[i] + best if bl >= 0 else ls[i]
        back[i] = bl
    return cum, back


def _beat_dp_monotone(ls, fpb, stride=8):
    """beat.cu <MONO = true>: per wavefront of `near` frames, every stride-th frame (and the last) gets the full scan; a
    frame between two anchors scans only [best(anchor before), best(anchor after)]."""
    n = len(ls)
    near, far = int(np.rint(fpb / 2.0)), 2 * fpb
    logf = np.log(float(fpb))
    pen = np.array([100.0 * (np.log(float(d)) - logf) ** 2 for d in range(near, far + 1)])
    cum, back = np.zeros(n), np.full(n, -1, np.int64)

    def scan(i, lo, hi):
        best, bl = -np.inf, -1
        for loc in range(hi, lo - 1, -1):
            sc = cum[loc] - pen[i - loc - near]
            if sc > best:
                best, bl = sc, loc
        return best, bl

    evaluations = 0
    for base in range(0, n, near):
        nf = min(near, n - base)
        anchors = sorted(set(list(range(0, nf, stride)) + [nf - 1]))
        wloc = {}
        for j in anchors:
            i = base + j
            lo, hi = max(0, i - far), i - near
            best, bl = scan(i, lo, hi) if hi >= lo else (-np.inf, -1)
            evaluations += max(0, hi - lo + 1)
            wloc[j] = bl
            cum[i] = ls[i] + best if bl >= 0 else ls[i]
            back[i] = bl
        for j in range(nf):
            if j in wloc:
                continue
            i = base + j
            ja = (j // stride) * stride
            jb = min(ja + stride, nf - 1)
            lo, hi = max(0, i - far), i - near
            if wloc[ja] >= 0:
                lo = max(lo, wloc[ja])
            if wloc[jb] >= 0:
                hi = min(hi, wloc[jb])
            best, bl = scan(i, lo, hi) if hi >= lo else (-np.inf, -1)
            evaluations += max(0, hi - lo + 1)
            cum[i] = ls[i] + best if bl >= 0 else ls[i]
            back[i] = bl
    return cum, back, evaluations


def test_beat_dp_monotone_argmax_equals_full_scan():
    """beat.cu: the transition penalty 100·ln²(d / fpb) is strictly convex on the search window d <= 2·fpb, so the
    score matrix cum[loc] − pen(i − loc) is inverse-Monge and the winning predecessor (max score, ties to the nearest)
    never moves backwards from one frame to the next.  The restricted search must therefore reproduce the full scan
    bit for bit — cumulative scores AND backlinks — including on quantised scores full of exact ties."""
    rng = np.random.default_rng(7)
    total_full = total_mono = 0
    for case in range(12):
        fpb = int(rng.integers(6, 60))
        n = int(rng.integers(5 * fpb, 14 * fpb))
        ls = rng.gamma(0.6, 2.0, n)                      # spiky local scores, like a normalised onset envelope
        if case % 3 == 1:
            ls = np.round(ls)                            # exact ties between candidates
        if case % 3 == 2:
            ls[:] = 0.0                                   # all ties: every frame must still pick its nearest maximum
            ls[:: max(1, fpb)] = 5.0
        cum_a, back_a = _beat_dp_full_scan(ls, fpb)
        cum_b, back_b, ev = _beat_dp_monotone(ls, fpb)
        assert np.array_equal(back_a, back_b), (case, fpb)
        assert np.array_equal(cum_a, cum_b), (case, fpb)
        near, far = int(np.rint(fpb / 2.0)), 2 * fpb
        total_full += sum(max(0, min(i - near, i) - max(0, i - far) + 1) for i in range(n) if i - near >= 0)
        total_mono += ev
    assert total_mono < 0.6 * total_full                  # and it is much less work (≈ 5x at hop-64 sizes)


def test_beat_spacing_bounds_the_beat_count():
    """Every predecessor lies at least round(lag / 2) frames back, so consecutive beats are at least that far apart and
    an envelope of N frames has at most N // round(k_min / 2) + 2 beats for every lag >= k_min, the smallest lag the
    tempogram can return (bpm < 320).  That is Engine.max_beats_for, the row size of the beat buffer: with it the
    kernel's overflow flag (a count of −1) cannot be reached from the pipeline.  Checked on the oracle for every lag
    from k_min to k_min + 40 and a geometric sample up to the tempogram's largest lag, at hops 64, 96 and 512."""
    import os
    import __graft_entry__ as ge
    if not os.path.exists(ge.LIB):
        ge._build_native()
    from nightcore_analyzer._engine import Engine
    from oracle import librosa_restated as lr
    sr = 22050
    for hop in (64, 96, 512):
        W = int(np.floor(8.0 * sr / hop))
        k_min = next(k for k in range(1, W) if 60.0 * sr / (hop * k) < 320.0)
        lags = sorted(set(range(k_min, k_min + 41)) | {int(v) for v in np.geomspace(k_min + 41, W, 8)})
        assert lags[-1] == W
        for lag in lags:
            n = 3000 + lag % 7
            env = np.random.default_rng(hop + lag).exponential(1.0, n).astype(np.float32)
            beats = lr.beat_track_frames(env, 60.0 * sr / (hop * float(lag)), sr, hop)
            assert len(beats) >= 2 and np.all(np.diff(beats) >= int(np.round(lag / 2.0))), (hop, lag)
            assert len(beats) <= Engine.max_beats_for(n, hop, sr), (hop, lag, len(beats))


def test_xcorr_block_decomposition_identity():
    """xcorr.cu: with stride = win // 4 the candidate at position j·stride is B blocks j..j+3 (+ a tail of win − 4·stride
    samples): dot(wa, wb_j) = D[0][j] + D[1][j+1] + D[2][j+2] + D[3][j+3] + tail, ‖wb_j‖² = S[j] + … + S[j+3] + tail."""
    rng = np.random.default_rng(11)
    win, n_cand = 1003, 9
    stride = win // 4
    a = rng.standard_normal(win)
    b = rng.standard_normal((n_cand - 1) * stride + win)
    nb = n_cand + 3
    D = np.array([[np.dot(a[q * stride:(q + 1) * stride], b[m * stride:(m + 1) * stride]) if (m + 1) * stride <= len(b)
                   else 0.0 for m in range(nb)] for q in range(4)])
    S = np.array([np.dot(b[m * stride:(m + 1) * stride], b[m * stride:(m + 1) * stride]) if (m + 1) * stride <= len(b)
                  else 0.0 for m in range(nb)])
    for j in range(n_cand):
        wb = b[j * stride: j * stride + win]
        tail = slice(4 * stride, win)
        dot = sum(D[q][j + q] for q in range(4)) + np.dot(a[tail], wb[tail])
        nrm = sum(S[j + q] for q in range(4)) + np.dot(wb[tail], wb[tail])
        assert abs(dot - np.dot(a, wb)) < 1e-9 and abs(nrm - np.dot(wb, wb)) < 1e-9


def test_tf32_truncation_split_is_exact():
    """chroma.cu: x = hi + lo with hi = x with its low 13 mantissa bits cleared (a valid tf32 value) and lo = x − hi computed
    in float32: the subtraction is exact, |lo| < 2^-10·|x|, and hi + lo reproduces x bit for bit."""
    rng = np.random.default_rng(13)
    x = (rng.standard_normal(100000) * np.exp(rng.uniform(-20, 20, 100000))).astype(np.float32)
    hi = (x.view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)
    lo = (x - hi).astype(np.float32)
    assert np.array_equal((hi + lo).astype(np.float32), x)
    assert np.all(np.abs(lo) < np.abs(x) * 2.0 ** -10 + 1e-45)
    assert np.all((hi.view(np.uint32) & np.uint32(0x1FFF)) == 0)
