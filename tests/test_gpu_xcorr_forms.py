"""GPU: the two searches of xcorr.cu at every block form, chunking, gate and tie, against the restatement
oracle/xcorr_restated.py.

Speed search (ncfa_xcorr_search_batched).  (win, stride) picks the form: the block form xcorr_blocks_ring_kernel<NQ>
when NQ = win / stride is 1..4 and the tail win − NQ·stride is at most 16, the direct form otherwise.  The block kernel
streams every stride-long block through a 4-stage ring of 1024-sample chunks, 8 B blocks per CTA; the pick kernels
scan candidates j = lane, lane + 32, … with a strict >, then merge lanes keeping the lower index on equal c.

Most inputs are integer-valued with |x| <= 4 and win <= 2**20, so every partial sum stays below 2**24 and is exact in
float32 and float64 in any order.  best_j AND best_c must then equal the restatement bit for bit, and exact ties and
exact gate thresholds can be built on purpose.  Buffers are laid out by `place` (test_gpu_segment_placement.py): a_pos
and b_lo run through every residue mod 4 with loud noise around each window, and every call gets exactly the workspace
its size query asks for, followed by a byte pattern that must come back unchanged.

The restatement is not pipeline_port.speed_xcorr_arrays: under numpy 2 (NEP 50) the port's `np.float32 / float`
rounds c to float32, while the reference (numpy < 2) and the kernel compute it in float64 (tests/test_xcorr_restated.py).

Alignment search (ncfa_align_search).  The stretched rows are the first region of its workspace (offset 0, row stride
max_stretched) and must equal np.interp bit for bit.  With integer src_env and n_nc − 1, n_stretched − 1 powers of two
every sum is exact, so peaks and scores must match bit for bit too."""
import numpy as np
import pytest
import scipy.signal
import torch

from oracle import librosa_restated as lr
from oracle import synth
from oracle import xcorr_restated as xr
from test_gpu_segment_placement import place

pytestmark = pytest.mark.gpu
SR = 22050
FENCE = 8192          # bytes of pattern after the workspace
PAT = 0xA5
OUT_FENCE = 16        # elements of pattern after each output array
TINY = np.float32(2.0 ** -50)   # scales a window far below the 1e-10 norm gates, exactly


@pytest.fixture(scope="module", autouse=True)
def profiled(engine):
    """Every launch is recorded under its kernel name, so a test can tell which form ran."""
    from nightcore_analyzer import _native
    torch.cuda.synchronize()
    _native.lib.ncfa_profile_enable(1)
    _native.profile_report()
    yield
    torch.cuda.synchronize()
    _native.profile_report()
    _native.lib.ncfa_profile_enable(0)


def ints(rng, n):
    return rng.integers(-4, 5, n).astype(np.float32)


def dev(engine, x, dtype):
    return torch.from_numpy(np.ascontiguousarray(x, dtype=dtype)).to(engine.device)


def check_tail(t, value):
    assert bool((t[-OUT_FENCE:] == value).all()), "an output was written past its last element"


# ------------------------------------------------------------------------------------------------ speed search
def run_search(engine, audio, a_pos, b_lo, n_cand, win, stride, rms_gate, max_cand=None):
    """One ncfa_xcorr_search_batched call on `audio` (A and B in the same buffer) with exactly the workspace its size
    query gives → (best_j, best_c, sorted names of the kernels launched)."""
    from nightcore_analyzer._native import check, lib, profile_report
    n_w = len(a_pos)
    max_cand = max(1, int(np.max(n_cand))) if max_cand is None else max_cand
    need = lib.ncfa_xcorr_workspace_bytes(n_w, max_cand)
    ws = torch.full((need + FENCE,), PAT, dtype=torch.uint8, device=engine.device)
    best_j = torch.full((n_w + OUT_FENCE,), -7, dtype=torch.int32, device=engine.device)
    best_c = torch.full((n_w + OUT_FENCE,), 7.0, dtype=torch.float64, device=engine.device)
    d_pos, d_lo, d_n = dev(engine, a_pos, np.int64), dev(engine, b_lo, np.int64), dev(engine, n_cand, np.int32)
    torch.cuda.synchronize()
    profile_report()
    with torch.cuda.device(engine.device):
        check(lib.ncfa_xcorr_search_batched(audio.data_ptr(), audio.data_ptr(), d_pos.data_ptr(), d_lo.data_ptr(),
                                            d_n.data_ptr(), n_w, max_cand, int(win), int(stride), float(rms_gate),
                                            best_j.data_ptr(), best_c.data_ptr(), ws.data_ptr(), need,
                                            torch.cuda.current_stream().cuda_stream),
              "ncfa_xcorr_search_batched")
    torch.cuda.synchronize()
    names = sorted(profile_report())
    assert bool((ws[need:] == PAT).all()), "the search wrote past ncfa_xcorr_workspace_bytes"
    check_tail(best_j, -7)
    check_tail(best_c, 7.0)
    return best_j[:n_w].cpu().numpy(), best_c[:n_w].cpu().numpy(), names


FORM_KERNELS = {"block": ["xcorr_blocks_kernel", "xcorr_pick_kernel"],
                "direct": ["xcorr_dots_kernel", "xcorr_pick_kernel"]}


def form_of(win, stride):
    nq = win // stride
    return "block" if 1 <= nq <= 4 and win - nq * stride <= 16 else "direct"


def search_case(engine, a_list, b_list, n_cand, win, stride, rms_gate=1e-3, shift=0):
    """Place the A windows and B spans (window w's a_pos ≡ w + shift, its b_lo ≡ w // 4 + 3w + shift mod 4), run the
    search, check the form and compare with the restatement bit for bit → (best_j, c of every candidate)."""
    arrays = [x for ab in zip(a_list, b_list) for x in ab]
    phases = [(w + shift) % 4 if k == 0 else (w // 4 + 3 * w + shift) % 4 for w in range(len(a_list)) for k in (0, 1)]
    audio, off, _ = place(engine, arrays, phases, seed=77 + shift)
    a_pos, b_lo = off[0::2], off[1::2]
    if len(a_list) >= 4:
        assert set((a_pos % 4).tolist()) == set((b_lo % 4).tolist()) == {0, 1, 2, 3}
    bj, bc, names = run_search(engine, audio, a_pos, b_lo, n_cand, win, stride, rms_gate)
    assert names == FORM_KERNELS[form_of(win, stride)], names
    host = audio.cpu().numpy()
    c = xr.candidate_c(host, host, a_pos, b_lo, n_cand, win, stride, rms_gate)
    want_j, want_c = xr.first_max(c)
    assert bj.tolist() == want_j.tolist()
    assert np.array_equal(bc, want_c), np.flatnonzero(bc != want_c).tolist()
    return bj, c


def int_case(seed, win, stride, n_cands):
    """Integer-valued A windows and B spans of exactly the samples their candidates reach.  Two windows in three hold
    a noisy copy of A at one candidate; the third is noise only."""
    rng = np.random.default_rng(seed)
    a_list, b_list = [], []
    for w, nc in enumerate(n_cands):
        a = ints(rng, win)
        b = ints(rng, (max(nc, 1) - 1) * stride + win)
        if nc > 0 and w % 3 != 2:
            p = int(rng.integers(0, nc)) * stride
            b[p : p + win] = np.clip(a + rng.integers(-2, 3, win), -4, 4)
        a_list.append(a)
        b_list.append(b)
    return a_list, b_list


RAGGED = (0, 1, 7, 8, 9, 31, 32, 33, 130, 0, 2)


@pytest.mark.parametrize("tail", [0, 1, 3, 15, 16])
@pytest.mark.parametrize("nq", [1, 2, 3, 4])
def test_block_form_every_nq_and_tail(engine, nq, tail):
    """xcorr_blocks_ring_kernel<NQ> for NQ = 1..4 (the product's grid, stride = win // 4, only reaches NQ = 4) and
    tails up to the 16 samples the pick kernel sums one lane at a time."""
    stride = 1000 + 17 * nq + tail
    win = nq * stride + tail
    a_list, b_list = int_case(100 * nq + tail, win, stride, (1, 7, 9, 33, 0, 20))
    bj, _ = search_case(engine, a_list, b_list, np.array([1, 7, 9, 33, 0, 20]), win, stride, shift=nq + tail)
    assert int((bj >= 0).sum()) >= 3


@pytest.mark.parametrize("win,stride", [(4 * 1000 + 17, 1000), (1 * 1013 + 17, 1013), (5 * 801, 801),
                                        (5 * 802 + 3, 802), (1003, 1021), (17, 64)],
                         ids=["nq4-tail17", "nq1-tail17", "nq5", "nq5-tail3", "win-below-stride", "win17-stride64"])
def test_direct_form_just_past_the_switch(engine, win, stride):
    """A tail of 17, five blocks per window, or a window shorter than the stride take the direct form, and must agree
    with the restatement just as well."""
    n_cands = (1, 7, 9, 33, 0, 20)
    a_list, b_list = int_case(win + stride, win, stride, n_cands)
    search_case(engine, a_list, b_list, np.array(n_cands), win, stride, shift=win % 4)


CHUNK_STRIDES = (5, 6, 63, 1022, 1023, 1024, 1025, 4095, 4096, 4097, 4098, 16537)


@pytest.mark.parametrize("stride", CHUNK_STRIDES)
def test_block_form_chunking(engine, stride):
    """Strides of every residue mod 4 around the 1024-sample chunk (one chunk up to 1024, two from 1025) and the
    4-stage ring (4096 samples fill it, 4097 is the first to wrap), and the product's 16 537 at its window of 66 150
    (NQ = 4, tail 2): 17 chunks, the ring wrapped four times."""
    win = 4 * stride + 2
    n_cands = (1, 8, 9, 40)
    a_list, b_list = int_case(stride, win, stride, n_cands)
    search_case(engine, a_list, b_list, np.array(n_cands), win, stride, shift=stride % 4)


@pytest.mark.parametrize("form", ["block", "direct"])
def test_ragged_windows_one_launch(engine, form):
    """n_cand = 0, 1, 7, 8, 9, 31, 32, 33 and 130 in one launch: max_cand sizes the grid and the workspace rows, so
    most windows leave CTAs wholly or partly idle (live < 8 blocks) and lanes without candidates."""
    stride = 997
    win = 4 * stride + 3 if form == "block" else 8 * stride + 3
    a_list, b_list = int_case(11, win, stride, RAGGED)
    bj, _ = search_case(engine, a_list, b_list, np.array(RAGGED), win, stride, shift=1)
    assert bj[0] == -1 and bj[9] == -1
    assert int((bj >= 0).sum()) >= 5


@pytest.mark.parametrize("form", ["block", "direct"])
def test_rms_gate_is_strict_at_the_float32_rms(engine, form):
    """The window is dropped when float64(rms_a) < rms_gate, rms_a being the float32 RMS: a gate equal to it keeps the
    window, the next float64 above it drops the window."""
    stride = 1001
    win = 4 * stride + 3 if form == "block" else 6 * stride + 3
    a_list, b_list = int_case(5, win, stride, (12,))          # one window, a noisy copy of A at one candidate
    a64 = a_list[0].astype(np.float64)
    rms = np.float64(np.float32(np.sqrt(np.sum(a64 * a64, dtype=np.float64) / np.float64(win))))
    above = np.nextafter(rms, np.float64(np.inf))
    bj, _ = search_case(engine, a_list, b_list, np.array([12]), win, stride, rms_gate=float(rms))
    assert bj[0] >= 0
    bj, _ = search_case(engine, a_list, b_list, np.array([12]), win, stride, rms_gate=float(above), shift=2)
    assert bj[0] == -1


@pytest.mark.parametrize("form", ["block", "direct"])
def test_norm_gates_and_nonpositive_windows(engine, form):
    """rms_gate = 0, so only the 1e-10 norm gates and the c > 0 rule decide (every window must give (−1, 0.0)):
      0  an all-zero A window;
      1  a nonzero A window with ‖wa‖ < 1e-10 (integers × 2⁻⁵⁰) against a B holding the same pattern;
      2  A and B periodic in whole blocks with B = −A, so every candidate has c = −1, except candidate 2, whose B is
         A × 2⁻⁵⁰ (‖wb‖ < 1e-10, c would be +1 without the gate), and candidate 12, whose B is zero;
      3  every candidate at c = −1;
      4  every candidate at c = 0 exactly (A nonzero only at even, B only at odd samples, even stride)."""
    stride = 1000
    nq = 4 if form == "block" else 8
    win = nq * stride + 2
    rng = np.random.default_rng(17)
    n_c = 20
    span = (n_c - 1) * stride + win

    def periodic(p, n):
        return np.tile(p, n // stride + 2)[:n].astype(np.float32)

    a_list, b_list = [], []
    a_list.append(np.zeros(win, np.float32))
    b_list.append(ints(rng, span))
    pat = ints(rng, win)
    a_list.append(pat * TINY)
    b_list.append(np.tile(pat, n_c * 2)[:span])
    p = rng.integers(1, 5, stride).astype(np.float32) * rng.choice([-1, 1], stride).astype(np.float32)
    a = periodic(p, win)
    b = -periodic(p, span)
    j0, j1 = 2, 2 + nq + 2
    b[j0 * stride : j0 * stride + win] = a * TINY
    b[j1 * stride : j1 * stride + win] = 0.0
    a_list.append(a)
    b_list.append(b)
    a_list.append(periodic(p, win))
    b_list.append(-periodic(p, span))
    even = ints(rng, win)
    even[1::2] = 0.0
    odd = ints(rng, span)
    odd[0::2] = 0.0
    a_list.append(even)
    b_list.append(odd)
    n_cand = np.full(5, n_c)
    bj, c = search_case(engine, a_list, b_list, n_cand, win, stride, rms_gate=0.0)
    assert bj.tolist() == [-1] * 5
    assert np.all(c[0] == -np.inf) and np.all(c[1] == -np.inf)             # the ‖wa‖ gate
    assert c[2, j0] == -np.inf and c[2, j1] == -np.inf                      # the ‖wb‖ gate
    assert np.all(c[2][np.isfinite(c[2])] < 0) and np.isfinite(c[2]).sum() == n_c - 2
    assert np.all(c[3] < 0) and np.all(c[4] == 0.0)


TIE_PERIODS = (1, 5, 8, 13, 32)


@pytest.mark.parametrize("period", TIE_PERIODS)
@pytest.mark.parametrize("form", ["block", "direct"])
def test_ties_keep_the_first_candidate(engine, form, period):
    """B periodic in whole blocks: candidate j and j + period are the same window.  Period 32 puts equal candidates
    in the same lane, 5 and 13 in different lanes (and, 160 = 5·32 apart, in one lane again), 8 in different CTAs of
    the block form, 1 makes every candidate equal.  A is a noisy copy of the candidate `first`, so the maximum is
    positive and ties; the first of the tied candidates must win."""
    stride = 301
    win = 4 * stride + 3 if form == "block" else 8 * stride + 3
    n_c = 200
    rng = np.random.default_rng(period)
    span = (n_c - 1) * stride + win
    b = np.tile(ints(rng, period * stride), span // (period * stride) + 2)[:span]
    first = int(rng.integers(0, period))
    a = np.clip(b[first * stride : first * stride + win] + rng.integers(-1, 2, win), -4, 4).astype(np.float32)
    bj, c = search_case(engine, [a, a], [b, b], np.array([n_c, n_c - 37]), win, stride, shift=period)
    assert bj.tolist() == [first, first]
    assert c[0, first + period] == c[0, first] and c[0, first] > 0


FLOAT_FORMS = {1: (2999, 7), 2: (2051, 11), 3: (1531, 2), 4: (2203, 13)}


@pytest.mark.parametrize("nq", [1, 2, 3, 4])
def test_float_audio_block_forms(engine, nq):
    """Synthetic audio and its 1000/1003 resampling plus noise, at a (win, stride) the product never uses.  Sums are no
    longer exact, so: best_j exactly wherever the restatement's two best c differ by more than 1e-6 relative, and
    best_c within two float32 ulps of the restatement's c of the same candidate."""
    stride, tail = FLOAT_FORMS[nq]
    win = nq * stride + tail
    y = synth.synth(500 + nq, 30.0, SR, bpm=123.0)
    z = scipy.signal.resample_poly(y, 1000, 1003).astype(np.float32)
    z = (z + np.random.default_rng(nq).standard_normal(len(z)).astype(np.float32) * 0.01).astype(np.float32)
    n_c = 30
    a_list, b_list = [], []
    for w in range(6):
        pa = 60000 + 60000 * w
        lo = int(pa * 1000 / 1003) - 15 * stride + 37 * w
        a_list.append(y[pa : pa + win])
        b_list.append(z[lo : lo + (n_c - 1) * stride + win])
    arrays = [x for ab in zip(a_list, b_list) for x in ab]
    audio, off, _ = place(engine, arrays, [(k + nq) % 4 for k in range(len(arrays))], seed=nq)
    a_pos, b_lo = off[0::2], off[1::2]
    n_cand = np.full(6, n_c)
    bj, bc, names = run_search(engine, audio, a_pos, b_lo, n_cand, win, stride, 1e-3)
    assert names == FORM_KERNELS["block"]
    host = audio.cpu().numpy()
    c = xr.candidate_c(host, host, a_pos, b_lo, n_cand, win, stride, 1e-3)
    want_j, _ = xr.first_max(c)
    clear = 0
    for w in range(6):
        top = np.sort(c[w])[::-1]
        if top[0] > 0 and top[0] - top[1] > 1e-6 * abs(top[0]):
            clear += 1
            assert bj[w] == want_j[w], w
        assert bj[w] >= 0, w
        want = c[w, bj[w]]
        assert abs(bc[w] - want) <= 2 * float(np.spacing(np.float32(want))), (w, bc[w], want)
    assert clear >= 5


def test_more_windows_than_one_call(engine):
    """Engine.xcorr_search_dev with 70 000 windows splits them into two C calls of at most MAX_SEGS_PER_CALL (65 535)
    windows; every window's result must still be the restatement's, the ones around the split included."""
    from nightcore_analyzer import _engine
    from nightcore_analyzer._native import profile_report
    n_w, win, stride = 70000, 16, 4
    assert n_w > _engine.MAX_SEGS_PER_CALL
    rng = np.random.default_rng(70000)
    a_host, b_host = ints(rng, 4099), ints(rng, 8191)
    w = np.arange(n_w, dtype=np.int64)
    n_cand = ((w * 5) % 11).astype(np.int32)
    a_pos = (w * 13) % (len(a_host) - win)
    b_lo = (w * 29) % (len(b_host) - 9 * stride - win)
    a, b = dev(engine, a_host, np.float32), dev(engine, b_host, np.float32)
    torch.cuda.synchronize()
    profile_report()
    bj, bc = engine.xcorr_search_dev(a, b, a_pos, b_lo, n_cand, win, stride, 1e-3)
    bj, bc = bj.cpu().numpy(), bc.cpu().numpy()
    assert profile_report()["xcorr_pick_kernel"][0] == 2
    want_j, want_c = xr.search(a_host, b_host, a_pos, b_lo, n_cand, win, stride, 1e-3)
    assert np.array_equal(bj, want_j), np.flatnonzero(bj != want_j)[:10].tolist()
    assert np.array_equal(bc, want_c)
    assert int((bj[65530:65540] >= 0).sum()) >= 3


@pytest.mark.parametrize("nq", [1, 2, 3, 4])
def test_block_form_smallest_workspace(engine, nq):
    """max_cand = 1 gives the smallest block-form workspace: one, two and three windows (one with no candidate), the
    bytes after ncfa_xcorr_workspace_bytes untouched (run_search checks them)."""
    stride = 257 + nq
    win = nq * stride + 5
    for n_cands in ((1,), (1, 0), (1, 0, 1)):
        a_list, b_list = int_case(nq * 10 + len(n_cands), win, stride, n_cands)
        search_case(engine, a_list, b_list, np.array(n_cands), win, stride, shift=len(n_cands))


# ------------------------------------------------------------------------------------------------ alignment search
def run_align(engine, src_env, nc_env, n_str, n_lag, max_stretched=None, max_lags=None):
    """One ncfa_align_search call with exactly the workspace its size query gives → (peak, score, stretched rows
    [n_speeds, max_stretched] read from the workspace)."""
    from nightcore_analyzer._native import check, lib
    n_str, n_lag = np.asarray(n_str, np.int32), np.asarray(n_lag, np.int32)
    n_sp = len(n_str)
    live = n_lag > 0
    max_stretched = max(2, int(n_str[live].max())) if max_stretched is None else max_stretched
    max_lags = int(n_lag[live].max()) if max_lags is None else max_lags
    need = lib.ncfa_align_workspace_bytes(n_sp, max_stretched, max_lags)
    ws = torch.full((need + FENCE,), PAT, dtype=torch.uint8, device=engine.device)
    pk = torch.full((n_sp + OUT_FENCE,), -7, dtype=torch.int32, device=engine.device)
    sc = torch.full((n_sp + OUT_FENCE,), 7.0, dtype=torch.float64, device=engine.device)
    d_src, d_nc = dev(engine, src_env, np.float64), dev(engine, nc_env, np.float64)
    d_ns, d_nl = dev(engine, n_str, np.int32), dev(engine, n_lag, np.int32)
    with torch.cuda.device(engine.device):
        check(lib.ncfa_align_search(d_src.data_ptr(), len(src_env), d_nc.data_ptr(), len(nc_env), d_ns.data_ptr(),
                                    d_nl.data_ptr(), n_sp, max_stretched, max_lags, pk.data_ptr(), sc.data_ptr(),
                                    ws.data_ptr(), need, torch.cuda.current_stream().cuda_stream),
              "ncfa_align_search")
    torch.cuda.synchronize()
    assert bool((ws[need:] == PAT).all()), "the alignment search wrote past ncfa_align_workspace_bytes"
    check_tail(pk, -7)
    check_tail(sc, 7.0)
    rows = ws[: n_sp * max_stretched * 8].view(torch.float64).reshape(n_sp, max_stretched).cpu().numpy()
    return pk[:n_sp].cpu().numpy(), sc[:n_sp].cpu().numpy(), rows


def assert_align_exact(got, want):
    (pk, sc, rows), (w_pk, w_sc, w_rows) = got, want
    assert pk.tolist() == w_pk.tolist()
    assert np.array_equal(sc, w_sc), (sc.tolist(), w_sc.tolist())
    for s, r in enumerate(w_rows):
        if r is not None:
            assert np.array_equal(rows[s, : len(r)], r), s


def align_exact(engine, src, nc, n_str, n_lag, **kw):
    got = run_align(engine, src, nc, n_str, n_lag, **kw)
    want = xr.align(src, nc, n_str, n_lag)
    assert_align_exact(got, want)
    return got


@pytest.mark.parametrize("n_nc", [2, 3, 5, 1000])
def test_align_stretch_is_np_interp(engine, n_nc):
    """The stretched rows equal np.interp(np.linspace(0, 1, ns), np.linspace(0, 1, n_nc), nc_env) bit for bit, for
    ns = 1, 2, 3, 4, n_nc and 2·n_nc − 1 (down- and upsampling, grids that do and do not share points)."""
    rng = np.random.default_rng(n_nc)
    nc = rng.random(n_nc) * 10.0 - 3.0
    ns = sorted({1, 2, 3, 4, 7, n_nc, 2 * n_nc - 1} | ({777, 1234} if n_nc == 1000 else set()))
    src = rng.random(max(ns) + 40)
    n_lag = [3] * len(ns)
    pk, sc, rows = run_align(engine, src, nc, ns, n_lag)
    w_pk, w_sc, w_rows = xr.align(src, nc, ns, n_lag)
    for s, r in enumerate(w_rows):
        assert np.array_equal(rows[s, : len(r)], r), ns[s]
    assert pk.tolist() == w_pk.tolist()
    assert np.all(np.abs(sc - w_sc) <= 1e-12 * np.abs(w_sc))


def dyadic_env(rng, n, hi=16):
    return rng.integers(0, hi, n).astype(np.float64)


def test_align_exact_peaks_at_every_lag_partition(engine):
    """n_lags = 1, 255, 256, 257 and 3000 around the 256-thread partition of the pick kernel, and speeds whose last
    lag is the last valid one (n_stretched + n_lags − 1 = n_src).  src_env rises slowly so peaks fall late."""
    rng = np.random.default_rng(256)
    speeds = [(257, 1), (129, 255), (513, 256), (1025, 257), (2049, 3000), (1025, 4024), (17, 5032), (65, 300)]
    n_src = max(ns + nl - 1 for ns, nl in speeds)
    assert n_src == 5048
    src = dyadic_env(rng, n_src, 8) + np.arange(n_src) * 8 // n_src
    nc = dyadic_env(rng, 513)
    ns, nl = np.array(speeds).T
    pk, _, _ = align_exact(engine, src, nc, ns, nl)
    assert (pk >= 256).sum() >= 3 and pk[2] <= 255


@pytest.mark.parametrize("case", ["period1", "period7", "period256", "flat"])
def test_align_ties_keep_the_first_lag(engine, case):
    """src_env periodic (period 1, i.e. constant, 7 and 256) makes corr[l] = corr[l + period] exactly; `flat` makes
    both envelopes constant, so every lag ties.  The first lag of the tied maximum must win."""
    rng = np.random.default_rng(len(case))
    ns, n_lag = 129, 1000
    n_src = ns + n_lag - 1
    period = {"period1": 1, "period7": 7, "period256": 256, "flat": 1}[case]
    src = np.tile(dyadic_env(rng, period) + 1.0, n_src // period + 1)[:n_src]
    nc = np.full(65, 3.0) if case == "flat" else dyadic_env(rng, 65)
    pk, sc, _ = align_exact(engine, src, nc, [ns, 33], [n_lag, 700])
    assert np.all(pk < period)
    if case == "flat":
        assert sc.tolist() == [1.0, 1.0]


def test_align_zero_envelopes_score_zero(engine):
    rng = np.random.default_rng(0)
    nc, src = dyadic_env(rng, 65), dyadic_env(rng, 600)
    for s, n in ((np.zeros(600), nc), (src, np.zeros(65)), (np.zeros(600), np.zeros(65))):
        pk, sc, _ = align_exact(engine, s, n, [129, 33, 1], [400, 568, 600])
        assert pk.tolist() == [0, 0, 0] and sc.tolist() == [0.0, 0.0, 0.0]


def test_align_skipped_and_live_speeds_mixed(engine):
    """Skipped speeds (n_lags 0 or negative) between live ones give (−1, 0.0), whatever their n_stretched — zero, within
    max_stretched or far beyond it — and leave the live speeds' rows alone."""
    rng = np.random.default_rng(9)
    src, nc = dyadic_env(rng, 3000), dyadic_env(rng, 257)
    max_str = 1025
    n_str = [129, 0, 1025, 1000, 257, 10 ** 6, 1, 1025 + 255, 513, max_str + 300]
    n_lag = [700, 0, 900, -1, 2744, -5, 3000, 0, 2488, -1]
    pk, sc, _ = align_exact(engine, src, nc, n_str, n_lag, max_stretched=max_str)
    skipped = [s for s, nl in enumerate(n_lag) if nl <= 0]
    assert all(pk[s] == -1 and sc[s] == 0.0 for s in skipped)
    assert all(pk[s] >= 0 for s in range(len(n_lag)) if s not in skipped)


def test_align_float_envelopes(engine):
    """RMS envelopes of synthetic audio and the product's 30-speed geometry: stretched rows bit for bit, peaks exact
    where the restatement's best correlation beats the next by more than 1e-9 relative, scores to 1e-12 relative."""
    sr = 11025
    body = synth.synth(41, 40.0, sr, bpm=112.0)
    src_audio = np.concatenate([synth.synth(42, 9.0, sr, bpm=95.0) * 0.3, body]).astype(np.float32)
    nc_audio = scipy.signal.resample_poly(body, 4, 5).astype(np.float32)
    src = lr.rms(src_audio, 2048, 512).astype(np.float64)
    nc = lr.rms(nc_audio, 2048, 512).astype(np.float64)
    n_str, n_lag = [], []
    for speed in np.linspace(1.03, 1.50, 30):
        ns = int(len(nc) / speed)
        n_str.append(ns)
        n_lag.append(min(2583, len(src) - ns) + 1)
    n_str[3], n_lag[3] = 0, -1
    pk, sc, rows = run_align(engine, src, nc, n_str, n_lag)
    w_pk, w_sc, w_rows = xr.align(src, nc, n_str, n_lag)
    clear = 0
    for s, (ns, nl) in enumerate(zip(n_str, n_lag)):
        if nl <= 0:
            assert (pk[s], sc[s]) == (-1, 0.0)
            continue
        assert np.array_equal(rows[s, :ns], w_rows[s]), s
        corr = np.correlate(src[: nl + ns - 1], w_rows[s], mode="valid")
        top = np.sort(corr)[::-1]
        if top[0] - top[1] > 1e-9 * abs(top[0]):
            clear += 1
            assert pk[s] == w_pk[s], s
        assert abs(sc[s] - w_sc[s]) <= 1e-12 * abs(w_sc[s]), s
    assert clear >= 20


def test_align_skipped_speed_stays_inside_the_workspace(engine):
    """A skipped speed's n_stretched may exceed max_stretched (include/ncfa.h: it is ignored).  Two speeds,
    max_stretched = 257, max_lags = 1; the second is skipped with n_stretched = 500.  The stretch kernel used to write
    500 values for it anyway, from the end of the first row on, 181 of them past the 4608-byte workspace."""
    rng = np.random.default_rng(500)
    src, nc = dyadic_env(rng, 300), dyadic_env(rng, 129)
    pk, sc, _ = align_exact(engine, src, nc, [257, 500], [1, 0], max_stretched=257, max_lags=1)
    assert pk.tolist() == [0, -1] and sc[1] == 0.0


def test_align_single_point_stretch_is_the_first_value(engine):
    """np.linspace(0, 1, 1) is [0], so n_stretched = 1 stretches nc_env to [nc_env[0]], not to its last value.
    nc_env[0] < 0 < nc_env[-1] also turns the peak into src_env's minimum."""
    rng = np.random.default_rng(1)
    nc = np.concatenate([[-2.0], dyadic_env(rng, 15), [3.0]])
    src = dyadic_env(rng, 40) + 1.0
    pk, _, rows = align_exact(engine, src, nc, [1, 2, 1], [40, 39, 7])
    assert rows[0, 0] == -2.0 and rows[2, 0] == -2.0
    assert pk[0] == int(np.argmin(src)) and pk[2] == int(np.argmin(src[:7]))
