"""CPU: the render family's host side — the sinc table and output-length rule the library exports, the filter quality
of the arithmetic (through its numpy restatement on the library's table), PCM WAV reading and writing, and the render
CLI's argument checks."""
import math
import wave

import numpy as np
import pytest

from oracle import render_restated as rr

SR = 44100
RATIOS = (0.8, 1.2315, 1.25, 1.5)


@pytest.fixture(scope="module")
def table():
    from nightcore_analyzer import _native
    t = np.zeros(rr.ZEROS * rr.PHASES + 1)
    _native.check(_native.lib.ncfa_host_render_table(t.ctypes.data), "ncfa_host_render_table")
    return t


def test_table_matches_the_formula(table):
    assert table[-1] == 0.0 and table[0] == 1.0
    assert float(np.max(np.abs(table - rr.table_formula()))) <= 1e-15


@pytest.mark.parametrize("ratio", (0.25, 0.8, 1.0, 1.2315, 1.25, 1.5, 2.0, 4.0, 1.25 * 44100 / 48000))
def test_out_len_rule(ratio):
    from nightcore_analyzer import _native
    for n in (0, 1, 2, 3, 511, 4097, 88200, 2**31 - 1):
        want = math.floor((n - 1) / ratio) + 1 if n else 0
        assert _native.lib.ncfa_render_out_len(n, ratio) == want, (n, ratio)
    assert _native.lib.ncfa_render_out_len(88200, 1.25) == 70560


def _amplitude(y, f):
    """Amplitude of the sinusoid of frequency f (Hz at SR) that best fits y (least squares on sin and cos)."""
    ph = 2 * np.pi * f * np.arange(len(y)) / SR
    co = np.linalg.lstsq(np.stack([np.sin(ph), np.cos(ph)], 1), y, rcond=None)[0]
    return float(np.hypot(*co))


def _tone(f, seconds=2.0):
    return np.sin(2 * np.pi * f * np.arange(int(seconds * SR)) / SR).astype(np.float32)


@pytest.mark.parametrize("ratio", RATIOS)
def test_filter_contract(table, ratio):
    inner = slice(2000, -2000)                 # away from the zero-extended edges
    nyq = SR / 2 * min(1.0, 1.0 / ratio)       # the new Nyquist frequency, in input Hz
    y = rr.render(_tone(1000.0, 3.0), ratio, table).astype(np.float64)
    assert len(y) == rr.out_len(3 * SR, ratio)
    ref = np.sin(2 * np.pi * 1000.0 * np.arange(len(y)) * ratio / SR)
    err_db = 20 * np.log10(np.sqrt(np.mean((y - ref)[inner] ** 2)) / np.sqrt(np.mean(ref[inner] ** 2)))
    assert err_db <= -105.0, err_db
    for frac in (0.05, 0.2, 0.4, 0.6, 0.8):
        f = frac * nyq
        gain_db = 20 * np.log10(_amplitude(rr.render(_tone(f), ratio, table).astype(np.float64)[inner], f * ratio))
        assert abs(gain_db) <= 1e-3, (frac, gain_db)
    if ratio > 1.0:  # below 1 the new Nyquist frequency is the input's own: nothing above it can be present
        y = rr.render(_tone(1.08 * nyq), ratio, table).astype(np.float64)[inner]
        alias_dbfs = 20 * np.log10(np.max(np.abs(y)))
        assert alias_dbfs <= -95.0, alias_dbfs


def _write_raw(path, ints, width, channels, rate):
    if width == 1:
        raw = (ints + 128).astype(np.uint8).tobytes()
    elif width == 3:
        raw = (ints.reshape(-1, 1) >> np.array([0, 8, 16])).astype(np.uint8).tobytes()
    else:
        raw = ints.astype(f"<i{width}").tobytes()
    with wave.open(str(path), "wb") as w:
        w.setnchannels(channels)
        w.setsampwidth(width)
        w.setframerate(rate)
        w.writeframes(raw)


def _random_ints(width, n, seed):
    full = 1 << (8 * width - 1)
    ints = np.random.default_rng(seed).integers(-full, full, n, dtype=np.int64)
    ints[:4] = [-full, full - 1, 0, -1]
    return ints


@pytest.mark.parametrize("width", (1, 2, 3))
def test_write_reproduces_read(tmp_path, width):
    from nightcore_analyzer.io import read_wav, write_wav
    src, dst = tmp_path / "a.wav", tmp_path / "b.wav"
    _write_raw(src, _random_ints(width, 2 * 5000, width), width, 2, SR)
    frames, rate, sw = read_wav(src)
    assert frames.shape == (5000, 2) and frames.dtype == np.float32 and (rate, sw) == (SR, width)
    write_wav(dst, frames, rate, sw)
    assert dst.read_bytes() == src.read_bytes()


def _parent_load(path, sr):
    """load_audio's decode, down-mix and rate conversion before read_wav existed."""
    import scipy.signal
    from fractions import Fraction
    with wave.open(str(path), "rb") as w:
        n, ch, sw, fr = w.getnframes(), w.getnchannels(), w.getsampwidth(), w.getframerate()
        raw = w.readframes(n)
    if sw == 2:
        y = np.frombuffer(raw, dtype="<i2").astype(np.float32) / 32768.0
    elif sw == 4:
        y = np.frombuffer(raw, dtype="<i4").astype(np.float32) / 2147483648.0
    else:
        y = (np.frombuffer(raw, dtype=np.uint8).astype(np.float32) - 128.0) / 128.0
    if ch > 1:
        y = y.reshape(-1, ch).mean(axis=1).astype(np.float32)
    if fr != sr:
        f = Fraction(int(sr), int(fr))
        y = scipy.signal.resample_poly(y.astype(np.float64), f.numerator, f.denominator).astype(np.float32)
    return y.astype(np.float32), sr


@pytest.mark.parametrize("width", (1, 2, 4))
@pytest.mark.parametrize("channels", (1, 2))
@pytest.mark.parametrize("rate", (22050, 44100))
def test_load_audio_unchanged(tmp_path, width, channels, rate):
    from nightcore_analyzer.io import load_audio
    path = tmp_path / "x.wav"
    _write_raw(path, _random_ints(width, channels * 7001, rate + width), width, channels, rate)
    y, sr = load_audio(str(path))
    want, _ = _parent_load(path, 22050)
    assert sr == 22050 and y.dtype == np.float32 and y.tobytes() == want.tobytes()


def test_load_audio_reads_24_bit(tmp_path):
    from nightcore_analyzer.io import load_audio, read_wav
    path = tmp_path / "x.wav"
    _write_raw(path, _random_ints(3, 2 * 4410, 24), 3, 2, 22050)
    y, sr = load_audio(str(path))
    assert sr == 22050 and y.dtype == np.float32
    assert y.tobytes() == read_wav(path)[0].mean(axis=1).astype(np.float32).tobytes()


def test_render_cli_rejects_bad_arguments(tmp_path, capsys):
    from nightcore_analyzer import render
    src = tmp_path / "src.wav"
    _write_raw(src, _random_ints(2, 100, 1), 2, 1, 22050)
    out = str(tmp_path / "out.wav")
    bad = [
        ["--source", str(src), "--output", out],                                          # neither mode
        ["--source", str(src), "--output", out, "--speed", "1.25", "--nightcore", str(src)],  # both modes
        ["--source", str(src), "--output", out, "--speed", "0.1"],                        # outside [0.25, 4]
        ["--source", str(src), "--output", out, "--speed", "nan"],
        ["--source", str(tmp_path / "missing.wav"), "--output", out, "--speed", "1.25"],
        ["--source", str(src), "--output", out, "--nightcore", str(tmp_path / "missing.wav")],
        ["--source", str(src), "--speed", "1.25"],                                        # no --output
        ["--source", str(src), "--output", out, "--speed", "fast"],
    ]
    for argv in bad:
        assert render.main(argv) == 2, argv
    assert not (tmp_path / "out.wav").exists()
    assert "ERROR" in capsys.readouterr().err
