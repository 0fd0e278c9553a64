"""
The render step of the reference's workflow (workflow.py:117 ``sox SRC HQNC speed X``) and the loop around it
(workflow.py:778-833): build the high-quality nightcore (HQNC) from a lossless source, verify it against the original
nightcore (NCOG), and re-render at the corrected speed until the tempo check passes.

``speed X`` plays the source X times faster at the same sample rate, so pitch and tempo both rise by X.  The resampler
is ``ncfa_render_batched`` (a Kaiser-windowed sinc, band-limited at the new Nyquist frequency; include/ncfa.h); every
channel of every track is one segment of one launch.  Parity with sox's own resampler is not claimed.

    python -m nightcore_analyzer.render --source SRC.wav --output HQNC.wav --speed 1.25
    python -m nightcore_analyzer.render --source SRC.wav --output HQNC.wav --nightcore NCOG.wav
"""
from __future__ import annotations

import argparse
import json
import math
import sys
from pathlib import Path
from typing import Callable, List, Optional, Sequence, Tuple

import numpy as np

from . import _engine, pipeline, verify
from .io import read_wav, write_wav

SPEED_MIN, SPEED_MAX = 0.25, 4.0   # the ratio range ncfa_render_batched accepts


def speed_arrays(tracks: Sequence[np.ndarray], speed) -> List[np.ndarray]:
    """Each track ([n] or [n, channels] float32) played `speed` times faster (one number, or one per track) → float32
    arrays of the same rank and channel count, floor((n − 1)/speed) + 1 frames long."""
    tracks = [np.asarray(t, dtype=np.float32) for t in tracks]
    speeds = np.broadcast_to(np.asarray(speed, dtype=np.float64), (len(tracks),))
    chans, ratios = [], []
    for t, s in zip(tracks, speeds):
        cols = t.reshape(len(t), -1)
        chans += [cols[:, j] for j in range(cols.shape[1])]
        ratios += [s] * cols.shape[1]
    if not chans:
        return []
    eng = _engine.get_engine()
    audio, seg_off, seg_len = eng.pack(chans)
    ratios = np.asarray(ratios, dtype=np.float64)
    out, out_off = eng.render_dev(audio, seg_off, seg_len, ratios)
    out_len = eng.render_layout(seg_len, ratios)[0]
    host = eng.to_host(out)
    res, k = [], 0
    for t in tracks:
        n_ch = 1 if t.ndim == 1 else t.shape[1]
        cols = [host[out_off[k + j] : out_off[k + j] + out_len[k + j]] for j in range(n_ch)]
        res.append(cols[0].copy() if t.ndim == 1 else np.stack(cols, axis=1))
        k += n_ch
    return res


def render(source_path: str, out_path: str, speed: float) -> None:
    """``sox SRC OUT speed X``: the source WAV `speed` times faster, written at its own rate, channel count and sample
    width."""
    frames, rate, width = read_wav(source_path)
    write_wav(out_path, speed_arrays([frames], speed)[0], rate, width)


def initial_speed(source_path: str, ncog_path: str, log: Optional[Callable[[str], None]] = None) -> float:
    """The speed the NCOG was made at, from one analysis of the pair: the IBI ratio when there is one, else the tempo
    ratio (the rule of ``verify.Verification.best_ratio``)."""
    res = pipeline.run(str(ncog_path), str(source_path), compute_pitch=False, log=log)
    return res.ibi_ratio if res.ibi_ratio is not None else res.tempo_ratio


def render_and_verify(source_path: str, ncog_path: str, out_path: str, speed: Optional[float] = None, rounds: int = 3,
                      log: Optional[Callable[[str], None]] = None) -> List[Tuple[float, verify.Verification]]:
    """workflow.py:117 and 778-833 as one loop: render the HQNC at `speed`, write it to `out_path`, verify it against
    the NCOG, and stop when the tempo check passes; otherwise multiply the speed by the verification's corrective factor
    (workflow.py:808-811) and render again, at most `rounds` times.  `speed` None: start from ``initial_speed``.
    → [(speed, Verification)] per round; `out_path` holds the last render."""
    if speed is None:
        speed = initial_speed(source_path, ncog_path, log)
    frames, rate, width = read_wav(source_path)
    history = []
    for _ in range(rounds):
        if not (math.isfinite(speed) and SPEED_MIN <= speed <= SPEED_MAX):
            raise ValueError(f"speed {speed} is outside [{SPEED_MIN}, {SPEED_MAX}]")
        write_wav(out_path, speed_arrays([frames], speed)[0], rate, width)
        v = verify.verify(out_path, ncog_path, log=log)
        history.append((float(speed), v))
        if v.tempo_ok:
            break
        speed = speed * v.corrected_speed_factor
    return history


def _round_dict(speed: float, v: verify.Verification) -> dict:
    return {"speed": speed, "best_ratio": v.best_ratio, "estimator": v.estimator, "tempo_ok": v.tempo_ok,
            "xcorr_quality": v.result.xcorr_quality}


def main(argv: Optional[List[str]] = None) -> int:
    p = argparse.ArgumentParser(prog="python -m nightcore_analyzer.render",
                                description="Render a high-quality nightcore: the source played X times faster "
                                            "(sox speed X), optionally verified against the original nightcore and "
                                            "re-rendered at the corrected speed.")
    p.add_argument("--source", "-s", metavar="FILE", required=True, help="Lossless source (PCM .wav)")
    p.add_argument("--output", "-o", metavar="FILE", required=True, help="HQNC to write (PCM .wav, source format)")
    p.add_argument("--speed", type=float, metavar="X", help="Render once at this speed")
    p.add_argument("--nightcore", "-n", metavar="FILE",
                   help="Original nightcore: estimate the speed, then render and verify until the tempo matches")
    p.add_argument("--quiet", "-q", action="store_true", help="Suppress progress output")
    try:
        args = p.parse_args(argv)
    except SystemExit as exc:      # argparse exits with 2 on bad arguments and 0 for --help
        return int(exc.code or 0)
    problems = []
    if (args.speed is None) == (args.nightcore is None):
        problems.append("give exactly one of --speed X and --nightcore FILE")
    if args.speed is not None and not (math.isfinite(args.speed) and SPEED_MIN <= args.speed <= SPEED_MAX):
        problems.append(f"--speed must be in [{SPEED_MIN}, {SPEED_MAX}]")
    if not Path(args.source).exists():
        problems.append(f"Source file not found: {args.source}")
    if args.nightcore is not None and not Path(args.nightcore).exists():
        problems.append(f"Nightcore file not found: {args.nightcore}")
    if problems:
        for msg in problems:
            print(f"ERROR: {msg}", file=sys.stderr)
        return 2
    try:
        if args.speed is not None:
            render(args.source, args.output, args.speed)
            print(json.dumps({"speed": args.speed, "output": args.output}))
            return 0
        history = render_and_verify(args.source, args.nightcore, args.output, log=None if args.quiet else print)
    except Exception as exc:  # noqa: BLE001 — like cli.py, any failure of the analysis is exit code 1
        print(f"\nERROR: {exc}", file=sys.stderr)
        return 1
    for speed, v in history:
        print(json.dumps(_round_dict(speed, v)))
    return 0 if history and history[-1][1].tempo_ok else 1


if __name__ == "__main__":
    sys.exit(main())
