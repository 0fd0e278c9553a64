"""Micro-benchmark of ncfa_render_batched, the HQNC render (sox `speed` replacement).

Workload: 125 stereo tracks of 180 s at 44.1 kHz (250 segments, 7.9 GB of float32 input, more than the 126 MB L2 many
times over, so every pass reads HBM) played at speed 1.25 in one launch.  The kernel is timed with CUDA events after
warm-up; the rates are over algorithmic work: outputs, taps (outputs × (ceil(2·half) + 1)) and bytes (input read once
plus output written once, float32).  Three tracks are checked bit for bit against oracle/render_restated.py at their
two edges and in the middle.  The card's name and power limit are read in the same run.

    python profiles/micro/render_bench.py [--tracks 125] [--seconds 180] [--iters 5] [--out FILE.json]
"""
import argparse
import json
import math
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "nightcore-to-flac-analyzer_b200")]

from nightcore_analyzer import _engine, _native  # noqa: E402
from oracle import render_restated as rr  # noqa: E402


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        return float(out.stdout.strip().splitlines()[0])
    except Exception:  # noqa: BLE001 — reported as unknown, never guessed
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tracks", type=int, default=125)
    ap.add_argument("--seconds", type=float, default=180.0)
    ap.add_argument("--sr", type=int, default=44100)
    ap.add_argument("--speed", type=float, default=1.25)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "render_bench_b200.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("render_bench needs a CUDA device")
    eng = _engine.get_engine()
    n_seg, n = 2 * args.tracks, int(args.seconds * args.sr)
    seg_len = np.full(n_seg, n, dtype=np.int32)
    seg_off = np.arange(n_seg, dtype=np.int64) * n
    ratio = np.full(n_seg, args.speed)
    out_len, out_off, total = eng.render_layout(seg_len, ratio)
    gen = torch.Generator(device=eng.device).manual_seed(1)
    audio = torch.randn(n_seg * n, generator=gen, device=eng.device, dtype=torch.float32).mul_(0.3)
    out = torch.empty(total, dtype=torch.float32, device=eng.device)
    d_off, d_len = eng.to_dev(seg_off), eng.to_dev(seg_len)
    d_ratio, d_out_off = eng.to_dev(ratio), eng.to_dev(out_off)
    st = torch.cuda.current_stream().cuda_stream

    def launch():
        _native.check(_native.lib.ncfa_render_batched(audio.data_ptr(), d_off.data_ptr(), d_len.data_ptr(),
                                                      d_ratio.data_ptr(), ratio.ctypes.data, n_seg, n,
                                                      d_out_off.data_ptr(), out.data_ptr(), st), "ncfa_render_batched")

    for _ in range(args.warmup):
        launch()
    torch.cuda.synchronize()
    times = []
    for _ in range(args.iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        launch()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1) / 1e3)
    t = float(np.median(times))

    half = rr.ZEROS / (rr.ROLLOFF / max(1.0, args.speed))
    taps = int(out_len.sum()) * (math.ceil(2.0 * half) + 1)
    nbytes = 4 * (n_seg * n + int(out_len.sum()))

    table = np.zeros(rr.ZEROS * rr.PHASES + 1)
    _native.check(_native.lib.ncfa_host_render_table(table.ctypes.data), "ncfa_host_render_table")
    checked, bad = [], []
    for seg in (0, n_seg // 2 + 1, n_seg - 1):
        x = audio[seg * n : (seg + 1) * n].cpu().numpy()
        nout = int(out_len[seg])
        m = np.concatenate([np.arange(0, 4096), np.arange(nout // 2, nout // 2 + 4096), np.arange(nout - 4096, nout)])
        got = out[int(out_off[seg]) : int(out_off[seg]) + nout].cpu().numpy()[m]
        (checked if got.tobytes() == rr.render(x, args.speed, table, m).tobytes() else bad).append(seg)

    res = {
        "what": "ncfa_render_batched, one launch",
        "device": torch.cuda.get_device_name(),
        "power_limit_w": power_limit_w(),
        "tracks": args.tracks, "channels": 2, "seconds": args.seconds, "sr": args.sr, "speed": args.speed,
        "segments": n_seg, "outputs": int(out_len.sum()), "taps_per_output": math.ceil(2.0 * half) + 1,
        "kernel_s_median": t, "kernel_s_all": times,
        "outputs_per_s": int(out_len.sum()) / t, "taps_per_s": taps / t, "algorithmic_GB_per_s": nbytes / t / 1e9,
        "audio_s_per_s": n_seg / 2 * args.seconds / t,
        "oracle_bit_equal_segments": checked, "oracle_mismatch_segments": bad,
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=2)
    print(json.dumps(res))
    if bad:
        sys.exit(1)


if __name__ == "__main__":
    main()
