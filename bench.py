#!/usr/bin/env python
"""Benchmark of the windowed spectral front-end on B200 (BASELINE.json metric: analysis windows/sec
and track-pairs/sec).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (config 5, the contract line)
    python bench.py --impl reference --steps K --warmup W    # the CPU path on the host cores, same config
    python bench.py --config 2|3|4 [--steps K]               # per-family lines of BASELINE configs 2 / 3 / 4
    python bench.py --single-pair                            # config 1: latency of one pair
    python bench.py --steps K --dump-outputs DIR             # config 5, plus the last timed step's results as DIR/*.npy

A step = one full analysis (strip → slice → gate → pitch → tempo src → prior → tempo nc → hop-64
IBI pass → bootstraps → result assembly) of a batch of synthetic track pairs of BASELINE config 5
(180 s source at 22 050 Hz + 1.25× nightcore; 32 distinct pairs tiled to the batch size).
`value` is measured with the batch resident in HBM; `e2e` goes through the public batch API
(`nightcore_analyzer.run_batch`) with the batch in pinned host memory (H2D inside the timed region,
results back on the host); `e2e_pageable` starts from ordinary numpy arrays.  One JSON line on stdout (rank 0).

The reference arm times the CPU port of the reference's pipeline (oracle/pipeline_port.py — the reference
itself needs librosa and does not exist on the GPU box) on the SAME configuration: 180 s pairs, all host
cores, a bounded sample of pairs per step, its independent units (windows, chunks, whole-track passes) dealt
to one process per core (oracle/pipeline_tasks.py).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "nightcore-to-flac-analyzer_b200"))

import numpy as np  # noqa: E402

SR = 22050
PAIR_SEC = 180.0
N_DISTINCT = 32          # distinct synthetic pairs, tiled to the batch size (SURVEY §8d; stated in `data`)
NC_SEC_PER_SRC_SEC = 0.8  # nightcore = resample_poly(src, 4, 5)

WORKLOAD = ("config 5: batch of 1000 synthetic 180 s track pairs (22050 Hz source + 1.25x nightcore), "
            "full windowed tempo+pitch+IBI+bootstrap analysis, pairs sharded across ranks")


def workload_config(pairs: int, pair_sec: float) -> dict:
    """The workload description — identical in the GPU arm and the reference arm."""
    gb = pairs * pair_sec * (1.0 + NC_SEC_PER_SRC_SEC) * SR * 4 / 1e9
    return {"workload": WORKLOAD, "pairs": pairs, "pair_sec": pair_sec, "sr": SR, "n_distinct": N_DISTINCT,
            "l2": f"inputs larger than L2: {gb:.1f} GB of audio per step, every sample read from HBM (126 MB L2)"}


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def load_traffic(kernel: str):
    """DRAM bytes per launch of `kernel` from the committed `ncu --set full` capture (profiles/ncu_traffic.json)."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            t = json.load(f)[kernel]
        return int(t["dram_bytes_per_launch"]), t["source"]
    except Exception:
        return None, None


def _synth_pair(args):
    i, dur = args
    from oracle import synth
    src, nc = synth.make_pair(5000 + i, dur, SR)
    return i, nc, src


def make_pairs(ids, dur: float, procs: int = 0) -> dict:
    """{i: (nc, src)} for the distinct pair indices `ids` (oracle/synth.py, seeds 5000 + i), synthesised in parallel."""
    import multiprocessing as mp
    ids = sorted(set(int(i) for i in ids))
    procs = max(1, min(len(ids), procs or (os.cpu_count() or 1)))
    if procs == 1:
        out = [_synth_pair((i, dur)) for i in ids]
    else:
        with mp.get_context("fork").Pool(procs) as pool:
            out = pool.map(_synth_pair, [(i, dur) for i in ids], chunksize=1)
    return {i: (nc, src) for i, nc, src in out}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any(r[3 + j].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


# --------------------------------------------------------------------------------------- CPU arm
class CpuArm:
    """The CPU port on `procs` host processes: a step analyses a sample of `n_sample` pairs of `dur` seconds, their
    independent units dealt to the pool (oracle/pipeline_tasks.py)."""

    def __init__(self, dur: float, procs: int, n_sample: int, pairs: dict = None):
        from oracle import pipeline_tasks
        self.procs, self.n, self.dur = procs, max(1, n_sample), dur
        n_distinct = min(N_DISTINCT, 2 * self.n)
        if pairs is None or any(i not in pairs for i in range(n_distinct)):
            pairs = make_pairs(range(n_distinct), dur, procs)
        self.pairs = [pairs[i] for i in range(n_distinct)]
        self.runner = pipeline_tasks.TaskRunner(self.pairs, SR, procs=procs, faithful_cost=True)
        self.cursor = 0

    def step(self, n=None):
        n = self.n if n is None else n
        ids = [(self.cursor + j) % len(self.pairs) for j in range(n)]
        self.cursor += n
        t0 = time.perf_counter()
        results, windows = self.runner.run(ids)
        wall = time.perf_counter() - t0
        bad = [r for r in results if isinstance(r, Exception)]
        if bad:
            raise bad[0]
        return windows, n, wall

    def sample_text(self):
        return (f"{self.n} pairs of {self.dur:.0f} s source + 1.25x nightcore per step (config 5 shape: 35 + 27 windows, "
                f"7 chunk pairs, 2 hop-64 whole-track passes per pair), units dealt to {self.procs} processes; "
                f"throughput extrapolates linearly to the 1000-pair batch")

    def close(self):
        self.runner.close()


def audio_seconds(n_pairs: float, pair_sec: float) -> float:
    return n_pairs * pair_sec * (1.0 + NC_SEC_PER_SRC_SEC)


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir: str, results, pair_ids, prefix: str = "") -> None:
    """Write what the analysis handed its caller, one float64 .npy per field, so that two builds can be compared output
    for output: the per-pair record (status, tempo / pitch / IBI ratios and CIs, window counts, median BPMs; see
    parallel.result_record), the analysed durations, and the per-window tempo and per-chunk pitch lists padded with NaN
    (None and failed pairs are NaN too).  `pair_index` names the pair of every row; above DUMP_MAX_BYTES the rows are a
    fixed, seeded sample of the pairs."""
    from nightcore_analyzer import parallel as npar
    ok = [None if r is None or isinstance(r, Exception) else r for r in results]
    nan = float("nan")

    def padded(name):
        rows = [[] if r is None else (getattr(r, name) or []) for r in ok]
        a = np.full((len(rows), max((len(x) for x in rows), default=0)), nan)
        for i, x in enumerate(rows):
            a[i, :len(x)] = [nan if v is None else v for v in x]
        return a

    arrays = {"pair_index": np.asarray(pair_ids, dtype=np.float64),
              "records": npar.records_of(results),
              "durations": np.array([[nan, nan] if r is None else
                                     [nan if r.nc_duration is None else r.nc_duration,
                                      nan if r.src_duration is None else r.src_duration] for r in ok]).reshape(-1, 2)}
    for name in ("src_tempos_raw", "nc_tempos_raw", "src_pitches_raw", "nc_pitches_raw"):
        arrays[name] = padded(name)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        n = len(ok)
        keep = np.sort(np.random.default_rng(0).choice(n, int(n * DUMP_MAX_BYTES / total), replace=False))
        arrays = {k: a[keep] for k, a in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"), a)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    procs = max(1, min(cores, args.cpu_procs or cores))
    arm = CpuArm(args.pair_sec, procs, args.cpu_sample or max(1, procs // 4))
    vals, pps, walls = [], [], []
    try:
        for s in range(args.warmup):
            arm.step(1)                       # warm-up on a one-pair sample (page cache, FFT plans, BLAS pools)
        for s in range(args.steps):
            w, n, wall = arm.step()
            vals.append(w / wall)
            pps.append(n / wall)
            walls.append(wall)
    finally:
        arm.close()
    v = float(np.sum([a * b for a, b in zip(vals, walls)]) / np.sum(walls))      # windows of all steps / time of all steps
    p = float(len(walls) * arm.n / np.sum(walls))
    line = {
        "impl": "reference", "metric": "analysis_windows_per_sec", "value": v, "unit": "windows/s",
        "pairs_per_sec": p, "audio_sec_per_sec": audio_seconds(p, args.pair_sec), "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * float(np.mean(walls)), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": f"synthetic ({N_DISTINCT} distinct pairs; oracle/synth.py)",
        "config": workload_config(args.pairs, args.pair_sec),
        "cpu_baseline": {"value": v, "unit": "windows/s", "cores": procs, "kind": "port", "sample": arm.sample_text(),
                         "pairs_per_sec": p, "warmup_sample": "1 pair per warm-up step"},
        "e2e": {"value": v, "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------- GPU arm
def run_gpu(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    blocking = False
    if os.environ.get("NCFA_BLOCKING_SYNC"):   # experiment only: measured slower (profiles/r3d_blocking_sync.log)
        sys.path.insert(0, os.path.join(ROOT, "nightcore-to-flac-analyzer_b200"))
        from nightcore_analyzer import parallel as _npar0
        blocking = _npar0.use_blocking_sync(local_rank)
    torch.cuda.set_device(local_rank)
    cpus_local = []
    if world > 1 and not os.environ.get("NCFA_NO_NUMA_BIND"):
        sys.path.insert(0, os.path.join(ROOT, "nightcore-to-flac-analyzer_b200"))
        from nightcore_analyzer import parallel as _npar
        cpus_local = _npar.bind_to_gpu_cpus(local_rank)   # pinned buffers on the GPU's own NUMA node
    # torchrun exports OMP_NUM_THREADS=1 to every rank, which makes the pageable → pinned staging copy of
    # run_batch(list of numpy arrays) single-threaded; give every rank its share of the host cores instead
    torch.set_num_threads(max(1, (os.cpu_count() or 1) // max(1, world)))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    import nightcore_analyzer as na
    from nightcore_analyzer import _engine, _native, batch as nbatch, parallel as npar

    eng = _engine.get_engine()
    total_pairs = args.pairs
    my_ids = npar.shard_indices(total_pairs, rank, world)
    n_distinct = min(N_DISTINCT, max(1, total_pairs))
    cores = os.cpu_count() or 1
    need = set(i % n_distinct for i in my_ids) | (set(range(n_distinct)) if rank == 0 else set())
    distinct = make_pairs(need, args.pair_sec, max(1, cores // world))
    pairs_np = [distinct[i % n_distinct] for i in my_ids]          # ordinary (pageable) numpy arrays
    kw = dict(compute_pitch=not args.no_pitch, compute_ibi=not args.no_ibi)

    # the rank's pairs in pinned host memory (the contract's e2e starts here) and resident in HBM (`value`)
    pinned = nbatch.pin_pairs(pairs_np, SR)
    n_mine = len(my_ids)
    if args.sub_batch > 0:
        sub = args.sub_batch                                                        # explicit: as given
    else:
        # default 125 pairs per job whatever the share: small jobs inflate the kernel time (latency-bound kernels: 87 ms of
        # kernels for 125 pairs in one job, 116-126 ms in five), measured profiles/r2q_*: one job 1287 pairs/s, five jobs 1081
        sub = 125
    sizes = nbatch.stagger_sizes(n_mine, sub, args.workers)          # first job short: the workers run out of phase
    starts = [sum(sizes[:j]) for j in range(len(sizes))]
    resident = [nbatch.upload(pinned, k, start_pair=s) for s, k in zip(starts, sizes)]
    torch.cuda.synchronize()
    resident_bytes = sum(st.h2d_bytes for st in resident)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident():
        stats = {}
        res = nbatch.analyse_resident(resident, stats=stats, workers=args.workers, **kw)
        return res, stats

    def step_e2e(source):
        # the public batch API: pinned (or pageable) host arrays in, host results out; staging, H2D copies and the
        # analysis of different sub-batches overlap inside the call
        stats = {}
        res = na.run_batch(source, SR, sub_batch=sub, workers=args.workers, stats=stats, **kw)
        return res, stats

    # ---- device-resident timing (value)
    for _ in range(args.warmup):
        step_resident()
    barrier()
    l0 = _engine.total_launches()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk:
        ev0.record()
        for _ in range(args.steps):
            res, stats = step_resident()
        ev1.record()
        barrier()
    ms = ev0.elapsed_time(ev1) / args.steps
    launches = (_engine.total_launches() - l0) // max(1, args.steps)
    n_ok = sum(1 for r in res if not isinstance(r, Exception))
    windows = stats["windows"]

    # ---- per-kernel shares and the front-end roofline: one extra step with the library's event profiler on
    # (single host worker here: with two streams the event brackets of one stream would include the other's kernels)
    _native.lib.ncfa_profile_enable(1)
    pstats = {}
    nbatch.analyse_resident(resident, stats=pstats, workers=1, **kw)
    torch.cuda.synchronize()
    prof = _native.profile_report()
    _native.lib.ncfa_profile_enable(0)
    roof = npar.frontend_roofline(prof, pstats)

    # ---- end-to-end timing through the public API, pinned host buffers
    def time_e2e(source, warm, steps):
        for _ in range(warm):
            step_e2e(source)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            r, s = step_e2e(source)
        e1.record()
        barrier()
        return max(e0.elapsed_time(e1), 1e3 * (time.perf_counter() - t0)) / steps, r, s

    ms_e2e, res_e, stats_e = time_e2e(pinned, min(args.warmup, 3), args.steps)
    windows_e = stats_e["windows"]
    h2d, d2h = stats_e["h2d_bytes"], npar.result_bytes(stats_e)
    if args.no_pageable:
        ms_page, windows_p = None, 0
    else:
        ms_page, _, stats_p = time_e2e(pairs_np, 1, args.steps)
        windows_p = stats_p["windows"]

    # ---- max over ranks, totals over ranks
    if world > 1:
        t = torch.tensor([ms, ms_e2e, ms_page or 0.0], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e, ms_page = float(t[0]), float(t[1]), (float(t[2]) if ms_page is not None else None)
        c = torch.tensor([windows, n_mine, n_ok, h2d, d2h, launches, windows_e, windows_p], dtype=torch.float64, device="cuda")
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
        windows, n_pairs_all, n_ok, h2d, d2h, launches, windows_e, windows_p = (int(x) for x in c.tolist())
        gathered = npar.gather_result_records(res_e, my_ids, total_pairs)   # the NCCL gather of per-pair records
    else:
        n_pairs_all = n_mine
        gathered = npar.records_of(res_e)

    if rank == 0:
        # N-rank identity: every gathered row must equal the record of the same pair analysed ALONE on this rank
        alone = npar.records_of(na.run_batch([distinct[i] for i in range(n_distinct)], SR, **kw))
        want = alone[np.arange(total_pairs) % n_distinct]
        gather_identical = bool(gathered.shape == want.shape and
                                np.array_equal(np.nan_to_num(gathered, nan=-1.0), np.nan_to_num(want, nan=-1.0)))
        peak, peak_kind = load_peaks()
        traffic, traffic_src = load_traffic("stft_logmel_kernel[hop<=128]")
        value = windows / (ms / 1e3)
        pps = n_pairs_all / (ms / 1e3)
        pps_e = n_pairs_all / (ms_e2e / 1e3)
        line = {
            "metric": "analysis_windows_per_sec", "value": value, "unit": "windows/s",
            "pairs_per_sec": pps, "audio_sec_per_sec": audio_seconds(pps, args.pair_sec), "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": f"synthetic ({n_distinct} distinct pairs tiled to {total_pairs}; oracle/synth.py)",
            "config": workload_config(total_pairs, args.pair_sec),
            "schedule": {"sub_batch_pairs": sub, "resident_sub_batches": sizes, "e2e_sub_batches": stats_e.get("sub_batches"),
                         "host_workers": args.workers, "windows_per_step": windows, "pairs_ok": n_ok,
                         "rank0_cpu_affinity": len(cpus_local) or None, "blocking_sync": bool(blocking),
                         "pitch": not args.no_pitch, "ibi": not args.no_ibi,
                         "resident_audio_mb_per_rank": round(resident_bytes / 1e6, 1)},
            "e2e": {"value": windows_e / (ms_e2e / 1e3), "unit": "windows/s", "ms_per_step": ms_e2e,
                    "pairs_per_sec": pps_e, "audio_sec_per_sec": audio_seconds(pps_e, args.pair_sec),
                    "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "h2d_copy_gbs_rank0": round(float(stats_e.get("h2d_copy_gbs", 0.0)), 2),
                    "h2d_copy_ms_rank0": round(float(stats_e.get("h2d_copy_ms", 0.0)), 1),
                    "api": "nightcore_analyzer.run_batch(PinnedBatch) — pinned host memory in, AnalysisResult objects out"},
            "gather_identical": gather_identical,
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": roof["gbs"], "peak": peak, "unit": "GB/s",
                         "frac": roof["gbs"] / peak, "traffic": traffic, "peak_kind": peak_kind,
                         "kernel": roof["kernel"], "launches": roof["launches"],
                         "algorithmic_bytes_per_launch": roof["bytes_per_launch"],
                         "ms_per_launch": roof["ms_per_launch"], "traffic_source": traffic_src,
                         "fp32_tflops": roof["tflops"], "fp32_peak_tflops": 74.5,
                         "fp32_frac": roof["tflops"] / 74.5, "share_of_step": roof["share"],
                         "note": "compute bound (AI 249 flop/B vs ridge 11.5): the FP32 fraction is the binding one",
                         "front_end": roof["front_end"]},
            "kernels": roof["table"],
            "clocks": clk.summary(),
        }
        if ms_page is not None:
            pps_p = n_pairs_all / (ms_page / 1e3)
            line["e2e_pageable"] = {"value": windows_p / (ms_page / 1e3), "unit": "windows/s", "ms_per_step": ms_page,
                                    "pairs_per_sec": pps_p,
                                    "api": "nightcore_analyzer.run_batch(list of numpy array pairs) — pageable memory in"}
        if not args.no_cpu_baseline and world == 1:
            procs = max(1, min(cores, args.cpu_procs or cores))
            arm = CpuArm(args.pair_sec, procs, args.cpu_sample or max(1, procs // 4), distinct)
            try:
                w, n, wall = arm.step()
            finally:
                arm.close()
            line["cpu_baseline"] = {"value": w / wall, "unit": "windows/s", "cores": procs, "kind": "port",
                                    "pairs_per_sec": n / wall, "audio_sec_per_sec": audio_seconds(n / wall, args.pair_sec),
                                    "sample": arm.sample_text() + f"; one step, {wall:.1f} s wall"}
        print(json.dumps(line), flush=True)
    if args.dump_outputs:
        # `res` is the last timed step of the resident path, the one `value` measures
        dump_outputs(args.dump_outputs, res, my_ids, f"rank{rank}_" if world > 1 else "")
    if world > 1:
        dist.destroy_process_group()



# --------------------------------------------------------------------------------------- per-family lines (configs 2-4)
def run_family(args):
    """BASELINE configs 2 / 3 / 4 as their own lines (not the contract line): one kernel family each, inputs resident
    in HBM, CUDA events around K steps, per-kernel event times from the library profiler, roofline of the family's
    dominant kernel on SURVEY §8(d)'s algorithmic figures."""
    import scipy.signal
    import torch
    from nightcore_analyzer import _engine, _native, pitch as npitch, xcorr as nxcorr
    from oracle import synth
    torch.cuda.set_device(0)
    eng = _engine.get_engine()
    peak, peak_kind = load_peaks()
    cfg = args.config
    if cfg == 4:
        sr, n_pairs = 44100, args.family_pairs or 16
        base = []
        for k in range(2):
            a = np.tile(synth.synth(4000 + k, 60.0, sr, bpm=124.0 + k), 10)            # 10 minutes = 26 460 000 samples
            b = scipy.signal.resample_poly(a, 1000, 1003).astype(np.float32)
            b = (b + np.random.default_rng(k).standard_normal(len(b)).astype(np.float32) * 0.01).astype(np.float32)
            base.append((a, b))
        pairs = [base[i % 2] for i in range(n_pairs)]
        audio, off, ln = eng.pack([t for p in pairs for t in p])
        tabs = [nxcorr._search_tables(int(ln[2 * i]), int(ln[2 * i + 1]), sr, 20, 3.0, 0.05, 0.10) for i in range(n_pairs)]
        win, stride = tabs[0][3], tabs[0][4]
        a_pos = np.concatenate([off[2 * i] + t[0] + t[5] for i, t in enumerate(tabs)])
        b_lo = np.concatenate([off[2 * i + 1] + t[0] + t[6] for i, t in enumerate(tabs)])
        n_cand = np.concatenate([t[7] for t in tabs])
        alg_bytes = float(sum(4 * (win + (int(c) - 1) * stride + win) for c in n_cand if c > 0))

        def step():
            return eng.xcorr_search_dev(audio, audio, a_pos, b_lo, n_cand, win, stride, nxcorr.XCORR_RMS_GATE)

        def check(out):
            bj = out[0].cpu().numpy()
            return {"windows_matched": int((bj >= 0).sum()), "windows": int(len(bj))}
        units, unit, metric, kernel = n_pairs, "pairs/s", "xcorr_pairs_per_sec", "xcorr_blocks_kernel"
        workload = (f"config 4: waveform cross-correlation speed search, {n_pairs} pairs of 10 min at 44.1 kHz "
                    f"(2 distinct, tiled), 20 windows x ~64 candidates of {win} samples each")
        bound_note = "memory bound (0.5 flop/B): algorithmic bytes = per window, the A window + its B search span, once"
    elif cfg == 2:
        sr = SR
        y = np.tile(synth.synth(2000, 60.0, sr), 60)                                  # 60 minutes = 79 380 000 samples
        audio, off, ln = eng.pack([y])
        frames = 1 + len(y) // 64
        alg_bytes = float(frames * 260)

        def step():
            return eng.tempo_segments_dev(audio, off, ln, np.array([120.0]), 64, sr)

        def check(out):
            return {"lag": int(out[3].cpu().numpy()[0]), "beats": int(out[5].cpu().numpy()[0])}
        units, unit, metric, kernel = frames, "frames/s", "hop64_frames_per_sec", "stft_logmel_kernel[hop<=128]"
        workload = "config 2: hop-64 onset envelope + tempogram lag + beat tracking of one 60-minute track (1 240 313 frames)"
        bound_note = "compute bound (AI 249 flop/B): FP32 fraction of the STFT kernel is the binding one"
    else:
        sr, n_pairs = SR, args.family_pairs or 125
        distinct = make_pairs(range(min(N_DISTINCT, n_pairs)), args.pair_sec)
        tracks = [t for i in range(n_pairs) for t in distinct[i % len(distinct)]]
        audio, off, ln = eng.pack(tracks)
        jobs = [(i, off[2 * i + 1], ln[2 * i + 1], off[2 * i], ln[2 * i]) for i in range(n_pairs)]
        n_chunks = sum(2 * len(npitch._chunk_bounds(int(ln[2 * i + 1]), int(ln[2 * i]), sr)) for i in range(n_pairs))
        alg_bytes = float(n_chunks * 1764048)

        def step():
            return npitch.chroma_shifts_staged(audio, jobs, sr)

        def check(out):
            return {"median_shift_st": float(np.median(np.concatenate(out)))}
        units, unit, metric, kernel = n_chunks, "chunks/s", "chroma_chunks_per_sec", "cqt_tc_kernel"
        workload = (f"config 3: CQT-chroma pitch stage (tuning, 6 decimations, 7-octave tcgen05 contraction, fold, cyclic "
                    f"xcorr) of {n_pairs} pairs = {n_chunks} twenty-second chunks")
        bound_note = "tensor-pipe kernel: see profiles/ for the ncu tensor-pipe utilisation"
    for _ in range(max(3, args.warmup)):
        out = step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = eng.launches
    with ClockSampler(0) as clk:
        e0.record()
        for _ in range(args.steps):
            out = step()
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    launches = (eng.launches - l0) // max(1, args.steps)
    _native.lib.ncfa_profile_enable(1)
    step()
    torch.cuda.synchronize()
    prof = _native.profile_report()
    _native.lib.ncfa_profile_enable(0)
    total = sum(v[1] for v in prof.values()) or 1e-9
    table = {k: {"launches": v[0], "ms": round(v[1], 4), "share": round(v[1] / total, 4)}
             for k, v in sorted(prof.items(), key=lambda kv: -kv[1][1])}
    kn, kms = prof.get(kernel, (1, ms))
    fam_bytes = alg_bytes if cfg != 3 else alg_bytes
    line = {"metric": metric, "value": units / (ms / 1e3), "unit": unit, "n_gpus": 1, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms, "higher_is_better": True, "dtype": "f32/f64",
            "data": "synthetic (oracle/synth.py), resident in HBM", "config": {"workload": workload},
            "gpu_launches": int(launches), "result": check(out),
            "roofline": {"bound": "tensor" if cfg == 3 else "hbm", "kernel": kernel, "launches": kn,
                         "ms_per_launch": kms / max(kn, 1), "algorithmic_bytes_per_step": fam_bytes,
                         "achieved": fam_bytes / (kms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": fam_bytes / (kms * 1e-3) / 1e9 / peak, "peak_kind": peak_kind, "traffic": None,
                         "whole_step_gbs": fam_bytes / (ms * 1e-3) / 1e9, "note": bound_note},
            "kernels": table, "clocks": clk.summary()}
    print(json.dumps(line), flush=True)


def run_single_pair(args):
    """BASELINE config 1 (the reference's own CPU-runnable case): latency of ONE 3-minute pair through the drop-in
    `pipeline.run_arrays` (host arrays in, AnalysisResult out) beside the CPU port on one core.  Not the contract line."""
    import torch
    from nightcore_analyzer import pipeline as npipe
    from oracle import pipeline_port
    nc, src = make_pairs([0], args.pair_sec, 1)[0]
    for _ in range(2):
        res = npipe.run_arrays(nc, src, SR, log=None)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = npipe.run_arrays(nc, src, SR, log=None)
    torch.cuda.synchronize()
    gpu_ms = 1e3 * (time.perf_counter() - t0) / args.steps
    t0 = time.perf_counter()
    want = pipeline_port.run_arrays(nc, src, SR, log=None)
    cpu_s = time.perf_counter() - t0
    same = (res.tempo_ratio, res.tempo_ci) == want["tempo"] and (res.ibi_ratio, res.ibi_ci) == want["ibi"] and \
        res.nc_pitches_raw == want["nc_hz"]
    print(json.dumps({"metric": "single_pair_latency_ms", "value": gpu_ms, "unit": "ms", "config": {
        "workload": "config 1: single synthetic 3-min pair, full pipeline through pipeline.run_arrays", "pair_sec": args.pair_sec},
        "cpu_port_seconds_1core": cpu_s, "speedup_vs_1core": cpu_s * 1e3 / gpu_ms, "identical_to_cpu_port": bool(same),
        "tempo_ratio": res.tempo_ratio, "ibi_ratio": res.ibi_ratio, "classification": res.classification}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="graft", choices=["graft", "reference"])
    ap.add_argument("--config", type=int, default=5, choices=[2, 3, 4, 5], help="BASELINE config (5 = the contract line)")
    ap.add_argument("--pairs", type=int, default=1000, help="total track pairs per step (all ranks)")
    ap.add_argument("--pair-sec", type=float, default=PAIR_SEC)
    ap.add_argument("--sub-batch", type=int, default=0, help="pairs analysed per device pass (per rank); 0 = 125")
    ap.add_argument("--workers", type=int, default=2, help="host threads / CUDA streams the sub-batches are dealt to")
    ap.add_argument("--no-pitch", action="store_true")
    ap.add_argument("--no-ibi", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-pageable", action="store_true", help="skip the pageable-memory e2e figure")
    ap.add_argument("--cpu-sample", type=int, default=0, help="pairs per CPU step (default: cores // 4)")
    ap.add_argument("--cpu-procs", type=int, default=0)
    ap.add_argument("--family-pairs", type=int, default=0, help="pairs of the --config 3 / 4 family lines")
    ap.add_argument("--single-pair", action="store_true", help="config 1: latency of one pair through pipeline.run_arrays")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step as DIR/<name>.npy (config 5 GPU run)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.single_pair or args.impl != "graft" or args.config != 5):
        ap.error("--dump-outputs applies to the config 5 GPU run")
    if args.single_pair:
        return run_single_pair(args)
    if args.impl == "reference":
        return run_reference(args)
    if args.config != 5:
        return run_family(args)
    run_gpu(args)


if __name__ == "__main__":
    main()
