#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's config.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Metric: audio-seconds rendered per wall-second ("x realtime") of the batched single-band STFT
quantize+distort pipeline (configs[1]: 4096 synthetic 10 s mono clips per GPU, default n_fft/hop,
pre-quant -> wavefold -> post-quant -> limiter, quantize_mode="spectral_bins").

One "step" = one render of the whole per-GPU batch.  `value` is timed with the batch already in
HBM; `e2e` is the same render through the public API (`process_batch`) from pinned HOST buffers,
host<->device copies inside the timed region.  One JSON line is printed by rank 0.

--dump-outputs DIR writes what the last timed step returned, as DIR/y.npy (float32 [clips, samples]): the rendered
clips of a fixed, seeded sample of DUMP_CLIPS clips of rank 0's batch (61 MB).  The inputs are seeded, so two builds
run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the source tree as it found it

SR = 48000
CLIP_SECONDS = 10
N_SAMPLES = SR * CLIP_SECONDS
WORKLOAD = "configs[1]: 4096 synthetic 10 s mono clips/GPU, single-band STFT pre-quant->wavefold->post-quant->limiter, n_fft 2048 hop 512, spectral_bins defaults"
# --workload multiband: BASELINE configs[2] (not the default bench line; for the record in profiles/)
WORKLOAD_MB = "configs[2]: 4096 synthetic 10 s mono clips/GPU, multiband: LR4 crossover @300 Hz, low-band saturation, high-band STFT chain + lookahead limiter, n_fft 2048 hop 512"
RENDER_KW = {"quantize_mode": "spectral_bins"}   # process_audio keyword arguments of the selected workload (the STFT path)
METRIC = "audio-seconds/sec for batched STFT quantize+distort pipeline"
UNIT = "audio-s/s"
DUMP_CLIPS = 32


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------ CPU arm
def _cpu_worker(args):
    seed, n, sr, kw = args   # kw travels explicitly: the pool's workers are spawned and do not see RENDER_KW
    import contextlib
    import io

    import numpy as np  # noqa: F401
    from oracle import qd_oracle as orc
    from quantumdistortion_b200 import synth
    x = synth.bass_clip(seed, n, sr)
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(io.StringIO()):
        y, _ = orc.process_audio(x, sr, **kw)
    return time.perf_counter() - t0, float(abs(y).max())


def cpu_baseline(clips_per_core: int, pool=None):
    """Oracle port (oracle/qd_oracle.py + oracle/qd_seq.c) on all host cores, whole clips of the same
    synthetic workload.  Returns (audio-s/s, cores, n_clips, wall seconds)."""
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    n_clips = cores * clips_per_core
    own = pool is None
    if own:
        pool = mp.get_context("spawn").Pool(cores)
    try:
        pool.map(_cpu_worker, [(10_000 + i, 4800, SR, dict(RENDER_KW)) for i in range(cores)])  # import + warm-up, untimed
        t0 = time.perf_counter()
        pool.map(_cpu_worker, [(i, N_SAMPLES, SR, dict(RENDER_KW)) for i in range(n_clips)], chunksize=1)
        wall = time.perf_counter() - t0
    finally:
        if own:
            pool.close()
            pool.join()
    return n_clips * CLIP_SECONDS / wall, cores, n_clips, wall


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (oracle port; the reference itself is pure Python
    and cannot travel to the GPU box) on every host core.  Rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import multiprocessing as mp
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "-s"])
    cores = os.cpu_count() or 1
    per_core = 2
    times = []
    with mp.get_context("spawn").Pool(cores) as pool:
        for i in range(args.warmup + args.steps):
            v, cores, n_clips, wall = cpu_baseline(per_core, pool)
            if i >= args.warmup:
                times.append(wall)
    ms = 1e3 * sum(times) / len(times)
    value = cores * per_core * CLIP_SECONDS / (ms / 1e3)
    sample = f"{cores * per_core} of the 4096 clips per step ({per_core} per core), full 10 s each"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------ GPU arm
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap,utilization.gpu")

    def __init__(self, index: int):
        self.index = index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, pw, reasons = [], [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for line in out.splitlines():
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                clk, cmax, power, util = float(parts[0]), float(parts[1]), float(parts[2]), float(parts[7])
            except ValueError:
                continue
            if util < 50.0:  # keep only samples taken under load
                continue
            sm.append(clk)
            mx.append(cmax)
            pw.append(power)
            for nm, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples_under_load": len(sm), "reasons": sorted(reasons)}


def copy_ceiling(xh, yh, chunk: int, dev, world: int, reps: int = 2):
    """Kernel-free copy benchmark with the e2e leg's traffic pattern: the pinned `xh` [clips, n] H2D and a same-sized
    result D2H into the pinned `yh`, in chunks of `chunk` clips on two streams at once.  Seconds per pass, max over ranks."""
    import torch
    import torch.distributed as dist
    clips, n, dt = int(xh.shape[0]), int(xh.shape[1]), xh.dtype
    dx = [torch.empty((chunk, n), dtype=dt, device=dev) for _ in range(2)]
    dy = [torch.zeros((chunk, n), dtype=dt, device=dev) for _ in range(2)]
    s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def one_pass():
        for i, b0 in enumerate(range(0, clips, chunk)):
            nb = min(chunk, clips - b0)
            with torch.cuda.stream(s_in):
                dx[i & 1][:nb].copy_(xh[b0:b0 + nb], non_blocking=True)
            with torch.cuda.stream(s_out):
                yh[b0:b0 + nb].copy_(dy[i & 1][:nb], non_blocking=True)
        torch.cuda.synchronize(dev)

    one_pass()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for _ in range(reps):
        one_pass()
    t = (time.perf_counter() - t0) / reps
    if world > 1:
        tt = torch.tensor([t], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t = float(tt.item())
    return t


GROWL = dict(key="F", scale="minor", snap_strength=0.9, smear=0.3, distortion_mode="wavefold",
             distortion_params={"fold_amount": 5.0, "bias": 0.1, "drive": 1.0, "warmth": 0.5}, limiter_ceiling_db=-1.0)
# BASELINE configs[2..4], device-resident, for the record inside the driver's own run (not the headline)
OTHER_CONFIGS = [
    ("configs[2] multiband LR4 @300 Hz", dict(use_multiband=True, crossover_hz=300.0), 2048, None),
    ("configs[3] growl + multiband + bitcrush 0.5", dict(GROWL, use_multiband=True, spectral_fx_mode="bitcrush", spectral_fx_strength=0.5), 2048, 1234),
    ("configs[3] growl + multiband + phase_dispersal 0.6", dict(GROWL, use_multiband=True, spectral_fx_mode="phase_dispersal", spectral_fx_strength=0.6), 2048, 1234),
    ("configs[3] growl + multiband + bin_scramble 0.55", dict(GROWL, use_multiband=True, spectral_fx_mode="bin_scramble", spectral_fx_strength=0.55), 2048, 1234),
    ("configs[3] growl + multiband + bin_scramble 0.3 (swap)", dict(GROWL, use_multiband=True, spectral_fx_mode="bin_scramble", spectral_fx_strength=0.3), 2048, 1234),
    ("configs[4] n_fft 512", {}, 512, None),
    ("configs[4] n_fft 1024", {}, 1024, None),
    ("configs[4] n_fft 4096", {}, 4096, None),
    ("configs[4] n_fft 8192 (precision=auto -> float64 kernels)", {}, 8192, None),
]


def other_configs(qd, x, clips: int):
    """One device-resident number per BASELINE config outside the headline: `clips` clips x 10 s, 2 warm-ups, then the
    median of 3 individually timed renders (CUDA events)."""
    import torch
    out = []
    xs = x[:clips]
    for name, kw, n_fft, seed in OTHER_CONFIGS:
        try:
            r = qd.make_renderer(N_SAMPLES, SR, n_fft, seeds=seed, quantize_mode="spectral_bins", **kw)
            r.set_fx_seeds(clips, seed)
            nclips = clips if n_fft < 8192 else max(1, clips // 4)    # float64 parity path: a quarter of the clips
            xi = xs[:nclips]
            for _ in range(2):   # two warm-ups: the second one makes torch's allocator create the second output block
                y, _ = r.render_device(xi)
            torch.cuda.synchronize()
            times = []
            for _ in range(3):   # each render timed on its own: the record keeps the median and says how far the others were
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                y, _ = r.render_device(xi)
                e1.record()
                torch.cuda.synchronize()
                times.append(e0.elapsed_time(e1))
            times.sort()
            ms = times[1]
            out.append({"config": name, "clips": nclips, "ms_per_render": round(ms, 3), "ms_min_max": [round(times[0], 3), round(times[2], 3)],
                        "audio_s_per_s": round(nclips * CLIP_SECONDS / (ms / 1e3)), "peak": round(float(y.abs().max()), 4)})
            del r, y
        except Exception as exc:  # noqa: BLE001 -- the record says what failed instead of hiding the headline
            out.append({"config": name, "error": f"{type(exc).__name__}: {exc}"})
    return out


def dump_outputs(out_dir: str, y) -> None:
    """DIR/y.npy: the rendered clips of a fixed, seeded sample of the batch, in ascending clip order."""
    import numpy as np
    import torch
    clips = np.sort(np.random.default_rng(0).choice(y.shape[0], min(DUMP_CLIPS, y.shape[0]), replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "y.npy"), y[torch.from_numpy(clips).to(y.device)].cpu().numpy())


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: quantumdistortion_b200 has no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    import quantumdistortion_b200 as qd
    from quantumdistortion_b200 import synth
    from quantumdistortion_b200.distributed import bind_to_gpu_numa

    numa_cpus = bind_to_gpu_numa(local)  # pinned host buffers below become node-local to this rank's GPU
    B = args.clips
    x = synth.bass_batch_torch(B, N_SAMPLES, SR, dev, seed=rank)  # each rank renders its own shard
    r = qd.make_renderer(N_SAMPLES, SR, **RENDER_KW)  # reference defaults, quantize_mode="spectral_bins"
    r.enable_timing(True)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident: `value`
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()  # nvidia-smi needs ~1 s to deliver its first sample: start it before the warm-up
    for _ in range(args.warmup):
        y, _ = r.render_device(x)
    barrier()
    r.read_timing()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        y, _ = r.render_device(x)
    ev1.record()
    barrier()
    ms_dev = max_over_ranks(ev0.elapsed_time(ev1)) / args.steps
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, y)
    timing = r.read_timing()
    launches = sum(v["launches"] for v in timing.values())
    audio_s = B * CLIP_SECONDS * world
    value = audio_s / (ms_dev / 1e3)

    # ---- parity spot check against the oracle (outside every timed region)
    parity = None
    if rank == 0 and args.check_clips > 0:
        from oracle import qd_oracle as orc
        errs, nulls = [], []
        for i in range(args.check_clips):
            idx = (i * 997) % B
            ref, _ = orc.process_audio(x[idx].cpu().numpy(), SR, **RENDER_KW)
            got = y[idx].cpu().numpy()
            errs.append(float(np.max(np.abs(got.astype(np.float64) - ref))))
            nulls.append(orc.null_test_db(got, ref))
        parity = {"clips": args.check_clips, "max_abs_err": max(errs), "null_db": max(nulls),
                  "tolerance": "max_abs<=1e-4, null<=-80 dBFS"}
        if max(errs) > 1e-4 or max(nulls) > -80.0:
            raise SystemExit(f"parity check failed: {parity}")

    # ---- end to end through the public API from pinned host memory: `e2e`
    y_dev_first = y[0].clone()
    del y
    x_host = torch.empty((B, N_SAMPLES), dtype=torch.float32, pin_memory=True)
    y_host = torch.empty((B, N_SAMPLES), dtype=torch.float32, pin_memory=True)
    x_host.copy_(x)
    torch.cuda.synchronize()
    for _ in range(max(1, args.warmup - 1)):
        qd.process_batch(x_host, SR, out=y_host, chunk_clips=args.chunk_clips, **RENDER_KW)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        qd.process_batch(x_host, SR, out=y_host, chunk_clips=args.chunk_clips, **RENDER_KW)
    torch.cuda.synchronize()
    ms_e2e = max_over_ranks((time.perf_counter() - t0) * 1e3) / args.steps
    barrier()
    if not torch.equal(y_host[0], y_dev_first.cpu()):
        raise SystemExit("host pipeline output differs from the device-resident render")
    e2e_value = audio_s / (ms_e2e / 1e3)

    # ---- what the machine's host<->device links deliver with the same traffic and no kernels: `e2e.copy_ceiling`
    t_copy = copy_ceiling(x_host, y_host, args.chunk_clips, dev, world)
    copy_ceil = {"audio_s_per_s": audio_s / t_copy, "gbs_each_way": 4.0 * B * N_SAMPLES * world / t_copy / 1e9,
                 "ms_per_step": t_copy * 1e3,
                 "how": "same pinned buffers, chunking and two copy streams as the e2e leg, H2D and D2H at once, no kernels; max over ranks"}

    # ---- the same render with 16-bit PCM on the PCIe link (what a WAV-to-WAV batch moves): `e2e_pcm16`, not the headline
    def leg_pcm16():
        # int16 views of the float buffers' pinned storage: no further pinned allocation
        x16 = x_host.view(torch.int16).view(-1)[:B * N_SAMPLES].view(B, N_SAMPLES)
        y16 = y_host.view(torch.int16).view(-1)[:B * N_SAMPLES].view(B, N_SAMPLES)
        x16.copy_((x * 32767.0).round().clamp_(-32768, 32767).to(torch.int16))
        torch.cuda.synchronize()
        for _ in range(2):
            qd.process_batch(x16, SR, out=y16, chunk_clips=args.chunk_clips, **RENDER_KW)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            qd.process_batch(x16, SR, out=y16, chunk_clips=args.chunk_clips, **RENDER_KW)
        torch.cuda.synchronize()
        ms_pcm = max_over_ranks((time.perf_counter() - t0) * 1e3) / args.steps
        barrier()
        t_copy16 = copy_ceiling(x16, y16, args.chunk_clips, dev, world)
        return {"value": audio_s / (ms_pcm / 1e3), "unit": UNIT, "ms_per_step": ms_pcm,
                "h2d_bytes_per_step": 2 * B * N_SAMPLES * world, "d2h_bytes_per_step": 2 * B * N_SAMPLES * world,
                "copy_ceiling": {"audio_s_per_s": audio_s / t_copy16, "gbs_each_way": 2.0 * B * N_SAMPLES * world / t_copy16 / 1e9},
                "frac_of_copy_ceiling": (audio_s / (ms_pcm / 1e3)) / (audio_s / t_copy16),
                "api": "process_batch(pinned int16 tensor, out=pinned int16 tensor): sample/32768 and lrint(y*32767) on the device"}

    e2e_pcm16 = None if args.no_extras else leg_pcm16()

    # ---- a caller that holds a plain NumPy array (pageable memory): library-side pinned staging ring, one step
    e2e_pageable = None
    if world == 1 and not args.no_pageable and not args.no_extras:
        Bp = min(B, 1024)
        xp = x[:Bp].cpu().numpy()
        t0 = time.perf_counter()
        yp, _ = qd.process_batch(xp, SR, chunk_clips=args.chunk_clips, **RENDER_KW)
        t_first = time.perf_counter() - t0
        del yp
        t0 = time.perf_counter()
        yp, _ = qd.process_batch(xp, SR, chunk_clips=args.chunk_clips, **RENDER_KW)
        tp = time.perf_counter() - t0
        e2e_pageable = {"value": Bp * CLIP_SECONDS / tp, "unit": UNIT, "clips": Bp, "ms": tp * 1e3, "first_call_ms": t_first * 1e3,
                        "api": "process_batch(numpy float32 array) -> numpy array: input staged through the library's pinned ring by "
                               "copy threads, result written by the device into page-locked memory (allocation inside the timing; "
                               "the first call also pays the page-locking)"}
        if not np.array_equal(yp[0], y_dev_first.cpu().numpy()):
            raise SystemExit("pageable host path differs from the device-resident render")
        del xp, yp
    del x_host, y_host

    # ---- the limiter-engaged variant of the same batch (the headline workload never reaches the ceiling)
    def leg_loud():
        variants = {}
        x_loud = (x * 6.0).clamp_(-1.5, 1.5)
        for _ in range(2):
            yl, _ = r.render_device(x_loud)
        barrier()
        r.read_timing()
        ev0.record()
        for _ in range(args.steps):
            yl, _ = r.render_device(x_loud)
        ev1.record()
        barrier()
        ms_loud = max_over_ranks(ev0.elapsed_time(ev1)) / args.steps
        t_loud = r.read_timing()
        ceiling = 10.0 ** (-1.0 / 20.0)
        variants["loud"] = {"what": "the same batch as clamp(6 x, -1.5, 1.5): the wavefolded signal exceeds the -1 dB ceiling on every clip, so the limiter scan runs",
                            "ms_per_step": ms_loud, "value": audio_s / (ms_loud / 1e3), "unit": UNIT,
                            "kernel_ms_per_step": {k: v["ms"] / args.steps for k, v in t_loud.items() if v["launches"]},
                            "output_peak": float(yl.abs().max()), "ceiling": ceiling,
                            "clips_limited_frac": float((yl.abs().amax(dim=1) >= ceiling * 0.999).float().mean())}
        if rank == 0 and args.check_clips > 0:
            from oracle import qd_oracle as orc
            ref, _ = orc.process_audio(x_loud[1].cpu().numpy(), SR, **RENDER_KW)
            err = float(np.max(np.abs(yl[1].cpu().numpy().astype(np.float64) - ref)))
            variants["loud"]["parity_max_abs_err"] = err
            if err > 1e-4:
                raise SystemExit(f"parity check of the loud variant failed: {err}")
        # every clip limited: the same loud batch against a -6 dB ceiling (the wavefold saturates near +-1, so only about
        # half the clips cross the default -1 dB ceiling)
        r6 = qd.make_renderer(N_SAMPLES, SR, limiter_ceiling_db=-6.0, **RENDER_KW)
        r6.enable_timing(True)
        for _ in range(2):
            yl, _ = r6.render_device(x_loud)
        barrier()
        r6.read_timing()
        ev0.record()
        for _ in range(args.steps):
            yl, _ = r6.render_device(x_loud)
        ev1.record()
        barrier()
        ms6 = max_over_ranks(ev0.elapsed_time(ev1)) / args.steps
        t6 = r6.read_timing()
        c6 = 10.0 ** (-6.0 / 20.0)
        variants["loud_ceiling_-6dB"] = {"what": "the loud batch with limiter_ceiling_db = -6: the limiter scan runs on every clip",
                                         "ms_per_step": ms6, "value": audio_s / (ms6 / 1e3), "unit": UNIT,
                                         "kernel_ms_per_step": {k: v["ms"] / args.steps for k, v in t6.items() if v["launches"]},
                                         "output_peak": float(yl.abs().max()), "ceiling": c6,
                                         "clips_limited_frac": float((yl.abs().amax(dim=1) >= c6 * 0.999).float().mean())}
        del x_loud, yl
        return variants

    variants = None if args.no_extras else leg_loud()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (spectral pass), from CUDA events on its launch stream
    peak, peak_src = _peaks()
    spec = timing["spectral"]
    spec_ms = spec["ms"] / max(spec["launches"], 1)
    alg_bytes = 8.0 * B * N_SAMPLES  # read float32 x once + write float32 y once per pass (SURVEY.md 8(d))
    achieved = alg_bytes / (spec_ms / 1e3) / 1e9
    step_share = {k: v["ms"] / args.steps for k, v in timing.items() if v["launches"]}
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": None, "kernel": "qd::spec_pass_kernel<float,1024,8,TS,noFX,NG=2>", "ms_per_launch": spec_ms,
                "algorithmic_bytes_per_launch": alg_bytes, "peak_source": peak_src,
                "kernel_ms_per_step": step_share,
                "note": "the pass is bound by instruction issue and shared-memory wavefronts (about 600 flop per sample), "
                        "not by HBM; the limiter launch skips clips that never exceed the ceiling (gain exactly 1); see DESIGN.md"}
    # the roofs that actually bind the pass (SURVEY.md 8(d): report both): FP32 arithmetic and instruction issue
    import ctypes as C
    from quantumdistortion_b200 import _lib
    tf = C.c_double(0.0)
    _lib.check(_lib.load().qd_measure_fp32_peak(C.byref(tf), None))
    frames = B * (1 + N_SAMPLES // 512)
    FLOP_PER_FRAME = 152e3   # SURVEY.md 8(d): two 2048-point real FFTs (61 kflop each) + 30 kflop of bin math per frame and pass
    fp32_achieved = FLOP_PER_FRAME * frames / (spec_ms / 1e3) / 1e12
    roofline.update({"fp32_peak_tflops": tf.value, "fp32_achieved_tflops": fp32_achieved, "fp32_frac": fp32_achieved / tf.value if tf.value else None,
                     "fp32_peak_source": "qd_measure_fp32_peak: fma.rn.f32x2 (FFMA2) chains, measured on this box in this run",
                     "algorithmic_flop_per_launch": FLOP_PER_FRAME * frames})
    ncu_issue = os.path.join(ROOT, "profiles", "spec_issue_per_frame.json")
    if os.path.exists(ncu_issue):
        try:
            ij = json.load(open(ncu_issue))
            sm_hz = (clocks.get("sm_mhz") or 1965.0) * 1e6
            cyc = spec_ms / 1e3 * sm_hz * ij.get("sms", 148) / frames
            roofline.update({"cycles_per_frame_per_sm": cyc, "issue_bound_cycles_per_frame": ij["warp_instructions_per_frame"] / 4.0,
                             "issue_frac": ij["warp_instructions_per_frame"] / 4.0 / cyc,
                             "smem_wavefronts_per_frame": ij.get("smem_wavefronts_per_frame"),
                             "smem_frac": (ij["smem_wavefronts_per_frame"] / cyc) if ij.get("smem_wavefronts_per_frame") else None,
                             "issue_source": ij.get("source")})
        except Exception:  # noqa: BLE001
            pass
    ncu_traffic = os.path.join(ROOT, "profiles", "spec_traffic_bytes_per_launch.json")
    if os.path.exists(ncu_traffic):
        try:
            tj = json.load(open(ncu_traffic))
            roofline["traffic"] = tj["bytes_per_sample"] * B * N_SAMPLES
            roofline["traffic_source"] = tj.get("source")
        except Exception:  # noqa: BLE001
            pass

    others = None
    if world == 1 and args.other_clips > 0 and not args.no_extras:
        sampler2 = ClockSampler(local)
        sampler2.start()
        time.sleep(1.0)          # nvidia-smi needs about a second to deliver its first sample
        others = other_configs(qd, x, args.other_clips)
        others.append({"clocks_during_other_configs": sampler2.stop()})

    cpu = None
    if not args.no_cpu_baseline and world == 1:   # reported on rank 0 at N = 1 only
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "-s"])
        v, cores, n_clips, wall = cpu_baseline(args.cpu_clips_per_core)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{n_clips} of the {B} clips ({args.cpu_clips_per_core} per core), full 10 s each, {wall:.1f} s wall",
               "note": "oracle port with the limiter/IIR loops in C; the reference's own Python limiter loop is about 10x slower (SURVEY.md 6.2: 1.63x realtime per core)"}

    print(json.dumps({
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "clips_per_gpu": B, "samples_per_clip": N_SAMPLES, "sample_rate": SR,
                   "parallelism": f"dp{world} (clips sharded, no collective)",
                   "l2": "inputs (7.9 GB per GPU) are far larger than the 126 MB L2; no flush needed"},
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e, "h2d_bytes_per_step": 4 * B * N_SAMPLES * world,
                "d2h_bytes_per_step": 4 * B * N_SAMPLES * world, "chunk_clips": args.chunk_clips,
                "host_numa_cpus": numa_cpus, "copy_ceiling": copy_ceil, "frac_of_copy_ceiling": e2e_value / copy_ceil["audio_s_per_s"],
                "api": "quantumdistortion_b200.process_batch(pinned host tensor, out=pinned host tensor)"},
        "e2e_pcm16": e2e_pcm16, "e2e_pageable": e2e_pageable, "variants": variants, "other_configs": others,
        "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks, "parity": parity,
    }))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--clips", type=int, default=4096, help="clips per GPU (BASELINE config: 4096)")
    ap.add_argument("--chunk-clips", type=int, default=128)
    ap.add_argument("--check-clips", type=int, default=2)
    ap.add_argument("--cpu-clips-per-core", type=int, default=4)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-pageable", action="store_true", help="skip the pageable-memory (NumPy) e2e leg")
    ap.add_argument("--no-extras", action="store_true", help="headline only: skip e2e_pcm16, e2e_pageable, variants and other_configs")
    ap.add_argument("--other-clips", type=int, default=1024, help="clips for the device-resident numbers of the other BASELINE configs (0 = skip)")
    ap.add_argument("--workload", default="single_band", choices=["single_band", "multiband"],
                    help="single_band = BASELINE configs[1] (the bench line); multiband = configs[2], for the record")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help=f"write the last timed step's output (a seeded sample of {DUMP_CLIPS} clips) to DIR/y.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.workload == "multiband":
        global WORKLOAD
        WORKLOAD = WORKLOAD_MB
        RENDER_KW.update(use_multiband=True, crossover_hz=300.0, lowband_drive=1.0)
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
