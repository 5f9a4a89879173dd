"""Throughput of the scale-alignment metric's device half (spectral_peak_bins, qd_spectral_peaks_device[_varlen]) on
ragged batches, one GPU: 1024 clips of 1-20 s (48 kHz, seeded lengths, the synth bass recipe built on the device by
synth.bass_batch_torch and cut to length), n_fft 2048, topn 3, in float64 (the default) and float32.

  (a) the list call from CUDA tensors (packing on the device + one qd_spectral_peaks_device_varlen call), and that
      kernel call alone on the packed buffer, timed with CUDA events;
  (b) the same total audio as a uniform batch of mean-length clips (qd_spectral_peaks_device), CUDA events;
  (c) the list call from NumPy arrays end to end (host packing into pinned memory, copy, kernel, copy back), host
      clock around a call that returns host arrays;
  (d) one call per clip from NumPy, on a subset, extrapolated per clip to the whole workload (labelled as such).

Every shape runs once before it is timed; timed legs repeat --reps times.  A seeded sample of ragged outputs is checked
bit for bit against the same clips run alone.  The card's name and power limit are read in the same run.

    python profiles/ragged_peaks_bench.py [--clips 1024] [--reps 5] [--out profiles/r05_ragged_peaks.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

SR = 48000
N_FFT = 2048
TOPN = 3


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def stats(xs):
    xs = sorted(xs)
    return {"min": xs[0], "median": xs[len(xs) // 2], "max": xs[-1], "runs": xs}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clips", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--subset", type=int, default=16)
    ap.add_argument("--check", type=int, default=16)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_ragged_peaks.json"))
    args = ap.parse_args()

    import torch
    assert torch.cuda.is_available(), "ragged_peaks_bench measures on the GPU only"
    from quantumdistortion_b200 import _lib, analyses, synth
    from quantumdistortion_b200.pipeline import pack_layout

    rng = np.random.default_rng(2025)
    lengths = rng.integers(1 * SR, 20 * SR + 1, size=args.clips)
    total_audio_s = float(lengths.sum()) / SR
    n_max = int(lengths.max())
    src = synth.bass_batch_torch(args.clips, n_max, SR, "cuda", seed=7)
    clips_dev = [src[i, :lengths[i]].clone() for i in range(args.clips)]
    del src
    torch.cuda.empty_cache()
    starts, span = pack_layout(lengths, 4)
    hop = N_FFT // 4
    row0, frames, n_rows = analyses.peak_rows(starts, lengths, hop)
    lib = _lib.load()
    res = {"card": card(), "clips": args.clips, "lengths_s": [1, 20], "total_audio_s": total_audio_s,
           "span_samples": int(span), "longest": n_max, "frames": int(frames.sum()), "n_fft": N_FFT, "topn": TOPN,
           "unit": "audio-seconds per second", "timing": "CUDA events (a, b), host clock with a synchronise (c, d)"}

    def events(fn):
        fn()
        torch.cuda.synchronize()
        out = []
        for _ in range(args.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            out.append(e0.elapsed_time(e1) / 1e3)
        return out

    def host(fn):
        fn()
        torch.cuda.synchronize()
        out = []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            out.append(time.perf_counter() - t0)
        return out

    def leg(t, audio=total_audio_s, **extra):
        return dict({"s": stats(t), "audio_s_per_s": stats([audio / v for v in t])}, **extra)

    clips_np = [c.cpu().numpy() for c in clips_dev]
    for precision in ("float64", "float32"):
        kw = dict(n_fft=N_FFT, topn=TOPN, precision=precision)
        r = res[precision] = {}
        held = {}

        def list_dev():
            held["bins"] = analyses.spectral_peak_bins(clips_dev, **kw)
        r["a_list_cuda"] = leg(events(list_dev))

        xf = torch.cat([torch.cat([c, torch.zeros(int(s1 - s0 - len(c)), device="cuda")])
                        for c, s0, s1 in zip(clips_dev, starts, list(starts[1:]) + [span])])
        d_starts = torch.from_numpy(starts).cuda()
        d_lengths = torch.from_numpy(lengths.astype(np.int32)).cuda()
        bins = torch.empty((n_rows, TOPN), dtype=torch.int16, device="cuda")
        prec = {"float32": 0, "float64": 1}[precision]
        stream = torch.cuda.current_stream().cuda_stream

        def kernel_only():
            _lib.check(lib.qd_spectral_peaks_device_varlen(xf.data_ptr(), d_starts.data_ptr(), d_lengths.data_ptr(),
                                                           args.clips, n_max, N_FFT, TOPN, 10.0 ** (-60.0 / 20.0), prec,
                                                           bins.data_ptr(), stream))
        r["a_varlen_call_packed"] = leg(events(kernel_only))
        assert all(torch.equal(bins[r0:r0 + f], b) for r0, f, b in zip(row0.tolist(), frames.tolist(), held["bins"]))
        del xf, bins

        n_mean = int(round(lengths.mean()))
        xu = synth.bass_batch_torch(args.clips, n_mean, SR, "cuda", seed=7)
        r["b_uniform_cuda"] = leg(events(lambda: analyses.spectral_peak_bins(xu, **kw)),
                                  audio=args.clips * n_mean / SR, n_mean=n_mean)
        del xu
        torch.cuda.empty_cache()

        held_np = {}

        def list_np():
            held_np["bins"] = analyses.spectral_peak_bins(clips_np, **kw)
        r["c_list_numpy_e2e"] = leg(host(list_np))

        pick = np.sort(np.random.default_rng(5).choice(args.clips, size=min(args.check, args.clips), replace=False))
        ok = sum(int(np.array_equal(held_np["bins"][i], analyses.spectral_peak_bins(clips_np[i][None, :], **kw)[0]))
                 for i in pick)
        r["bit_identical_sample"] = {"checked": int(len(pick)), "identical": int(ok)}
        assert ok == len(pick), r["bit_identical_sample"]

        sub = clips_np[:args.subset]
        analyses.spectral_peak_bins(sub[0][None, :], **kw)
        t0 = time.perf_counter()
        for c in sub:
            analyses.spectral_peak_bins(c[None, :], **kw)
        dt = time.perf_counter() - t0
        sub_audio = float(lengths[:args.subset].sum()) / SR
        r["d_per_clip_calls"] = {"subset_clips": args.subset, "s": dt, "s_per_clip": dt / args.subset,
                                 "audio_s_per_s": sub_audio / dt,
                                 "extrapolated_s_for_all_clips": dt / args.subset * args.clips,
                                 "note": "extrapolated per clip from the subset, not measured on the whole workload"}
        print(precision, json.dumps({k: (v["audio_s_per_s"]["median"] if isinstance(v.get("audio_s_per_s"), dict)
                                         else v.get("audio_s_per_s", v)) for k, v in r.items()}), flush=True)

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"]}))


if __name__ == "__main__":
    main()
