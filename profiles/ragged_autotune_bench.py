"""Ragged-batch throughput of quantize_mode="autotune_v1" (the reference's default mode) on one GPU: 1024 clips of 1-20 s
(48 kHz, seeded lengths, the synth bass recipe built on the device by synth.bass_batch_torch and cut to length), default
autotune_v1 parameters.

  (a) the ragged render: device-resident (qd_autotune_render_device_varlen on the packed buffer, one call) and end to
      end from packed pinned host buffers (AutotuneRenderer.render_host_varlen), float32 and PCM16 on the link;
  (b) the same total audio as a uniform batch of mean-length clips (qd_autotune_render_device): the ceiling for (a);
  (c) one process_batch call per distinct length (what a list of files of different lengths cost before ragged
      batches in this mode), on a subset from NumPy, extrapolated per clip to the whole workload (labelled as such).

Also checks a seeded sample of ragged outputs bit for bit against single-clip renders, reports the workspace bytes per
call, and with --dump DIR writes a seeded sample of uniform outputs (DIR/at_uniform.npy) so that two builds can be
compared output for output.  Every shape is rendered once before it is timed; timed legs repeat --reps times.

    python profiles/ragged_autotune_bench.py [--clips 1024] [--reps 5] [--out profiles/r04_ragged_autotune.json]
    python profiles/ragged_autotune_bench.py --uniform-only --dump DIR   # only the seeded uniform sample
"""
from __future__ import annotations

import argparse
import ctypes as C
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


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def stats(xs):
    xs = sorted(xs)
    return {"min": xs[0], "median": xs[len(xs) // 2], "max": xs[-1], "runs": xs}


def dump_uniform(path):
    """A seeded uniform batch (256 clips x 10 s) through the default mode; the bits two builds must share are those
    of 8 seeded clips (15 MB)."""
    import quantumdistortion_b200 as qd
    from quantumdistortion_b200 import synth
    x = synth.bass_batch_torch(256, 10 * SR, SR, "cuda", seed=11)
    y, _ = qd.process_batch(x, SR)
    pick = np.sort(np.random.default_rng(3).choice(256, size=8, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "at_uniform.npy"), y[pick].cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clips", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--subset", type=int, default=16)
    ap.add_argument("--check", type=int, default=12)
    ap.add_argument("--dump", default=None)
    ap.add_argument("--uniform-only", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_ragged_autotune.json"))
    args = ap.parse_args()

    import torch
    assert torch.cuda.is_available(), "ragged_autotune_bench measures on the GPU only"
    if args.dump:
        dump_uniform(args.dump)
    if args.uniform_only:
        return
    import quantumdistortion_b200 as qd
    from quantumdistortion_b200 import _lib, synth
    from quantumdistortion_b200.pipeline import make_renderer, pack_layout

    rng = np.random.default_rng(2024)
    lengths = rng.integers(1 * SR, 20 * SR + 1, size=args.clips)
    total_audio_s = float(lengths.sum()) / SR
    n_max = int(lengths.max())
    src = synth.bass_batch_torch(args.clips, n_max, SR, "cuda", seed=7)
    starts, span = pack_layout(lengths, 4)
    ends = starts + lengths
    xf = torch.zeros(span, dtype=torch.float32, device="cuda")
    for i in range(args.clips):
        xf[starts[i]:ends[i]] = src[i, :lengths[i]]
    del src
    d_starts = torch.from_numpy(starts).cuda()
    d_lengths = torch.from_numpy(lengths.astype(np.int32)).cuda()
    r = make_renderer(n_max, SR, ragged=True)
    lib = _lib.load()
    res = {"card": card(), "clips": args.clips, "lengths_s": [1, 20], "total_audio_s": total_audio_s,
           "span_samples": int(span), "longest": n_max, "config": "autotune_v1 defaults (PipelineConfig())",
           "unit": "audio-seconds per second",
           "workspace_bytes_device_call": int(lib.qd_autotune_workspace_bytes_varlen(C.byref(r.params), args.clips,
                                                                                    int(span)))}

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        out = []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            out.append(time.perf_counter() - t0)
        return out

    # (a) device-resident, one call
    y_holder = {}

    def ragged_dev():
        y_holder["y"], _ = r.render_device_varlen(xf, d_starts, d_lengths, span, n_max)
    t = timed(ragged_dev)
    res["a_device"] = {"s": stats(t), "audio_s_per_s": stats([total_audio_s / v for v in t])}
    y_dev = y_holder["y"].cpu().numpy()
    r._ws = None   # the host legs allocate their own (chunk-sized) workspace
    torch.cuda.empty_cache()

    # (a) end to end from packed pinned host buffers, float32 and PCM16
    xh = xf.cpu().pin_memory()
    yh = torch.empty_like(xh, pin_memory=True)
    budget = 128 * int(span // args.clips)
    t = timed(lambda: r.render_host_varlen(xh, yh, starts, lengths, chunk_samples=budget))
    res["a_e2e_f32"] = {"s": stats(t), "audio_s_per_s": stats([total_audio_s / v for v in t]), "chunk_samples": budget,
                        "workspace_bytes_per_chunk": int(lib.qd_autotune_workspace_bytes_varlen(
                            C.byref(r.params), 128, budget + 3 * 128))}
    assert np.array_equal(yh.numpy()[starts[0]:ends[0]], y_dev[starts[0]:ends[0]])
    xh16 = torch.from_numpy(np.clip(np.rint(xh.numpy() * 32767.0), -32768, 32767).astype(np.int16)).pin_memory()
    yh16 = torch.empty_like(xh16, pin_memory=True)
    t = timed(lambda: r.render_host_varlen(xh16, yh16, starts, lengths, chunk_samples=budget))
    res["a_e2e_pcm16"] = {"s": stats(t), "audio_s_per_s": stats([total_audio_s / v for v in t]), "chunk_samples": budget}
    del xh16, yh16
    r._ws = None
    torch.cuda.empty_cache()

    # (b) the same total audio as uniform mean-length clips, one device call (chunk = the whole batch)
    n_mean = int(round(lengths.mean()))
    xu = synth.bass_batch_torch(args.clips, n_mean, SR, "cuda", seed=7)
    ru = make_renderer(n_mean, SR)
    t = timed(lambda: ru.render_device(xu, chunk_clips=args.clips))
    uni_audio = args.clips * n_mean / SR
    res["b_uniform_device"] = {"s": stats(t), "audio_s_per_s": stats([uni_audio / v for v in t]), "n_mean": n_mean,
                               "workspace_bytes": int(lib.qd_autotune_workspace_bytes(C.byref(ru.params), args.clips))}
    ru.close()
    del xu
    torch.cuda.empty_cache()

    # correctness: a seeded sample of ragged outputs against single-clip renders (device path)
    pick = np.random.default_rng(5).choice(args.clips, size=min(args.check, args.clips), replace=False)
    ok = 0
    for i in pick:
        yi, _ = qd.process_batch(xf[starts[i]:ends[i]].reshape(1, -1), SR)
        ok += int(np.array_equal(yi[0].cpu().numpy(), y_dev[starts[i]:ends[i]]))
    res["bit_identical_sample"] = {"checked": int(len(pick)), "identical": ok}
    assert ok == len(pick), res["bit_identical_sample"]

    # (c) one process_batch per distinct length (NumPy in), on a subset
    sub = [xh.numpy()[starts[i]:ends[i]].copy() for i in range(args.subset)]
    qd.process_batch(sub[0][None, :], SR)   # first-call costs (module load) out of the window
    t0 = time.perf_counter()
    for c in sub:
        qd.process_batch(c[None, :], SR)
    dt = time.perf_counter() - t0
    sub_audio = float(lengths[:args.subset].sum()) / SR
    res["c_per_length_calls"] = {"subset_clips": args.subset, "s": dt, "s_per_clip": dt / args.subset,
                                 "audio_s_per_s": sub_audio / dt,
                                 "extrapolated_s_for_all_clips": dt / args.subset * args.clips,
                                 "note": "extrapolated per clip from the subset, not measured on the whole workload"}
    qd.process_batch(sub[:4], SR)
    t0 = time.perf_counter()
    qd.process_batch(sub, SR)
    dt = time.perf_counter() - t0
    res["a_list_api_subset"] = {"subset_clips": args.subset, "s": dt, "audio_s_per_s": sub_audio / dt,
                                "note": "process_batch(list of NumPy clips) on the same subset: packing + one ragged call"}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: (v["audio_s_per_s"]["median"] if isinstance(v, dict) and isinstance(v.get("audio_s_per_s"), dict)
                          else v.get("audio_s_per_s") if isinstance(v, dict) else v) for k, v in res.items()}))


if __name__ == "__main__":
    main()
