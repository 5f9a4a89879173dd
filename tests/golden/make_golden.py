#!/usr/bin/env python
"""Generate tests/golden/*.npz by running the LIVE reference (build container only).

    python tests/golden/make_golden.py            # needs /root/reference

The reference is imported read-only from /root/reference (it cannot travel to the GPU
box); its outputs are committed as small fixtures so the oracle restatement
(oracle/qd_oracle.py) and the CUDA path can be checked anywhere.  Nothing in tests/,
smoke() or bench.py reads /root/reference at run time.
"""
from __future__ import annotations

import contextlib
import io
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)
sys.path.insert(0, "/root/reference")

import qd_cases  # noqa: E402
from quantum_distortion.dsp import pipeline as ref_pipeline  # noqa: E402
from quantum_distortion.dsp import quantizer as ref_q  # noqa: E402
from quantum_distortion.dsp import spectral_fx as ref_fx  # noqa: E402
from quantum_distortion.dsp import stft_utils as ref_stft  # noqa: E402
from quantum_distortion.dsp.crossover import design_linkwitz_riley_sos, linkwitz_riley_split  # noqa: E402
from quantum_distortion.dsp.distortion import apply_distortion  # noqa: E402
from quantum_distortion.dsp.limiter import peak_limiter  # noqa: E402
from quantum_distortion.dsp.saturation import saturate_lowband  # noqa: E402


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def gen_pipeline():
    out = {}
    for name, (kind, seed, n, sr, n_fft, rng_seed, kw) in qd_cases.CASES.items():
        x = qd_cases.make_signal(kind, seed, n, sr)
        ref_pipeline.N_FFT_DEFAULT = n_fft  # SURVEY.md section 0.2
        if rng_seed is not None:
            np.random.seed(rng_seed)
        y, taps = quiet(ref_pipeline.process_audio, x, sr, quantize_mode="spectral_bins", **kw)
        ref_pipeline.N_FFT_DEFAULT = 2048
        out[f"{name}/x"] = x
        out[f"{name}/y"] = y
        out[f"{name}/pre_quant"] = taps["pre_quant"].astype(np.float32)
        out[f"{name}/post_dist"] = taps["post_dist"].astype(np.float32)
        print(f"pipeline {name}: n={n} peak={np.max(np.abs(y)):.4f}")
    qd_cases.save_golden("pipeline", out)


def gen_tables():
    out = {}
    for sr, n_fft, key, scale in [(48000, 2048, "D", "minor"), (44100, 2048, "D", "minor"),
                                  (48000, 2048, "F", "minor"), (48000, 512, "D", "minor"),
                                  (48000, 1024, "Bb", "dorian"), (48000, 4096, "C", "major"),
                                  (48000, 8192, "D", "minor"), (48000, 2048, "A", "pentatonic"),
                                  (96000, 2048, "G#", "harmonic_minor"), (48000, 2048, "Eb", "mixolydian")]:
        freqs = np.fft.rfftfreq(n_fft, d=1.0 / sr)
        tag = f"{sr}_{n_fft}_{key}_{scale}"
        out[f"tb/{tag}"] = ref_q.build_target_bins_for_freqs(freqs, key, scale).astype(np.int64)
        out[f"mask/{tag}"] = ref_pipeline._build_quantize_band_mask(freqs, 110.0, 5000.0)
    freqs = np.fft.rfftfreq(2048, d=1.0 / 48000)
    out["mask/wide"] = ref_pipeline._build_quantize_band_mask(freqs, 0.0, 0.0)
    for f0 in (55.0, 110.0, 441.3):
        out[f"htb/{f0}"] = ref_q.build_harmonic_target_bins(freqs, f0).astype(np.int64)
    # reference KAT (tests/test_quantizer.py:10-23)
    out["tb/kat4"] = ref_q.build_target_bins_for_freqs(np.array([0.0, 430.0, 440.0, 450.0]), "A", "minor")
    qd_cases.save_golden("tables", out)
    print("tables:", len(out))


def gen_analysis():
    """avg_cents_offset_from_scale (dsp/analyses.py:53-142) on a few clips, raw and rendered."""
    from quantum_distortion.dsp.analyses import avg_cents_offset_from_scale
    out = {}
    for name, (kind, seed, n, sr, key, scale, kw) in qd_cases.ANALYSIS_CASES.items():
        x = qd_cases.make_signal(kind, seed, n, sr)
        avg, per = avg_cents_offset_from_scale(x, sr, key, scale, **kw)
        out[f"{name}/x"], out[f"{name}/avg"], out[f"{name}/per_peak"] = x, np.float64(avg), per
        print(f"analysis {name}: avg {avg:.3f} cents over {len(per)} peaks")
    qd_cases.save_golden("analysis", out)


def gen_autotune():
    """quantize_mode="autotune_v1": every stage of dsp/autotune.py on one clip, then whole renders."""
    from quantum_distortion.dsp import autotune as ref_at
    out = {}
    sr = 48000
    x = qd_cases.make_signal("tone", 0, qd_cases.AT_N, sr)
    cfg = ref_at.AutotuneV1Config(key="D", scale="minor")
    res = ref_at.apply_autotune_v1(x, sr, cfg)
    det = ref_at.make_detector_sidechain(res.body_band, sr, cfg.detector_low_hz, cfg.detector_high_hz)
    out["st/x"], out["st/sub"], out["st/body"], out["st/air"], out["st/det"] = x, res.sub_band, res.body_band, res.air_band, det
    out["st/ratio_track"], out["st/corrected"], out["st/output"] = res.diagnostics.ratio_track, res.corrected_body, res.output
    out["st/sub_layer"] = ref_at.generate_sub_layer(x, sr, cfg)
    out["st/env"] = ref_at.envelope_follow(x, sr)
    feats = []
    for start in range(0, len(det), 512):   # the detector's own framing (dsp/autotune.py:217-236)
        fr = det[start:start + 4096]
        if len(fr) < 4096:
            fr = np.pad(fr, (0, 4096 - len(fr)), mode="constant")
        p, c = ref_at.detect_pitch_yin(fr, sr, min_freq=max(60.0, 110.0 * 0.65), max_freq=3000.0)
        feats.append([float(np.sqrt(np.mean(fr * fr))), ref_at._spectral_flatness(fr), p, c])
    out["st/features"] = np.array(feats)
    # a hand-made ratio track exercises the shifter away from 1 (both directions, wraps of both taps)
    rt = (1.0 + 0.2 * np.sin(2.0 * np.pi * 3.0 * np.arange(len(x)) / sr)).astype(np.float32)
    out["st/ratio_manual"], out["st/shift_manual"] = rt, ref_at.granular_pitch_shift(res.body_band, rt)
    out["st/nearest"] = np.array([ref_at.nearest_scale_freq(f, "D", "minor") for f in (97.3, 233.1, 440.0, 1234.5)])
    for name, (kind, seed, n, srr, kw) in qd_cases.AUTOTUNE_CASES.items():
        xx = qd_cases.make_signal(kind, seed, n, srr)
        y, taps = quiet(ref_pipeline.process_audio, xx, srr, quantize_mode="autotune_v1", **kw)
        out[f"{name}/x"], out[f"{name}/y"] = xx, y
        out[f"{name}/pre_quant"], out[f"{name}/post_dist"] = taps["pre_quant"].astype(np.float32), taps["post_dist"].astype(np.float32)
        print(f"autotune {name}: n={n} peak={np.max(np.abs(y)):.4f} moved={np.max(np.abs(y - xx)):.4f}")
    qd_cases.save_golden("autotune", out)


def gen_stages():
    out = {}
    rng = np.random.default_rng(7)
    sr, n_fft = 48000, 2048
    freqs = np.fft.rfftfreq(n_fft, d=1.0 / sr)
    tb = ref_q.build_target_bins_for_freqs(freqs, "D", "minor")
    mask = ref_pipeline._build_quantize_band_mask(freqs, 110.0, 5000.0)
    # --- quantize_spectrum on random frames (incl. a silent frame and exact zeros)
    mags = np.abs(rng.standard_normal((6, 1025))) * np.exp(-np.arange(1025) / 200.0)[None, :]
    mags[3] = 0.0
    mags[4, ::3] = 0.0
    phases = rng.uniform(-np.pi, np.pi, size=(6, 1025))
    out["q/mags"], out["q/phases"] = mags, phases
    for tag, (snap, smear, smooth, m) in {"default": (1.0, 0.1, True, mask), "growl": (0.9, 0.3, True, mask),
                                          "nosmooth": (0.75, 0.4, False, mask), "nomask": (1.0, 0.1, True, None),
                                          "smear0": (1.0, 0.0, True, mask), "smear1": (0.5, 1.0, True, mask)}.items():
        nm, nph = [], []
        for t in range(mags.shape[0]):
            a, b = ref_q.quantize_spectrum(mags[t], phases[t], freqs, "D", "minor", snap, smear, smooth,
                                           target_bins=tb, active_mask=m)
            nm.append(a)
            nph.append(b)
        out[f"q/{tag}/mags"], out[f"q/{tag}/phases"] = np.array(nm), np.array(nph)
    # --- STFT / iSTFT
    x = qd_cases.make_signal("bass", 40, 9000, sr)
    for nf in (512, 2048):
        S, fr = ref_stft.stft_mono(x, sr, n_fft=nf)
        out[f"stft/{nf}/S"] = S
        out[f"stft/{nf}/y"] = ref_stft.istft_mono(S, sr, n_fft=nf, length=len(x))
    out["stft/x"] = x
    # --- spectral FX per frame with seeded global RNG
    fm = np.abs(rng.standard_normal(1025)) * np.exp(-np.arange(1025) / 150.0)
    fp = rng.uniform(-np.pi, np.pi, size=1025)
    out["fx/mag"], out["fx/phase"] = fm, fp
    for tag, (mode, s) in {"bitcrush05": ("bitcrush", 0.5), "bitcrush03": ("bitcrush", 0.3),
                           "bitcrush08": ("bitcrush", 0.8), "disp06": ("phase_dispersal", 0.6),
                           "disp03": ("phase_dispersal", 0.3), "scr055": ("bin_scramble", 0.55),
                           "scr03": ("bin_scramble", 0.3), "scr09": ("bin_scramble", 0.9)}.items():
        np.random.seed(99)
        cfg = ref_pipeline._SpectralFXConfig(mode, s, {})
        frames_m, frames_p = [], []
        for _ in range(3):  # three consecutive frames consume the RNG in order
            a, b = ref_pipeline.apply_spectral_fx(fm.copy(), fp.copy(), cfg)
            frames_m.append(np.array(a))
            frames_p.append(np.array(b))
        out[f"fx/{tag}/mag"], out[f"fx/{tag}/phase"] = np.array(frames_m), np.array(frames_p)
    a, b = ref_fx.bitcrush(fm, fp, method="uniform", step=0.07, threshold=0.01)
    out["fx/uniform/mag"] = a
    # --- formant shift (cepstral lifter), incl. a frame with exact zeros and a 257-bin frame
    fz = fm.copy()
    fz[::5] = 0.0
    out["fx/formant/zeros_in"] = fz
    f257 = np.abs(rng.standard_normal(257)) * np.exp(-np.arange(257) / 40.0)
    out["fx/formant/in257"] = f257
    for st in (3.0, -5.0, 12.0, -0.5):
        out[f"fx/formant/{st}"] = ref_fx.formant_shift_frame(fm, freqs, st)
        out[f"fx/formant/zeros/{st}"] = ref_fx.formant_shift_frame(fz, freqs, st)
        out[f"fx/formant/257/{st}"] = ref_fx.formant_shift_frame(f257, np.fft.rfftfreq(512, d=1.0 / sr), st)
    # --- time-domain stages
    xl = qd_cases.make_signal("loud", 41, 6000, sr)
    out["td/x"] = xl
    out["td/wavefold"] = apply_distortion(xl, "wavefold", fold_amount=5.0, bias=0.1)
    out["td/tube"] = apply_distortion(xl, "tube", drive=4.0, warmth=0.7)
    for srr in (48000, 44100):
        y, g = peak_limiter(xl, srr, ceiling_db=-1.0, lookahead_ms=5.0, release_ms=30.0)
        out[f"td/lim/{srr}/y"], out[f"td/lim/{srr}/g"] = y, g
    lo, hi = linkwitz_riley_split(xl, sr, 300.0)
    out["td/xo/low"], out["td/xo/high"] = lo, hi
    sl, sh = design_linkwitz_riley_sos(sr, 300.0)
    out["td/xo/sos_low"], out["td/xo/sos_high"] = sl, sh
    out["td/sat"] = saturate_lowband(lo, drive=2.5)
    qd_cases.save_golden("stages", out)
    print("stages:", len(out))


def gen_frontend():
    out = {}
    for name, (kind, seed, n, sr, rng_seed, cfg, kw) in qd_cases.UI_CASES.items():
        x = qd_cases.make_signal(kind, seed, n, sr)
        np.random.seed(rng_seed)
        y, taps = quiet(ref_pipeline.process_audio, x, sr, quantize_mode="spectral_bins", config=cfg, **kw)
        out[f"{name}/x"], out[f"{name}/y"] = x, y
        print(f"ui {name}: peak={np.max(np.abs(y)):.4f}")
    qd_cases.save_golden("frontend", out)


def _run_case(x, sr, n_fft, rng_seed, kw, mode="spectral_bins"):
    ref_pipeline.N_FFT_DEFAULT = n_fft  # SURVEY.md section 0.2
    try:
        if rng_seed is not None:
            np.random.seed(rng_seed)
        return quiet(ref_pipeline.process_audio, x, sr, quantize_mode=mode, **kw)
    finally:
        ref_pipeline.N_FFT_DEFAULT = 2048


def _scramble_indices(n_bins: int, window: int, mode: str, seed: int, frames: int = 3) -> np.ndarray:
    """Source-bin indices of `frames` consecutive reference bin_scramble calls (dsp/spectral_fx.py:326-390),
    recovered from its OUTPUT on mags = 1..n_bins: out = mags[idx] * sum(mags) / (sum(mags[idx]) + 1e-12), so the
    smallest gap between distinct output values is the scale and out / scale - 1 is idx.  The recovered table is
    only accepted if it reproduces the reference's output bit for bit."""
    a = np.arange(1, n_bins + 1, dtype=np.float64)
    np.random.seed(seed)
    rows = []
    for _ in range(frames):
        out, _ph = ref_fx.bin_scramble(a, np.zeros(n_bins), window=window, mode=mode)
        u = np.unique(out)
        scale = float(np.min(np.diff(u)))
        idx = np.rint(out / scale).astype(np.int64) - 1
        assert idx.min() >= 0 and idx.max() < n_bins
        again = a[idx] * (np.sum(a) / (np.sum(a[idx]) + 1e-12))
        assert np.array_equal(again, out), "index recovery failed"
        rows.append(idx)
    return np.array(rows)


def gen_round2():
    """Round-2 fixtures: FX parameter overrides and FX at other n_fft (CASES_R2), autotune_v1 kept inside a
    multiband render, UI dicts that stay in autotune_v1, and integer scramble-index tables."""
    out = {}
    for name, (kind, seed, n, sr, n_fft, rng_seed, kw) in qd_cases.CASES_R2.items():
        x = qd_cases.make_signal(kind, seed, n, sr)
        y, taps = _run_case(x, sr, n_fft, rng_seed, kw)
        out[f"{name}/x"], out[f"{name}/y"] = x, y
        out[f"{name}/pre_quant"] = taps["pre_quant"].astype(np.float32)
        out[f"{name}/post_dist"] = taps["post_dist"].astype(np.float32)
        print(f"r2 {name}: n={n} n_fft={n_fft} peak={np.max(np.abs(y)):.4f}")
    for name, (kind, seed, n, sr, kw) in qd_cases.AT_MB_CASES.items():
        x = qd_cases.make_signal(kind, seed, n, sr)
        y, taps = quiet(ref_pipeline.process_audio, x, sr, **kw)     # quantize_mode left at the reference default
        out[f"{name}/x"], out[f"{name}/y"] = x, y
        out[f"{name}/pre_quant"] = taps["pre_quant"].astype(np.float32)
        out[f"{name}/post_dist"] = taps["post_dist"].astype(np.float32)
        print(f"r2 {name}: peak={np.max(np.abs(y)):.4f}")
    for name, (kind, seed, n, sr, rng_seed, cfg, kw) in qd_cases.UI_AT_CASES.items():
        x = qd_cases.make_signal(kind, seed, n, sr)
        y, taps = quiet(ref_pipeline.process_audio, x, sr, config=cfg, **kw)   # default mode unless the dict says otherwise
        out[f"{name}/x"], out[f"{name}/y"] = x, y
        print(f"r2 {name}: peak={np.max(np.abs(y)):.4f} moved={np.max(np.abs(y - x)):.4f}")
    # integer gate of the north-star: "scramble permutations must be bit-exact"
    for n_bins in (1025, 257):
        for tag, (window, mode) in {"pick_w9": (9, "random_pick"), "pick_w3": (3, "random_pick"),
                                    "pick_w15": (15, "random_pick"), "swap": (5, "swap")}.items():
            out[f"scr/{n_bins}/{tag}"] = _scramble_indices(n_bins, window, mode, seed=4321).astype(np.int16)
    # the draw of a randomized phase_dispersal frame, recovered the same way: phase_out - phase = jitter * rand_amt
    np.random.seed(4321)
    jit = []
    for _ in range(3):
        m, ph = ref_fx.phase_dispersal(np.ones(1025), np.zeros(1025), thresh=0.0, amount=0.0, randomized=True, rand_amt=1.0)
        jit.append(ph)
    out["scr/1025/jitter"] = np.array(jit)
    qd_cases.save_golden("round2", out)
    print("round2:", len(out), os.path.getsize(os.path.join(HERE, "round2.npz")) // 1024, "KiB")


def gen_refwav():
    """The reference's own audio files (BASELINE configs[0] = examples/example_bass.wav through scripts/render_cli.py:32,
    plus tests/data/*.wav): input samples, the literal default render (quantize_mode="autotune_v1"), the STFT-path
    render (quantize_mode="spectral_bins"), and the reference's committed renders tests/data/processed/
    *_multiband(.|_bitcrush).wav as a secondary known-answer test (SURVEY.md section 4)."""
    from scipy.io import wavfile
    out = {}
    for name, rel in qd_cases.REF_WAVS.items():
        sr, d = wavfile.read(os.path.join("/root/reference", rel))
        assert d.dtype == np.int16 and d.ndim == 1
        x = d.astype(np.float32) / 32768.0          # io/audio_io.py:10-17 (libsndfile PCM16 -> float)
        out[f"{name}/x16"], out[f"{name}/sr"] = d, np.int64(sr)
        y_def, _ = quiet(ref_pipeline.process_audio, x, sr)                                   # scripts/render_cli.py:32
        y_sb, _ = quiet(ref_pipeline.process_audio, x, sr, quantize_mode="spectral_bins")
        out[f"{name}/y_default"], out[f"{name}/y_spectral_bins"] = y_def, y_sb
        print(f"refwav {name}: sr={sr} n={len(d)} default peak {np.max(np.abs(y_def)):.4f}, spectral_bins peak {np.max(np.abs(y_sb)):.4f}")
        for suffix in ("multiband", "multiband_bitcrush"):
            pth = os.path.join("/root/reference/tests/data/processed", f"{name}_{suffix}.wav")
            if os.path.exists(pth):
                sr2, k = wavfile.read(pth)
                assert sr2 == sr and k.dtype == np.int16
                out[f"{name}/kat_{suffix}"] = k
    inputs = {k: v for k, v in out.items() if k.endswith(("/x16", "/sr"))}
    qd_cases.save_golden("refwav", inputs)
    qd_cases.save_golden("refwav_renders", {k: v for k, v in out.items() if k not in inputs})
    print("refwav:", len(out), os.path.getsize(os.path.join(HERE, "refwav.npz")) // 1024, "KiB")


def gen_scenarios():
    """The reference's own pipeline-level test scenarios (qd_cases.REF_SCENARIOS): its signals and its arguments through
    the LIVE process_audio, output and taps kept, so that the CUDA path is checked on exactly what the reference's test
    suite exercises."""
    out = {}
    for name, (spec, sr, rng_seed, kw, prop, cite) in qd_cases.REF_SCENARIOS.items():
        x = qd_cases.scenario_signal(spec, sr)
        if rng_seed is not None:
            np.random.seed(rng_seed)
        y, taps = quiet(ref_pipeline.process_audio, x, sr=sr, **kw)
        assert y.dtype == np.float32 and set(taps) == {"input", "pre_quant", "post_dist", "output"}
        out[f"{name}/x"], out[f"{name}/y"] = x, y
        out[f"{name}/pre_quant"] = np.asarray(taps["pre_quant"], dtype=np.float32)
        out[f"{name}/post_dist"] = np.asarray(taps["post_dist"], dtype=np.float32)
        print(f"scenario {name} ({cite}): n={len(x)} peak={np.max(np.abs(y)):.4f} moved={np.max(np.abs(y - x[:len(y)])):.4f}")
    qd_cases.save_golden("scenarios", out)
    print("scenarios:", len(out), os.path.getsize(os.path.join(HERE, "scenarios.npz")) // 1024, "KiB")


def _ref_wav_slice(name, seconds):
    d = np.load(os.path.join(HERE, "refwav.npz"))
    sr = int(d[f"{name}/sr"])
    return d[f"{name}/x16"][: int(sr * seconds)], sr


def gen_scripts():
    """The process_audio / process_file_to_file calls of the reference's scripts/ (qd_cases.SCRIPT_SCENARIOS,
    HARNESS_SCENARIOS) on the first second of its own WAV files, through the LIVE reference; the file-to-file renders go
    through the reference's own harness and WAV layer and are kept as the PCM16 samples it wrote."""
    import tempfile
    import types
    from pathlib import Path
    from scipy.io import wavfile
    if "soundfile" not in sys.modules:
        # python-soundfile / libsndfile are not in this image.  The reference's io/audio_io.py only calls sf.read and
        # sf.write on 16-bit PCM WAV files; this stand-in gives them libsndfile's PCM_16 conventions (read: sample /
        # 32768 as float64; write: round-half-even of x * 0x7FFF, clipped), so that the reference's harness and WAV layer
        # run unmodified on top of it.
        sf = types.ModuleType("soundfile")

        def _read(path, always_2d=False):
            sr, d = wavfile.read(str(path))
            assert d.dtype == np.int16
            return d.astype(np.float64) / 32768.0, sr

        def _write(path, audio, sr):
            pcm = np.clip(np.rint(np.asarray(audio, dtype=np.float64) * 32767.0), -32768, 32767).astype(np.int16)
            wavfile.write(str(path), int(sr), pcm)

        sf.read, sf.write = _read, _write
        sys.modules["soundfile"] = sf
    from quantum_distortion.dsp.harness import process_file_to_file
    out = {}
    for name, (wav, seconds, rng_seed, _kw, cite) in qd_cases.SCRIPT_SCENARIOS.items():
        x16, sr = _ref_wav_slice(wav, seconds)
        x = x16.astype(np.float32) / 32768.0
        if rng_seed is not None:
            np.random.seed(rng_seed)
        y, taps = quiet(ref_pipeline.process_audio, audio=x, sr=sr, **qd_cases.script_scenario_kwargs(name))
        out[f"{name}/y"] = y
        out[f"{name}/pre_quant"] = np.asarray(taps["pre_quant"], dtype=np.float32)
        out[f"{name}/post_dist"] = np.asarray(taps["post_dist"], dtype=np.float32)
        print(f"script {name} ({cite}): n={len(x)} peak={np.max(np.abs(y)):.4f}")
    with tempfile.TemporaryDirectory() as td:
        for name, (wav, seconds, rng_seed, preset, _ep, cite) in qd_cases.HARNESS_SCENARIOS.items():
            x16, sr = _ref_wav_slice(wav, seconds)
            src, dst = Path(td) / f"{name}_in.wav", Path(td) / f"{name}_out.wav"
            wavfile.write(str(src), sr, x16)
            if rng_seed is not None:
                np.random.seed(rng_seed)
            quiet(process_file_to_file, src, dst, preset=preset, extra_params=qd_cases.harness_extra_params(name))
            sr2, y16 = wavfile.read(str(dst))
            assert sr2 == sr and y16.dtype == np.int16 and y16.shape == x16.shape
            out[f"{name}/y16"] = y16
            print(f"harness {name} ({cite}): n={len(x16)} peak={np.max(np.abs(y16.astype(np.int32)))}")
    qd_cases.save_golden("scripts", out)
    print("scripts:", len(out), os.path.getsize(os.path.join(HERE, "scripts.npz")) // 1024, "KiB")


if __name__ == "__main__":
    if sys.argv[1:] == ["scripts"]:
        gen_scripts()
        sys.exit(0)
    if sys.argv[1:] == ["scenarios"]:
        gen_scenarios()
        sys.exit(0)
    if sys.argv[1:] == ["round2"]:
        gen_round2()
        sys.exit(0)
    if sys.argv[1:] == ["refwav"]:
        gen_refwav()
        sys.exit(0)
    if sys.argv[1:] == ["analysis"]:   # only that file
        gen_analysis()
        sys.exit(0)
    if sys.argv[1:] == ["autotune"]:
        gen_autotune()
        sys.exit(0)
    gen_autotune()
    gen_analysis()
    gen_frontend()
    gen_tables()
    gen_stages()
    gen_pipeline()
    gen_round2()
    gen_refwav()
    gen_scenarios()
    gen_scripts()
    for f in ("tables.npz", "stages.npz", "pipeline.npz", "frontend.npz", "analysis.npz"):
        print(f, os.path.getsize(os.path.join(HERE, f)) // 1024, "KiB")
