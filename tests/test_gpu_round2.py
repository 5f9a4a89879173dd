"""GPU (B200), round-2 parity cases through the C ABI against fixtures of the LIVE reference
(tests/golden/round2.npz, refwav.npz; generator tests/golden/make_golden.py):

* spectral_fx_params overrides, uniform bitcrush, spectral FX at n_fft 512 / 1024 / 4096 / 8192, float64 FX kernels;
* the boundary: a bare ``process_audio(x, sr)`` runs the reference's default mode, autotune_v1 survives inside a
  multiband render with snap_strength = 0, UI dicts hand their sub-layer keys to the autotune render;
* the reference's own audio files (BASELINE configs[0]) in both modes and its committed multiband renders (KAT).

Tolerance: the north-star's max-abs <= 1e-4 and null <= -80 dBFS unless a tighter bound is written at the call.
"""

import numpy as np
import pytest

import qd_cases
from oracle import qd_oracle as orc

MAX_ABS = 1e-4
NULL_DB = -80.0
SB = {"quantize_mode": "spectral_bins"}


@pytest.fixture(scope="module")
def qd():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import quantumdistortion_b200 as q
    from quantumdistortion_b200 import _lib
    assert _lib.load().qd_device_count() >= 1, "libqd_b200.so sees no sm_100 device"
    return q


@pytest.fixture(scope="module")
def r2():
    return qd_cases.Golden("round2")


@pytest.fixture(scope="module")
def pipe():
    return qd_cases.Golden("pipeline")


@pytest.fixture(scope="module")
def wav():
    return qd_cases.Golden("refwav")


@pytest.fixture(scope="module")
def renders():
    return qd_cases.Golden("refwav_renders")


def _check(got, ref, what, max_abs=MAX_ABS):
    got = np.asarray(got)
    assert got.dtype == np.float32 and got.shape == ref.shape, what
    err = float(np.max(np.abs(got.astype(np.float64) - ref))) if ref.size else 0.0
    null = orc.null_test_db(got, ref) if ref.size else -200.0
    assert err <= max_abs, f"{what}: max abs err {err:.3e}"
    assert null <= NULL_DB, f"{what}: null {null:.1f} dB"
    return err


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(qd_cases.CASES_R2))
def test_round2_cases_vs_reference_fixtures(qd, r2, name):
    kind, seed, n, sr, n_fft, rng_seed, kw = qd_cases.CASES_R2[name]
    x = r2.input(name, qd_cases.make_signal(kind, seed, n, sr))
    if rng_seed is not None:
        np.random.seed(rng_seed)
    y, taps = qd.process_audio(x, sr, n_fft=n_fft, **SB, **kw)   # precision="auto"
    _check(*r2.at(f"{name}/y", y), f"{name}/y")
    _check(*r2.at(f"{name}/pre_quant", taps["pre_quant"]), f"{name}/pre_quant")
    _check(*r2.at(f"{name}/post_dist", taps["post_dist"]), f"{name}/post_dist")


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(qd_cases.F64_CASES))
def test_float64_fx_kernels_vs_reference_fixtures(qd, r2, pipe, name):
    """precision="float64" on the FX / formant variants of the pass, n_fft 512 ... 4096."""
    cases, fix = (qd_cases.CASES, pipe) if name in qd_cases.CASES else (qd_cases.CASES_R2, r2)
    kind, seed, n, sr, n_fft, rng_seed, kw = cases[name]
    if rng_seed is not None:
        np.random.seed(rng_seed)
    x = fix.input(name, qd_cases.make_signal(kind, seed, n, sr))
    y, taps = qd.process_audio(x, sr, n_fft=n_fft, precision="float64", **SB, **kw)
    _check(*fix.at(f"{name}/y", y), f"{name}/y f64", 5e-6)
    _check(*fix.at(f"{name}/pre_quant", taps["pre_quant"]), f"{name}/pre_quant f64", 5e-6)


def test_auto_precision_never_picks_a_path_outside_tolerance():
    """precision="auto": float64 kernels for every n_fft 8192 configuration (SURVEY.md section 7.4 item 2)."""
    from quantumdistortion_b200.pipeline import _resolve_kwargs
    mb = dict(SB, use_multiband=True)
    for kw in ({}, dict(mb, spectral_fx_mode="bitcrush", spectral_fx_strength=0.5),
               dict(mb, spectral_fx_mode="bin_scramble", spectral_fx_strength=0.55), {"spectral_freeze": True},
               {"formant_shift": 3.0}):
        assert _resolve_kwargs(20000, 48000, 8192, dict(SB, **kw))[0].params.precision == 1, kw


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(qd_cases.AT_MB_CASES))
def test_autotune_kept_inside_multiband_snap0(qd, r2, name):
    """dsp/pipeline.py:1326-1327, :1076, :537-601: default mode + use_multiband + snap_strength = 0."""
    kind, seed, n, sr, kw = qd_cases.AT_MB_CASES[name]
    x = r2.input(name, qd_cases.make_signal(kind, seed, n, sr))
    y, taps = qd.process_audio(x, sr, **kw)
    _check(*r2.at(f"{name}/y", y), f"{name}/y", 2e-6)
    _check(*r2.at(f"{name}/pre_quant", taps["pre_quant"]), f"{name}/pre_quant", 2e-6)
    _check(*r2.at(f"{name}/post_dist", taps["post_dist"]), f"{name}/post_dist", 2e-6)
    yb, _ = qd.process_batch(np.stack([x] * 3), sr, **kw)        # host pipeline, no taps
    assert np.array_equal(yb[2], y)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(qd_cases.UI_AT_CASES))
def test_ui_dict_keeps_autotune_and_its_sub_keys(qd, r2, name):
    kind, seed, n, sr, _rng, cfg, kw = qd_cases.UI_AT_CASES[name]
    y, _ = qd.process_audio(r2.input(name, qd_cases.make_signal(kind, seed, n, sr)), sr, config=cfg, **kw)
    _check(*r2.at(f"{name}/y", y), name)


@pytest.mark.gpu
def test_bare_call_is_the_reference_default(qd):
    """process_audio(x, sr), PipelineConfig(), from_preset() and the file harness without overrides run
    quantize_mode="autotune_v1" (config.py:44, :77, :140) -- compared with the live-reference fixture."""
    g = qd_cases.Golden("autotune")
    kind, seed, n, sr, _kw = qd_cases.AUTOTUNE_CASES["at_tone_default"]
    x = g.input("at_tone_default", qd_cases.make_signal(kind, seed, n, sr))
    y, taps = qd.process_audio(x, 48000)
    _check(*g.at("at_tone_default/y", y), "bare process_audio")
    _check(*g.at("at_tone_default/pre_quant", taps["pre_quant"]), "bare process_audio pre_quant")
    y2, _ = qd.process_audio(x, 48000, pipeline_config=qd.PipelineConfig())
    assert np.array_equal(y, y2)
    yb, _ = qd.process_batch(x[None, :], 48000)
    assert np.array_equal(yb[0], y)


# ---------------------------------------------------------------------------------------------- the reference's own files
def _wav_input(wav, name):
    return wav[f"{name}/x16"].astype(np.float32) / 32768.0, int(wav[f"{name}/sr"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(qd_cases.REF_WAVS))
def test_reference_files_both_modes(qd, wav, renders, name):
    """BASELINE configs[0]: examples/example_bass.wav (and tests/data/*.wav) through process_audio -- the literal
    scripts/render_cli.py:32 call (default mode) and the STFT path."""
    x, sr = _wav_input(wav, name)
    y, _ = qd.process_audio(x, sr)
    _check(*renders.at(f"{name}/y_default", y), f"{name} default mode")
    y, _ = qd.process_audio(x, sr, **SB)
    _check(*renders.at(f"{name}/y_spectral_bins", y), f"{name} spectral_bins")


@pytest.mark.gpu
def test_render_cli_semantics_on_example_bass(qd, wav, renders, tmp_path):
    """scripts/render_cli.py: load_audio -> process_audio(audio, sr) -> save_audio, here through the file harness with
    no preset and no overrides; the written PCM16 file against the reference's float output."""
    from quantumdistortion_b200.audio_io import float_to_pcm16, load_audio, save_audio
    x16, sr = wav["example_bass/x16"], int(wav["example_bass/sr"])
    from scipy.io import wavfile
    src, dst = tmp_path / "example_bass.wav", tmp_path / "out" / "example_bass_qd.wav"
    wavfile.write(str(src), sr, x16)
    qd.process_file_to_file(src, dst)
    got, sr2 = load_audio(dst)
    assert sr2 == sr
    got, ref = renders.at("example_bass/y_default", got)
    lsb = np.abs(np.rint(got * 32768.0) - float_to_pcm16(ref).astype(np.float64))
    assert lsb.max() <= 4, lsb.max()     # 1e-4 = 3.3 steps of 16-bit PCM
    del save_audio


@pytest.mark.gpu
@pytest.mark.parametrize("name", [n for n in qd_cases.REF_WAVS if n != "example_bass"])
def test_reference_processed_renders_kat(qd, wav, renders, name):
    """SURVEY.md section 4: the reference's committed *_multiband.wav / *_multiband_bitcrush.wav renders, <= 6 PCM16 steps."""
    from quantumdistortion_b200.audio_io import float_to_pcm16
    x, sr = _wav_input(wav, name)
    kw = dict(SB, use_multiband=True, crossover_hz=300.0, sub_cut_hz=0.0, air_cut_hz=0.0)
    y, _ = qd.process_audio(x, sr, **kw)
    got, ref = renders.at(f"{name}/kat_multiband", float_to_pcm16(y))
    d = np.abs(got.astype(np.int32) - ref.astype(np.int32))
    assert int(d.max()) <= 6, int(d.max())
    y, _ = qd.process_audio(x, sr, spectral_fx_mode="bitcrush", spectral_fx_strength=0.5, **kw)
    got, ref = renders.at(f"{name}/kat_multiband_bitcrush", float_to_pcm16(y))
    d = np.abs(got.astype(np.int32) - ref.astype(np.int32))
    assert int(d.max()) <= 6, int(d.max())


@pytest.mark.gpu
def test_process_files_preview_and_per_file_seeds(qd, tmp_path, monkeypatch):
    """ADVICE r1: process_files honours preview mode like process_file_to_file, and a per-file seed list follows the
    files through the (length, sample rate) grouping."""
    from quantumdistortion_b200 import synth
    from quantumdistortion_b200.audio_io import load_audio, save_audio
    sr = 8000     # 10 s preview = 80 000 samples
    lens = (90000, 20000, 90000, 20000)
    ins, outs_a, outs_b = [], [], []
    for i, n in enumerate(lens):
        p = tmp_path / f"in{i}.wav"
        save_audio(p, synth.loud_clip(200 + i, n, sr), sr)
        ins.append(p)
        outs_a.append(tmp_path / "a" / f"{i}.wav")
        outs_b.append(tmp_path / "b" / f"{i}.wav")
    extra = dict(qd_cases.GROWL, use_multiband=True, spectral_fx_mode="bin_scramble", spectral_fx_strength=0.55,
                 preview_enabled=True)
    seeds = [31, 32, 33, 34]
    assert qd.process_files(list(zip(ins, outs_a)), extra_params=extra, seeds=seeds) == 4
    for i in range(4):
        np.random.seed(seeds[i])
        qd.process_file_to_file(ins[i], outs_b[i], extra_params=extra)
        a, _ = load_audio(outs_a[i])
        b, _ = load_audio(outs_b[i])
        assert a.shape == b.shape == (min(lens[i], 80000),)
        assert np.array_equal(a, b), i
    monkeypatch.setenv("DSP_PREVIEW_MODE", "1")
    extra.pop("preview_enabled")
    out = tmp_path / "c" / "0.wav"
    assert qd.process_files([(ins[0], out)], extra_params=extra, seeds=5) == 1
    assert load_audio(out)[0].shape == (80000,)


# ---------------------------------------------------------------------------------------------- host transport
@pytest.mark.gpu
def test_pcm16_transport_and_pageable_staging(qd):
    """qd_render_host_ex: 16-bit PCM on the PCIe link (converted on the device with the WAV layer's rules) and pageable
    host memory staged through the pinned ring -- every variant bit-identical to the device-resident render."""
    import torch
    from quantumdistortion_b200 import synth
    from quantumdistortion_b200.audio_io import float_to_pcm16
    n, sr, b = 30000, 48000, 5
    x16 = float_to_pcm16(np.stack([synth.loud_clip(300 + i, n, sr) * 0.6 for i in range(b)]))
    xf = x16.astype(np.float32) / 32768.0                      # what load_audio hands to process_audio
    kw = dict(SB, use_multiband=True, dry_wet=0.8)
    y_dev, _ = qd.process_batch(torch.from_numpy(xf).cuda(), sr, **kw)
    y_dev = y_dev.cpu().numpy()
    want16 = float_to_pcm16(y_dev)
    # NumPy arrays are pageable: 5 one-clip chunks wrap the 3-slot ring in both directions
    y_np, _ = qd.process_batch(xf, sr, chunk_clips=1, **kw)
    assert y_np.dtype == np.float32 and np.array_equal(y_np, y_dev)
    y16, _ = qd.process_batch(x16, sr, chunk_clips=1, **kw)
    assert y16.dtype == np.int16 and np.array_equal(y16, want16)
    # pinned int16 tensors (direct copies), then int16 in / float32 out
    xp = torch.from_numpy(x16).pin_memory()
    out16 = torch.empty_like(xp).pin_memory()
    qd.process_batch(xp, sr, out=out16, chunk_clips=2, **kw)
    assert np.array_equal(out16.numpy(), want16)
    outf = torch.empty((b, n), dtype=torch.float32).pin_memory()
    qd.process_batch(xp, sr, out=outf, chunk_clips=2, **kw)
    assert np.array_equal(outf.numpy(), y_dev)
    # the other mode (autotune_v1 host path: torch streams) with PCM16
    xt = float_to_pcm16(np.stack([synth.tone_clip(i, 12000, sr) for i in range(3)]))
    ya, _ = qd.process_batch(torch.from_numpy(xt.astype(np.float32) / 32768.0).cuda(), sr)
    ya16, _ = qd.process_batch(xt, sr, chunk_clips=2)
    assert np.array_equal(ya16, float_to_pcm16(ya.cpu().numpy()))
    with pytest.raises(ValueError):
        qd.process_batch(x16, sr, return_taps=True, **kw)


@pytest.mark.gpu
def test_pageable_staging_large_chunks(qd):
    """Chunks large enough for the multi-threaded staging copies (> 8 MB), more chunks than ring slots."""
    import torch
    from quantumdistortion_b200 import synth
    n, sr, b = 480000, 48000, 40
    x = synth.bass_batch_torch(b, n, sr, "cuda", seed=9)
    y_dev, _ = qd.process_batch(x, sr, **SB)
    x_np = x.cpu().numpy()
    y_np, _ = qd.process_batch(x_np, sr, chunk_clips=8, **SB)
    assert np.array_equal(y_np, y_dev.cpu().numpy())


@pytest.mark.gpu
def test_render_timing_struct(qd):
    """RenderTiming (dsp/pipeline.py:153-161) is filled from the CUDA events of the launch stream."""
    import torch
    from quantumdistortion_b200 import synth
    x = synth.bass_batch_torch(4, 48000, 48000, "cuda", seed=1)
    r = qd.make_renderer(48000, 48000, use_multiband=True, **SB)
    r.enable_timing(True)
    r.render_device(x)
    torch.cuda.synchronize()
    t = r.timing()
    assert t.launches == r.launches_per_render == 4 and t.spectral_ms > 0 and t.crossover_ms > 0 and t.limiter_ms > 0
    assert abs(t.total_ms - (t.spectral_ms + t.limiter_ms + t.crossover_ms + t.other_ms)) < 1e-9
    assert t.line().startswith("[RENDER_TIMING] mode=spectral_bins")
    r.enable_timing(False)
