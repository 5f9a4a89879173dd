"""GPU (B200): the CUDA path through the C ABI vs the oracle and the live-reference fixtures.

Tolerances are the north-star's: float32 audio max-abs error <= 1e-4 and null-test residual
<= -80 dBFS (reference tests/utils/audio_test_utils.py definition); integer tables are checked
bit-exact on the CPU in test_host_logic.py.
"""
import os

import numpy as np
import pytest

import qd_cases
from oracle import qd_oracle as orc
from quantumdistortion_b200 import synth


G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
MAX_ABS = 1e-4
NULL_DB = -80.0
SB = {"quantize_mode": "spectral_bins"}   # the STFT path; the default mode is the reference's "autotune_v1" (config.py:44)


@pytest.fixture(scope="module")
def qd():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import quantumdistortion_b200 as q
    from quantumdistortion_b200 import _lib
    lib = _lib.load()
    assert lib.qd_device_count() >= 1, "libqd_b200.so sees no sm_100 device"
    return q


@pytest.fixture(scope="module")
def pipe():
    return qd_cases.Golden("pipeline")


def _check(got, ref, what, max_abs=MAX_ABS):
    got = np.asarray(got)
    assert got.dtype == np.float32 and got.shape == ref.shape, what
    err = float(np.max(np.abs(got.astype(np.float64) - ref))) if ref.size else 0.0
    null = orc.null_test_db(got, ref) if ref.size else -200.0
    assert err <= max_abs, f"{what}: max abs err {err:.3e}"
    assert null <= NULL_DB, f"{what}: null {null:.1f} dB"
    return err


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(qd_cases.CASES))
def test_pipeline_vs_reference_fixtures(qd, pipe, name):
    kind, seed, n, sr, n_fft, rng_seed, kw = qd_cases.CASES[name]
    x = pipe.input(name, qd_cases.make_signal(kind, seed, n, sr))
    if rng_seed is not None:
        np.random.seed(rng_seed)  # the random spectral FX replay the global np.random state like the reference
    y, taps = qd.process_audio(x, sr, n_fft=n_fft, **SB, **kw)
    # precision="auto": float32 kernels, except sb_wide_mask (fan-in > 64) and nfft8192, which run in float64
    _check(*pipe.at(f"{name}/y", y), f"{name}/y")
    _check(*pipe.at(f"{name}/pre_quant", taps["pre_quant"]), f"{name}/pre_quant")
    _check(*pipe.at(f"{name}/post_dist", taps["post_dist"]), f"{name}/post_dist")
    assert np.array_equal(taps["input"], x) and np.array_equal(taps["output"], y)


@pytest.mark.gpu
def test_batch_vs_oracle_default_config(qd):
    """Config #2 shape (single-band defaults) on a small seeded batch, every clip against the oracle."""
    n, sr, b = 48000, 48000, 6
    x = np.stack([synth.bass_clip(i, n, sr) if i % 2 == 0 else synth.noise_clip(i, n) for i in range(b)])
    y, taps = qd.process_batch(x, sr, return_taps=True, **SB)
    worst = 0.0
    for i in range(b):
        ref, rt = orc.process_audio(x[i], sr)
        worst = max(worst, _check(y[i], ref, f"clip {i}"))
        _check(taps["pre_quant"][i], rt["pre_quant"], f"clip {i} pre_quant")
        _check(taps["post_dist"][i], rt["post_dist"], f"clip {i} post_dist")
    print(f"worst max-abs error vs oracle: {worst:.3e}")
    y2, _ = qd.process_batch(x, sr, **SB)  # host pipeline path (qd_render_host) must agree bit for bit
    assert np.array_equal(y, y2)


@pytest.mark.gpu
def test_multiband_batch_vs_oracle(qd):
    n, sr = 30000, 48000
    x = np.stack([synth.loud_clip(40 + i, n, sr) for i in range(3)])
    kw = dict(use_multiband=True, crossover_hz=300.0, lowband_drive=1.5, dry_wet=0.9)
    y, taps = qd.process_batch(x, sr, return_taps=True, **SB, **kw)
    for i in range(3):
        ref, rt = orc.process_audio(x[i], sr, **kw)
        _check(y[i], ref, f"mb clip {i}")
        _check(taps["post_dist"][i], rt["post_dist"], f"mb clip {i} post_dist")


@pytest.mark.gpu
def test_tiling_and_batch_size_do_not_change_bits(qd):
    """A clip rendered alone (time-tiled over many CTAs) equals the same clip inside a large batch
    (whole-clip CTAs): overlap-add always sums frames in ascending order."""
    import torch
    n, sr = 100000, 48000
    clip = synth.bass_clip(77, n, sr)
    y1, _ = qd.process_batch(torch.from_numpy(clip[None, :]).cuda(), sr, **SB)
    big = torch.from_numpy(np.repeat(clip[None, :], 700, axis=0)).cuda()
    y700, _ = qd.process_batch(big, sr, **SB)
    assert torch.equal(y700[0], y1[0]) and torch.equal(y700[699], y1[0]) and torch.equal(y700[350], y1[0])


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,prec,copies", [(512, "float32", 1200), (1024, "float32", 1200), (4096, "float32", 400),
                                               (4096, "float64", 400), (8192, "auto", 350), (8192, "float32", 350)])
def test_team_kernel_is_deterministic_across_tilings_and_runs(qd, n_fft, prec, copies):
    """The team kernel (qd_spec_team.cuh: several warps per frame, named barriers, per-warp gather lists): the same clip
    alone (cut into time tiles), inside a batch that fills the GPU with whole-clip CTAs, and rendered three times over --
    bit for bit the same, and within the north-star tolerance of the oracle.  A missing barrier shows up here as a
    run-to-run difference (compute-sanitizer is not available on this pool)."""
    import torch
    n, sr = 60000, 48000
    clip = synth.bass_clip(78, n, sr)
    kw = dict(SB, n_fft=n_fft, precision=prec)
    y1, _ = qd.process_batch(torch.from_numpy(clip[None, :]).cuda(), sr, **kw)
    big = torch.from_numpy(np.repeat(clip[None, :], copies, axis=0)).cuda()
    runs = [qd.process_batch(big, sr, **kw)[0] for _ in range(3)]
    for y in runs:
        assert torch.equal(y[0], y1[0]) and torch.equal(y[copies - 1], y1[0]) and torch.equal(y[copies // 2], y1[0])
        assert torch.equal(y, runs[0])
    ref, _ = orc.process_audio(clip, sr, n_fft=n_fft)
    got = y1[0].cpu().numpy()
    # float32 at n_fft 8192 is the one configuration known to leave the 1e-4 bound (SURVEY 7.4: up to 3e-4 on noise), which
    # is why precision="auto" never picks it; forced float32 is held to 5e-4 / -60 dBFS here
    forced_f32 = n_fft == 8192 and prec == "float32"
    assert float(np.max(np.abs(got.astype(np.float64) - ref))) <= (5e-4 if forced_f32 else 1e-4)
    assert orc.null_test_db(got, ref) <= (-60.0 if forced_f32 else -80.0)


@pytest.mark.gpu
def test_full_size_properties(qd):
    """BASELINE config #2 clip length (480 000 samples): passthrough null, limiter ceiling, determinism."""
    import torch
    n, sr, b = 480000, 48000, 24
    x = synth.bass_batch_torch(b, n, sr, "cuda", seed=5)
    y, _ = qd.process_batch(x, sr, passthrough_test=True, **SB)
    d = (y - x).double()
    null = 20.0 * torch.log10(torch.sqrt((d * d).mean()).clamp_min(1e-10)).item()
    assert null < -110.0, null  # reference test bar is -80 dB (tests/test_passthrough_null.py:56-148)
    loud = (x * 3.0).clamp(-1.5, 1.5)
    kw = dict(distortion_params={"fold_amount": 3.0})
    y, _ = qd.process_batch(loud, sr, **SB, **kw)
    ceiling = 10.0 ** (-1.0 / 20.0)
    assert float(y.abs().max()) <= ceiling * 1.01  # reference tests/test_limiter.py:7-58 bound
    assert torch.isfinite(y).all()
    y_again, _ = qd.process_batch(loud, sr, **SB, **kw)
    assert torch.equal(y, y_again)
    # one clip of the batch against the oracle at full length
    ref, _ = orc.process_audio(loud[3].cpu().numpy(), sr, **kw)
    _check(y[3].cpu().numpy(), ref, "full-size clip")


@pytest.mark.gpu
def test_stage_limiter_and_crossover_and_distortion(qd):
    st = np.load(os.path.join(G, "stages.npz"))
    x = st["td/x"]
    for sr in (48000, 44100):
        y = qd.peak_limiter(x, sr, ceiling_db=-1.0, lookahead_ms=5.0, release_ms=30.0)
        assert np.max(np.abs(y.astype(np.float64) - st[f"td/lim/{sr}/y"])) <= 6e-8
    lo, hi = qd.linkwitz_riley_split(x, 48000, 300.0)
    assert np.max(np.abs(lo - st["td/xo/low"])) <= 1.2e-7 and np.max(np.abs(hi - st["td/xo/high"])) <= 1.2e-7
    wf = qd.apply_distortion(x, "wavefold", fold_amount=5.0, bias=0.1)
    assert np.max(np.abs(wf - st["td/wavefold"])) <= 2e-6
    tb = qd.apply_distortion(x, "tube", drive=4.0, warmth=0.7)
    assert np.max(np.abs(tb - st["td/tube"])) <= 1e-6
    with pytest.raises(ValueError):
        qd.apply_distortion(x, "fuzz")
    # long clip: chunk carries of both scans
    xl = np.clip(2.0 * synth.noise_clip(9, 200001), -2, 2).astype(np.float32)
    ref, _ = orc.peak_limiter(xl, 48000, -1.0, 5.0, 30.0)
    assert np.max(np.abs(qd.peak_limiter(xl, 48000, -1.0, 5.0, 30.0).astype(np.float64) - ref)) <= 6e-8
    rlo, rhi = orc.linkwitz_riley_split(xl, 48000, 300.0)
    lo, hi = qd.linkwitz_riley_split(xl, 48000, 300.0)
    assert np.max(np.abs(lo - rlo)) <= 2.4e-7 and np.max(np.abs(hi - rhi)) <= 2.4e-7


@pytest.mark.gpu
def test_edge_cases(qd):
    y, taps = qd.process_audio(np.zeros(0, dtype=np.float32), 48000, **SB)
    assert y.shape == (0,) and set(taps) == {"input", "pre_quant", "post_dist", "output"}
    # n = 1 is an impulse: every bin has |X| = 1 with alternating sign, the per-target phasor sums cancel to
    # rounding noise and the reference's own phase there is arbitrary -- only shape/finiteness is checked.
    y, _ = qd.process_audio(np.array([0.4], dtype=np.float32), 48000, **SB)
    assert y.shape == (1,) and np.isfinite(y).all()
    for n in (5, 511, 512, 513, 2047):
        x = synth.noise_clip(n, n)
        y, _ = qd.process_audio(x, 48000, **SB)
        ref, _ = orc.process_audio(x, 48000)
        _check(y, ref, f"n={n}")
    silent = np.zeros(4096, dtype=np.float32)
    y, _ = qd.process_audio(silent, 48000, **SB)
    assert np.array_equal(y, silent)
    stereo = np.stack([synth.bass_clip(1, 3000), synth.noise_clip(2, 3000)], axis=1)
    y, _ = qd.process_audio(stereo, 48000, **SB)
    ref, _ = orc.process_audio(stereo, 48000)
    _check(y, ref, "stereo->mono")


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft", [512, 1024, 4096, 8192])
def test_edge_cases_other_frame_sizes(qd, n_fft):
    """Ragged and tiny clips through the team kernel (n_fft != 2048): shorter than a hop, shorter than a frame, odd lengths
    (scalar load / store paths, no bulk-copy staging), a length that is a multiple of 4 but not of the hop, multiband, and a
    batch of unequal content -- each against the oracle."""
    sr = 48000
    # a single sample is a centred impulse: every bin has the same magnitude and alternating sign, the quantizer's phasor
    # sums cancel exactly and the reference's output phase is decided by rounding noise -- compared without the quantizer
    x1 = np.array([0.37], dtype=np.float32)
    y, _ = qd.process_audio(x1, sr, n_fft=n_fft, passthrough_test=True, **SB)
    _check(y, orc.process_audio(x1, sr, n_fft=n_fft, passthrough_test=True)[0], f"n_fft {n_fft} n 1 passthrough")
    for n in (2, 7, n_fft // 4 - 1, n_fft - 1, n_fft + 3, 3 * n_fft + 5, 20000, 20001):
        x = synth.noise_clip(300 + n % 97, n)
        y, taps = qd.process_audio(x, sr, n_fft=n_fft, **SB)
        ref, rt = orc.process_audio(x, sr, n_fft=n_fft)
        _check(y, ref, f"n_fft {n_fft} n {n}")
        _check(taps["pre_quant"], rt["pre_quant"], f"n_fft {n_fft} n {n} pre_quant")
    n = 6 * n_fft + 2
    xb = np.stack([synth.bass_clip(1, n, sr), np.zeros(n, dtype=np.float32), synth.noise_clip(3, n)])
    kw = dict(use_multiband=True, crossover_hz=250.0, distortion_mode="tube", dry_wet=0.8)
    yb, _ = qd.process_batch(xb, sr, n_fft=n_fft, **SB, **kw)
    for i in range(3):
        ref, _ = orc.process_audio(xb[i], sr, n_fft=n_fft, **kw)
        _check(yb[i], ref, f"n_fft {n_fft} multiband clip {i}")


@pytest.mark.gpu
def test_spectral_fx_batch_shared_and_per_clip_seeds(qd):
    """BASELINE config #4 shape: Growl preset + multiband + each FX; shared-seed batch and per-clip seeds."""
    n, sr = 20000, 48000
    x = np.stack([synth.loud_clip(60 + i, n, sr) for i in range(3)])
    base = dict(qd_cases.GROWL, use_multiband=True)
    for mode, s in (("bitcrush", 0.5), ("phase_dispersal", 0.6), ("bin_scramble", 0.55), ("bin_scramble", 0.3)):
        kw = dict(base, spectral_fx_mode=mode, spectral_fx_strength=s)
        y, _ = qd.process_batch(x, sr, seeds=1234, **kw)            # np.random.seed(1234) before every clip
        ys, _ = qd.process_batch(x, sr, seeds=[5, 6, 7], **kw)      # one seed per clip
        for i in range(3):
            np.random.seed(1234)
            ref, _ = orc.process_audio(x[i], sr, **kw)
            _check(y[i], ref, f"{mode} {s} shared clip {i}")
            np.random.seed(5 + i)
            ref, _ = orc.process_audio(x[i], sr, **kw)
            _check(ys[i], ref, f"{mode} {s} per-clip clip {i}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["sb_default_noise", "sb_growl", "mb_growl_bitcrush", "mb_growl_scramble_pick",
                                  "nfft512", "nfft4096", "sb_ragged_len"])
def test_float64_kernels_vs_reference_fixtures(qd, pipe, name):
    """The float64 instantiation of the spectral pass: reference parity to float32 rounding of the output."""
    kind, seed, n, sr, n_fft, rng_seed, kw = qd_cases.CASES[name]
    if rng_seed is not None:
        np.random.seed(rng_seed)
    x = pipe.input(name, qd_cases.make_signal(kind, seed, n, sr))
    y, taps = qd.process_audio(x, sr, n_fft=n_fft, precision="float64", **SB, **kw)
    _check(*pipe.at(f"{name}/y", y), f"{name}/y f64", 2e-6)
    _check(*pipe.at(f"{name}/pre_quant", taps["pre_quant"]), f"{name}/pre_quant f64", 2e-6)


def test_auto_precision_rule():
    from quantumdistortion_b200.pipeline import _resolve_kwargs
    assert _resolve_kwargs(1000, 48000, 2048, dict(SB))[0].params.precision == 0
    assert _resolve_kwargs(1000, 48000, 8192, dict(SB))[0].params.precision == 1
    assert _resolve_kwargs(1000, 48000, 2048, dict(SB, sub_cut_hz=0.0, air_cut_hz=0.0))[0].params.precision == 1
    assert _resolve_kwargs(1000, 48000, 2048, dict(SB, precision="float64"))[0].params.precision == 1
    assert _resolve_kwargs(1000, 48000, 2048, dict(SB, spectral_freeze=True))[0].params.precision == 1
    assert _resolve_kwargs(1000, 48000, 2048, dict(SB, spectral_freeze=True, precision="float32"))[0].params.precision == 0


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(qd_cases.UI_CASES))
def test_ui_config_dict_vs_reference_fixtures(qd, name):
    """Streamlit V2 nested config dict (dsp/pipeline.py:923-1008) through process_audio(config=...)."""
    g = qd_cases.Golden("frontend")
    kind, seed, n, sr, rng_seed, cfg, kw = qd_cases.UI_CASES[name]
    x = g.input(name, qd_cases.make_signal(kind, seed, n, sr))
    np.random.seed(rng_seed)
    y, _ = qd.process_audio(x, sr, config=cfg, **SB, **kw)
    _check(*g.at(f"{name}/y", y), name)


@pytest.mark.gpu
def test_file_harness_single_and_batched(qd, tmp_path):
    """process_file_to_file / process_files (dsp/harness.py:24-63): WAV in -> GPU render -> PCM16 WAV out."""
    from quantumdistortion_b200.audio_io import float_to_pcm16, load_audio, save_audio
    sr = 44100
    ins, outs = [], []
    for i in range(3):
        p = tmp_path / f"in{i}.wav"
        save_audio(p, synth.bass_clip(80 + i, 22050 if i < 2 else 11025, sr), sr)
        ins.append(p)
        outs.append(tmp_path / "out" / f"o{i}.wav")
    qd.process_file_to_file(ins[0], outs[0], preset="Perc To Tonal Clang", extra_params=dict(SB, dry_wet=0.8))
    assert qd.process_files(list(zip(ins, outs))[1:], preset="Perc To Tonal Clang", extra_params=dict(SB, dry_wet=0.8)) == 2
    from quantumdistortion_b200 import PipelineConfig
    for i in range(3):
        x, _ = load_audio(ins[i])
        pc = PipelineConfig.from_preset("Perc To Tonal Clang")
        kw = dict(key=pc.key, scale=pc.scale, snap_strength=pc.snap_strength, smear=pc.smear,
                  distortion_mode=pc.distortion_mode, distortion_params=pc.distortion_params,
                  limiter_ceiling_db=pc.limiter_ceiling_db, dry_wet=0.8)
        ref, _ = orc.process_audio(x, sr, **kw)
        got, sr2 = load_audio(outs[i])
        assert sr2 == sr
        lsb = np.abs(np.rint(got * 32768.0) - float_to_pcm16(ref).astype(np.float64))
        assert lsb.max() <= 4, lsb.max()   # 1e-4 parity bound = 3.3 LSB of 16-bit PCM


@pytest.mark.gpu
def test_host_pipeline_odd_batch_small_chunks(qd):
    """qd_render_host with a batch that is not a multiple of the chunk, chunks of 1 / 2 / > batch clips, multiband
    with a per-clip FX table (clip offsets inside the table follow the chunks)."""
    import torch
    n, sr = 9000, 48000
    x = np.stack([synth.loud_clip(90 + i, n, sr) for i in range(5)])
    kw = dict(qd_cases.GROWL, use_multiband=True, spectral_fx_mode="bin_scramble", spectral_fx_strength=0.55)
    ref, _ = qd.process_batch(torch.from_numpy(x).cuda(), sr, seeds=[1, 2, 3, 4, 5], **kw)
    ref = ref.cpu().numpy()
    for chunk in (1, 2, 64):
        y, _ = qd.process_batch(x, sr, seeds=[1, 2, 3, 4, 5], chunk_clips=chunk, **kw)
        assert np.array_equal(y, ref), chunk
    np.random.seed(3)
    o, _ = orc.process_audio(x[2], sr, **kw)
    _check(ref[2], o, "per-clip seeded scramble, clip 2")


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(qd_cases.ANALYSIS_CASES))
def test_cents_metric_vs_reference_fixtures(qd, name):
    """avg_cents_offset_from_scale (dsp/analyses.py:53-142): the peak bins come from the CUDA STFT (float64 kernels
    by default), the cents from the host table -> the reference's per-peak values bit for bit."""
    from quantumdistortion_b200 import analyses
    g = qd_cases.Golden("analysis")
    kind, seed, n, sr, key, scale, kw = qd_cases.ANALYSIS_CASES[name]
    x = g.input(name, qd_cases.make_signal(kind, seed, n, sr))
    avg, per = analyses.avg_cents_offset_from_scale(x, sr, key, scale, **kw)
    assert np.array_equal(per, g[f"{name}/per_peak"]), name
    assert avg == float(g[f"{name}/avg"])
    # peak bins vs the oracle, float64 exactly and float32 on all but near-tied bins
    _, _, ref_bins = orc.avg_cents_offset_from_scale(x, sr, key, scale, return_bins=True, **kw)
    nf, topn = kw.get("frame_length", 2048), kw.get("topn_peaks", 3)
    b64 = analyses.spectral_peak_bins(x[None, :], n_fft=nf, topn=topn, min_db=kw.get("min_db", -60.0))
    assert np.array_equal(b64[0], ref_bins)
    b32 = analyses.spectral_peak_bins(x[None, :], n_fft=nf, topn=topn, min_db=kw.get("min_db", -60.0), precision="float32")
    assert np.mean(b32[0] == ref_bins) >= 0.98
    avg32, _ = analyses.avg_cents_offset_from_scale(x, sr, key, scale, precision="float32", **kw)
    assert abs(avg32 - avg) <= 0.02 * avg


@pytest.mark.gpu
def test_cents_metric_batch_of_renders(qd):
    """The metric's purpose (scripts/validate_dsp_metrics.py:59-105): rendering with the scale-snap quantizer moves the
    strongest bins towards the scale.  Batch API, every clip against the oracle."""
    from quantumdistortion_b200 import analyses
    n, sr = 24000, 48000
    x = np.stack([synth.bass_clip(70 + i, n, sr) for i in range(4)])
    y, _ = qd.process_batch(x, sr, limiter_on=False, **SB)
    for sig in (x, y):
        avgs, per = analyses.avg_cents_offset_batch(sig, sr, "D", "minor")
        for i in range(len(sig)):
            a, p = orc.avg_cents_offset_from_scale(sig[i], sr, "D", "minor")
            assert np.array_equal(per[i], p) and avgs[i] == a
    wet, _ = analyses.avg_cents_offset_batch(y, sr, "D", "minor")
    dry, _ = analyses.avg_cents_offset_batch(x, sr, "D", "minor")
    assert np.mean(wet) < np.mean(dry)
    silent, per0 = analyses.avg_cents_offset_from_scale(np.zeros(5000, dtype=np.float32), sr, "D", "minor")
    assert np.isnan(silent) and per0.size == 0


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["sb_formant_up", "mb_formant_bitcrush", "nfft1024_formant"])
def test_formant_shift_float64_kernels(qd, pipe, name):
    """precision="float64": the cepstral FFTs of the formant shift run in float64 like the rest of the pass."""
    kind, seed, n, sr, n_fft, rng_seed, kw = qd_cases.CASES[name]
    x = pipe.input(name, qd_cases.make_signal(kind, seed, n, sr))
    if rng_seed is not None:
        np.random.seed(rng_seed)
    y, _ = qd.process_audio(x, sr, n_fft=n_fft, precision="float64", **SB, **kw)
    _check(*pipe.at(f"{name}/y", y), f"{name}/y float64", 5e-6)


@pytest.mark.gpu
def test_random_configs_vs_oracle(qd):
    """Keys, scales, snap / smear, band edges, distortion and mix settings drawn at random (seeded) on the STFT path,
    precision="auto", every render against the oracle at the north-star tolerance."""
    rng = np.random.default_rng(77)
    keys = ["C", "C#", "D", "Eb", "E", "F", "F#", "G", "Ab", "A", "Bb", "B"]
    scales = ["major", "minor", "pentatonic", "dorian", "mixolydian", "harmonic_minor"]
    n, sr = 12000, 48000
    worst = 0.0
    for i in range(12):
        kw = dict(key=keys[rng.integers(12)], scale=scales[rng.integers(6)], snap_strength=float(rng.uniform(0.2, 1.0)),
                  smear=float(rng.uniform(0.0, 0.6)), bin_smoothing=bool(rng.integers(2)),
                  sub_cut_hz=float(rng.choice([60.0, 110.0, 200.0])), air_cut_hz=float(rng.choice([3000.0, 5000.0, 8000.0])),
                  distortion_mode=str(rng.choice(["wavefold", "tube"])),
                  distortion_params={"fold_amount": float(rng.uniform(1.0, 4.0)), "bias": float(rng.uniform(-0.1, 0.1)),
                                     "drive": float(rng.uniform(0.5, 3.0)), "warmth": float(rng.uniform(0.0, 1.0))},
                  limiter_ceiling_db=float(rng.choice([-0.5, -1.0, -3.0])), dry_wet=float(rng.uniform(0.4, 1.0)),
                  use_multiband=bool(rng.integers(2)), crossover_hz=float(rng.choice([200.0, 300.0, 500.0])),
                  lowband_drive=float(rng.uniform(0.5, 2.0)), harmonic_lock_hz=float(rng.choice([0.0, 0.0, 55.0])))
        x = qd_cases.make_signal(["bass", "loud", "noise"][i % 3], 300 + i, n, sr)
        y, taps = qd.process_audio(x, sr, **SB, **kw)
        ref, rt = orc.process_audio(x, sr, **kw)
        worst = max(worst, _check(y, ref, f"case {i} {kw}"))
        _check(taps["pre_quant"], rt["pre_quant"], f"case {i} pre_quant")
    print(f"worst error over the random STFT-path configs: {worst:.3e}")
