"""GPU (B200): quantize_mode="autotune_v1" through the C ABI vs the live-reference fixtures (tests/golden/autotune.npz)
and the oracle (oracle/qd_autotune.py).  Same bar as the STFT path: max abs error <= 1e-4, null <= -80 dBFS."""

import numpy as np
import pytest

import qd_cases
from oracle import qd_autotune as at
from oracle import qd_oracle as orc

MAX_ABS = 1e-4
NULL_DB = -80.0


@pytest.fixture(scope="module")
def qd():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import quantumdistortion_b200 as q
    return q


@pytest.fixture(scope="module")
def gold():
    return qd_cases.Golden("autotune")


def _check(got, ref, what, max_abs=MAX_ABS):
    got = np.asarray(got)
    assert got.shape == ref.shape, what
    err = float(np.max(np.abs(got.astype(np.float64) - ref))) if ref.size else 0.0
    null = orc.null_test_db(got, ref) if ref.size else -200.0
    assert err <= max_abs, f"{what}: max abs err {err:.3e}"
    assert null <= NULL_DB, f"{what}: null {null:.1f} dB"
    return err


@pytest.mark.gpu
def test_autotune_stages_vs_reference(qd, gold):
    """Parity ladder: every intermediate of dsp/autotune.py:426-437 on one clip."""
    import torch
    from quantumdistortion_b200 import make_renderer
    x = gold["st/x"]
    r = make_renderer(len(x), 48000, quantize_mode="autotune_v1", limiter_on=False,
                      distortion_params={"fold_amount": 1.0})
    y, taps, dbg = r.render_device(torch.from_numpy(x[None, :]).cuda(), want_taps=True, debug=True)
    d = {k: v[0].cpu().numpy() for k, v in dbg.items()}
    for k in ("sub", "body", "air", "det"):          # float64 IIR sweeps in the reference's operation order
        assert gold.max_abs_err(f"st/{k}", d[k]) <= 2e-7, k
    f, gf = d["features"], gold["st/features"]
    assert f.shape == gf.shape
    assert np.allclose(f[:, 0], gf[:, 0], rtol=1e-5, atol=1e-8)            # rms (float32 mean)
    # flatness is only compared with 0.55 (dsp/autotune.py:234); the float32 FFT floor shows on very tonal frames
    # (reference 4e-6, here 9e-6), frames near the threshold agree to 1e-6
    assert np.allclose(f[:, 1], gf[:, 1], rtol=1e-4, atol=1e-4)
    voiced = gf[:, 2] > 0
    assert np.array_equal(f[:, 2] > 0, voiced)
    assert np.allclose(f[voiced, 2], gf[voiced, 2], rtol=1e-7, atol=0.0)   # YIN pitch (float64)
    assert np.allclose(f[:, 3], gf[:, 3], rtol=0.0, atol=1e-7)
    assert np.max(np.abs(d["ratio_track"].astype(np.float64) - gold["st/ratio_track"])) <= 1e-6
    _check(*gold.at("st/corrected", d["corrected"]), "corrected body", 2e-5)
    _check(*gold.at("st/sub_layer", d["sub_layer"]), "sub layer", 2e-6)
    _check(*gold.at("st/output", taps["pre_quant"][0].cpu().numpy()), "autotune output", 2e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(qd_cases.AUTOTUNE_CASES))
def test_autotune_pipeline_vs_reference_fixtures(qd, gold, name):
    kind, seed, n, sr, kw = qd_cases.AUTOTUNE_CASES[name]
    x = gold.input(name, qd_cases.make_signal(kind, seed, n, sr))
    y, taps = qd.process_audio(x, sr, quantize_mode="autotune_v1", **kw)
    _check(*gold.at(f"{name}/y", y), f"{name}/y")
    _check(*gold.at(f"{name}/pre_quant", taps["pre_quant"]), f"{name}/pre_quant")
    _check(*gold.at(f"{name}/post_dist", taps["post_dist"]), f"{name}/post_dist")
    assert np.array_equal(taps["input"], x) and np.array_equal(taps["output"], y)


@pytest.mark.gpu
def test_autotune_batch_vs_oracle(qd):
    """A batch through process_batch (device and host containers, chunked), every clip against the oracle."""
    n, sr = 12000, 48000
    x = np.stack([qd_cases.make_signal("tone" if i % 2 == 0 else "bass", 20 + i, n, sr) for i in range(5)])
    y, taps = qd.process_batch(x, sr, quantize_mode="autotune_v1", return_taps=True, key="E", scale="dorian")
    for i in range(len(x)):
        ref, rt = at.process_audio_autotune(x[i], sr, key="E", scale="dorian")
        _check(y[i], ref, f"clip {i}")
        _check(taps["pre_quant"][i], rt["pre_quant"], f"clip {i} pre_quant")
    y2, _ = qd.process_batch(x, sr, quantize_mode="autotune_v1", key="E", scale="dorian", chunk_clips=2)
    assert np.array_equal(y, y2)
    with pytest.raises(ValueError):
        qd.process_audio(np.zeros(10, dtype=np.float32), sr, quantize_mode="autotune_v1")


@pytest.mark.gpu
@pytest.mark.parametrize("n", [16, 17, 100, 513, 2049, 4097])
def test_autotune_tiny_and_silent_clips(qd, n):
    """Lengths around the padding (15), one hop, half a frame and one frame; silence; stereo input."""
    sr = 48000
    x = qd_cases.make_signal("tone", 30 + n, max(n, 64), sr)[:n]
    y, taps = qd.process_audio(x, sr, quantize_mode="autotune_v1")
    ref, rt = at.process_audio_autotune(x, sr)
    _check(y, ref, f"n={n}")
    _check(taps["pre_quant"], rt["pre_quant"], f"n={n} pre_quant")
    z = np.zeros(n, dtype=np.float32)
    yz, _ = qd.process_audio(z, sr, quantize_mode="autotune_v1")
    refz, _ = at.process_audio_autotune(z, sr)
    assert np.array_equal(yz, refz)
    st = np.stack([x, 0.5 * x], axis=1)
    ys, _ = qd.process_audio(st, sr, quantize_mode="autotune_v1")
    refs, _ = at.process_audio_autotune(st, sr)
    _check(ys, refs, f"stereo n={n}")


@pytest.mark.gpu
def test_autotune_full_length_clip_vs_oracle(qd):
    """BASELINE clip length (10 s @ 48 kHz): the shifter integrates 1 - ratio over 480 000 samples, so this is where a
    pitch-track mismatch would show as drift.  One pitched clip, whole render, against the oracle."""
    n, sr = 480000, 48000
    x = qd_cases.make_signal("tone", 77, n, sr)
    y, taps = qd.process_audio(x, sr, quantize_mode="autotune_v1")
    ref, rt = at.process_audio_autotune(x, sr)
    err = _check(taps["pre_quant"], rt["pre_quant"], "10 s pre_quant")
    _check(y, ref, "10 s output")
    print(f"10 s autotune clip: max abs err {err:.3e}")


@pytest.mark.gpu
@pytest.mark.parametrize("sr,n", [(96000, 96000), (22050, 40000), (44100, 80000), (192000, 70000)])
def test_autotune_other_sample_rates_vs_oracle(qd, sr, n):
    """The detector's lag range follows the sample rate (max_tau = sr / 71.5 Hz, at most 2047): 308 lags at 22.05 kHz,
    1342 at 96 kHz and 2047 at 192 kHz, where a clip's lags are split over two, three or four CTAs of the difference-function
    kernel.  Clips longer than four envelope tiles (65 536 samples) also take the segment-parallel follower."""
    x = qd_cases.make_signal("tone", 5 + sr % 97, n, sr)
    y, taps = qd.process_audio(x, sr, quantize_mode="autotune_v1")
    ref, rt = at.process_audio_autotune(x, sr)
    _check(taps["pre_quant"], rt["pre_quant"], f"sr={sr} pre_quant")
    _check(y, ref, f"sr={sr} output")


@pytest.mark.gpu
def test_autotune_through_the_file_harness(qd, tmp_path):
    """process_file_to_file / process_files with quantize_mode="autotune_v1" -- what the reference's harness and
    render_preset.py run by default (dsp/harness.py:24-63, SURVEY.md appendix C.13)."""
    from quantumdistortion_b200.audio_io import float_to_pcm16, load_audio, save_audio
    sr = 48000
    ins, outs = [], []
    for i in range(3):
        p = tmp_path / f"in{i}.wav"
        save_audio(p, qd_cases.make_signal("tone", 40 + i, 12000, sr), sr)
        ins.append(p)
        outs.append(tmp_path / "out" / f"o{i}.wav")
    extra = {"quantize_mode": "autotune_v1", "sub_level": 0.2}
    qd.process_file_to_file(ins[0], outs[0], preset="Subtle Tube Glue", extra_params=extra)
    assert qd.process_files(list(zip(ins, outs))[1:], preset="Subtle Tube Glue", extra_params=extra) == 2
    from quantumdistortion_b200 import PipelineConfig
    pc = PipelineConfig.from_preset("Subtle Tube Glue")
    for i in range(3):
        x, _ = load_audio(ins[i])
        ref, _ = at.process_audio_autotune(x, sr, key=pc.key, scale=pc.scale, snap_strength=pc.snap_strength,
                                           pre_quant=pc.pre_quant, distortion_mode=pc.distortion_mode,
                                           distortion_params=pc.distortion_params, limiter_on=pc.limiter_on,
                                           limiter_ceiling_db=pc.limiter_ceiling_db, dry_wet=pc.dry_wet, sub_level=0.2)
        got, sr2 = load_audio(outs[i])
        assert sr2 == sr
        lsb = np.abs(np.rint(got * 32768.0) - float_to_pcm16(ref).astype(np.float64))
        assert lsb.max() <= 4, lsb.max()   # 1e-4 parity bound = 3.3 LSB of 16-bit PCM


@pytest.mark.gpu
def test_autotune_random_configs_vs_oracle(qd):
    """Keys, scales, strengths, band edges and sub settings drawn at random (seeded), 0.5 s clips, against the oracle:
    exercises the note-hold transitions (confirm / release / candidate reset) on more material than the fixtures."""
    rng = np.random.default_rng(2026)
    keys = ["C", "C#", "D", "Eb", "E", "F", "F#", "G", "Ab", "A", "Bb", "B"]
    scales = ["major", "minor", "pentatonic", "dorian", "mixolydian", "harmonic_minor"]
    n, sr = 24000, 48000
    worst = 0.0
    for i in range(8):
        kw = dict(key=keys[rng.integers(12)], scale=scales[rng.integers(6)], snap_strength=float(rng.uniform(0.3, 1.0)),
                  sub_cut_hz=float(rng.choice([0.0, 80.0, 110.0, 150.0])), air_cut_hz=float(rng.choice([4000.0, 5000.0, 9000.0])),
                  sub_level=float(rng.uniform(0.0, 0.6)), sub_octave=int(rng.integers(0, 4)), air_mix=float(rng.uniform(0.0, 1.0)),
                  limiter_on=bool(rng.integers(2)), dry_wet=float(rng.uniform(0.5, 1.0)))
        x = qd_cases.make_signal("tone" if i % 4 else "bass", 200 + i, n, sr)
        y, taps = qd.process_audio(x, sr, quantize_mode="autotune_v1", **kw)
        ref, rt = at.process_audio_autotune(x, sr, **kw)
        worst = max(worst, _check(taps["pre_quant"], rt["pre_quant"], f"case {i} {kw} pre_quant"))
        _check(y, ref, f"case {i} {kw}")
    print(f"worst autotune error over the random configs: {worst:.3e}")
