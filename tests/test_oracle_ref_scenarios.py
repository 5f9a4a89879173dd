"""CPU: the oracle on the reference's own pipeline-level test scenarios (qd_cases.REF_SCENARIOS; fixtures
tests/golden/scenarios.npz from the LIVE reference, generator tests/golden/make_golden.py scenarios).

The signals and keyword arguments are the ones the reference's test suite passes to process_audio
(tests/test_pipeline.py, test_passthrough_null.py, test_multiband_alignment.py, test_pipeline_multiband_identity.py,
test_m12_quantum_fx.py, test_quantization_integration.py); quantize_mode stays at the reference default wherever
the reference test leaves it there, so these cases also pin the mode-resolution rules of dsp/pipeline.py:1315-1327.
"""

import numpy as np
import pytest

import qd_cases
from oracle import qd_autotune as at
from oracle import qd_oracle as orc

_AT_DROP = ("smear", "bin_smoothing", "post_quant", "use_multiband", "crossover_hz", "lowband_drive", "quantize_mode",
            # options the reference test passes at their "off" value: they do not leave autotune_v1 (:1315-1324)
            "spectral_fx_mode", "spectral_fx_strength", "spectral_freeze", "formant_shift", "harmonic_lock_hz")


@pytest.fixture(scope="module")
def sc():
    return qd_cases.Golden("scenarios")


def oracle_render(x, sr, kw):
    """The two oracles behind the reference's dispatch: qd_oracle.process_audio resolves the mode like
    dsp/pipeline.py:1315-1327 (FX / freeze / formant / lock options and passthrough_test run the STFT path, autotune_v1
    with snap_strength > 0 drops multiband) and refuses a render that stays in the time-domain autotune_v1 chain,
    which is oracle/qd_autotune.py."""
    kw = dict(kw)
    mode = kw.pop("quantize_mode", "autotune_v1")
    try:
        return orc.process_audio(x, sr, quantize_mode=mode, **{k: v for k, v in kw.items() if k != "sub_enabled"})
    except NotImplementedError:
        return at.process_audio_autotune(x, sr, **{k: v for k, v in kw.items() if k not in _AT_DROP})


@pytest.mark.parametrize("name", list(qd_cases.REF_SCENARIOS))
def test_oracle_on_reference_test_scenarios(sc, name):
    spec, sr, rng_seed, kw, prop, cite = qd_cases.REF_SCENARIOS[name]
    x = qd_cases.scenario_signal(spec, sr)
    assert sc.matches(f"{name}/x", x), "scenario signal drifted from the fixture"
    if rng_seed is not None:
        np.random.seed(rng_seed)
    y, taps = oracle_render(x, sr, kw)
    for got, key in ((y, "y"), (taps["pre_quant"], "pre_quant"), (taps["post_dist"], "post_dist")):
        got = np.asarray(got, dtype=np.float32)
        assert got.shape == sc.shape(f"{name}/{key}"), f"{name}/{key} ({cite})"
        err = sc.max_abs_err(f"{name}/{key}", got)
        assert err <= 2e-7, f"{name}/{key} ({cite}): max abs err {err:.3e}"


def test_reference_assertions_hold_on_the_fixtures(sc):
    """What the reference's tests assert holds on the reference's renders (a guard for the generator).  The fixtures keep
    a sample of each render, so the assertions run on the oracle's renders, checked against those samples first."""
    ys = {}
    for name, (spec, sr, rng_seed, kw, _prop, _cite) in qd_cases.REF_SCENARIOS.items():
        if rng_seed is not None:
            np.random.seed(rng_seed)
        ys[name] = np.asarray(oracle_render(qd_cases.scenario_signal(spec, sr), sr, kw)[0], dtype=np.float32)
        assert sc.max_abs_err(f"{name}/y", ys[name]) <= 2e-7, name
    for name, (spec, sr, *_rest) in qd_cases.REF_SCENARIOS.items():
        qd_cases.check_scenario_property(name, qd_cases.scenario_signal(spec, sr), ys[name], ys.get)


def test_reference_formant_second_pass_is_ill_conditioned(sc):
    """Why formant_six carries a wider tolerance on its final output (qd_cases.REF_SCENARIO_Y_TOL): the reference's
    second quantised pass amplifies a 1e-9 change of its input -- far below the float32 resolution of that input -- by
    five orders of magnitude.  The oracle reproduces the reference bit for bit on this case (test above), so its
    sensitivity is the reference's."""
    name, sr = "formant_six", 44100
    x = sc[f"{name}/post_dist"]

    def second_pass(sig):
        S, freqs = orc.stft(sig, sr, 2048)
        Sq = orc.spectral_quantize_stft(S, freqs, "D", "minor", 1.0, 0.1, True, formant_shift=6.0)
        return orc.istft(Sq, sr, 2048, length=len(sig)).astype(np.float32)

    y0 = second_pass(x)
    assert sc.matches(f"{name}/y", y0)   # limiter idle (peak 0.07): the pass output is the render
    rng = np.random.default_rng(0)
    y1 = second_pass(x.astype(np.float64) + 1e-9 * rng.standard_normal(len(x)))
    assert float(np.max(np.abs(y1 - y0))) > 1e-4


def test_reference_freeze_needs_a_float64_fft(sc):
    """Why precision="auto" renders spectral_freeze in float64 (tables.choose_precision): spectral noise at the float32
    FFT's level (1e-7 of the frame's strongest bin) moves the reference's frozen pass by more than the 1e-4 bound on the
    reference's own test signal, noise at the float64 level does not."""
    name, sr = "freeze_multiband", 44100
    _, high = orc.linkwitz_riley_split(qd_cases.scenario_signal(qd_cases.REF_SCENARIOS[name][0], sr), sr, 300.0)
    S, freqs = orc.stft(high.astype(np.float32), sr, 2048)

    def frozen_pass(Sx):
        Sq = orc.spectral_quantize_stft(Sx, freqs, "D", "minor", 1.0, 0.1, True, is_high_band=True, spectral_freeze=True)
        return orc.istft(Sq, sr, 2048, length=high.shape[0]).astype(np.float32)

    y0 = frozen_pass(S)
    rng = np.random.default_rng(1)
    peak = np.abs(S).max(axis=0, keepdims=True)
    unit = rng.standard_normal(S.shape) + 1j * rng.standard_normal(S.shape)
    assert float(np.max(np.abs(frozen_pass(S + 1e-7 * peak * unit) - y0))) > 1e-4
    assert float(np.max(np.abs(frozen_pass(S + 1e-15 * peak * unit) - y0))) < 1e-6


# ---------------------------------------------------------------- the reference's scripts (tests/golden/scripts.npz)
@pytest.fixture(scope="module")
def scr():
    return qd_cases.Golden("scripts")


def _wav_slice(name, seconds):
    d = qd_cases.Golden("refwav")
    sr = int(d[f"{name}/sr"])
    return d[f"{name}/x16"][: int(sr * seconds)], sr


@pytest.mark.parametrize("name", list(qd_cases.SCRIPT_SCENARIOS))
def test_oracle_on_reference_script_calls(scr, name):
    wav, seconds, rng_seed, _kw, cite = qd_cases.SCRIPT_SCENARIOS[name]
    x16, sr = _wav_slice(wav, seconds)
    x = x16.astype(np.float32) / 32768.0
    if rng_seed is not None:
        np.random.seed(rng_seed)
    y, taps = oracle_render(x, sr, qd_cases.script_scenario_kwargs(name))
    for got, key in ((y, "y"), (taps["pre_quant"], "pre_quant"), (taps["post_dist"], "post_dist")):
        err = scr.max_abs_err(f"{name}/{key}", np.asarray(got, dtype=np.float64))
        assert err <= 2e-7, f"{name}/{key} ({cite}): max abs err {err:.3e}"


@pytest.mark.parametrize("name", list(qd_cases.HARNESS_SCENARIOS))
def test_oracle_on_reference_harness_renders(scr, name):
    """process_file_to_file (dsp/harness.py:23-67): PipelineConfig() or from_preset(), extra_params override the fields
    they name, the render goes out as 16-bit PCM."""
    from quantumdistortion_b200.presets import get_preset
    wav, seconds, rng_seed, preset, _ep, cite = qd_cases.HARNESS_SCENARIOS[name]
    x16, sr = _wav_slice(wav, seconds)
    x = x16.astype(np.float32) / 32768.0
    kw = {}
    if preset is not None:
        p = get_preset(preset)
        kw = {k: p[k] for k in qd_cases._PRESET_ARGS}
    kw.update(qd_cases.harness_extra_params(name))
    if rng_seed is not None:
        np.random.seed(rng_seed)
    y, _ = oracle_render(x, sr, kw)
    pcm, ref = scr.at(f"{name}/y16", np.clip(np.rint(y.astype(np.float64) * 32767.0), -32768, 32767).astype(np.int32))
    d = int(np.max(np.abs(pcm - ref.astype(np.int32))))
    assert d <= 1, f"{name} ({cite}): {d} PCM16 steps"
