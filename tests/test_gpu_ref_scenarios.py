"""GPU (B200): the reference's own pipeline-level test scenarios through the drop-in ``process_audio``.

Every process_audio call of the reference's test suite (qd_cases.REF_SCENARIOS cites file:line) with the reference's
signals and keyword arguments; quantize_mode stays at the reference default wherever the reference test leaves it
there.  Each case is checked twice: against the LIVE reference's output and taps (tests/golden/scenarios.npz,
generator tests/golden/make_golden.py scenarios) at the north-star tolerance, and against the assertion the
reference's test makes (qd_cases.check_scenario_property), evaluated on OUR output.
"""

import numpy as np
import pytest

import qd_cases
from oracle import qd_oracle as orc

MAX_ABS = 1e-4
NULL_DB = -80.0


@pytest.fixture(scope="module")
def qd():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import quantumdistortion_b200 as q
    from quantumdistortion_b200 import _lib
    assert _lib.load().qd_device_count() >= 1, "libqd_b200.so sees no sm_100 device"
    return q


@pytest.fixture(scope="module")
def sc():
    return qd_cases.Golden("scenarios")


@pytest.fixture(scope="module")
def rendered(qd, sc):
    """Our output of every scenario (several reference assertions compare two renders)."""
    out = {}
    for name, (spec, sr, rng_seed, kw, prop, cite) in qd_cases.REF_SCENARIOS.items():
        if rng_seed is not None:
            np.random.seed(rng_seed)   # the random spectral FX replay the global np.random state like the reference
        out[name] = qd.process_audio(sc.input(name, qd_cases.scenario_signal(spec, sr)), sr=sr, **kw)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(qd_cases.REF_SCENARIOS))
def test_reference_test_scenarios(rendered, sc, name):
    spec, sr, rng_seed, kw, prop, cite = qd_cases.REF_SCENARIOS[name]
    x = sc.input(name, qd_cases.scenario_signal(spec, sr))
    y, taps = rendered[name]
    assert set(taps.keys()) == {"input", "pre_quant", "post_dist", "output"}, cite
    assert np.array_equal(taps["input"], x) and np.array_equal(taps["output"], y)
    for got, key in ((y, "y"), (taps["pre_quant"], "pre_quant"), (taps["post_dist"], "post_dist")):
        what = f"{name}/{key} ({cite})"
        assert got.dtype == np.float32 and got.shape == sc.shape(f"{name}/{key}") == x.shape, what
        got, ref = sc.at(f"{name}/{key}", got)
        err = float(np.max(np.abs(got.astype(np.float64) - ref)))
        if key == "y" and name in qd_cases.REF_SCENARIO_Y_TOL:   # the reference itself is ill-conditioned there
            assert err <= qd_cases.REF_SCENARIO_Y_TOL[name], f"{what}: max abs err {err:.3e}"
            continue
        assert err <= MAX_ABS, f"{what}: max abs err {err:.3e}"
        assert orc.null_test_db(got, ref) <= NULL_DB, what
    qd_cases.check_scenario_property(name, x, y, lambda other: rendered[other][0])


# ---------------------------------------------------------------- the reference's scripts (tests/golden/scripts.npz)
@pytest.fixture(scope="module")
def scr():
    return qd_cases.Golden("scripts")


def _wav_slice(name, seconds):
    d = qd_cases.Golden("refwav")
    sr = int(d[f"{name}/sr"])
    return d[f"{name}/x16"][: int(sr * seconds)], sr


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(qd_cases.SCRIPT_SCENARIOS))
def test_reference_script_calls(qd, scr, name):
    """The process_audio calls of scripts/validate_dsp_metrics.py, profile_pipeline.py and render_preset.py (keyword
    form, quantize_mode at its default) on the first second of the reference's own WAV files."""
    wav, seconds, rng_seed, _kw, cite = qd_cases.SCRIPT_SCENARIOS[name]
    x16, sr = _wav_slice(wav, seconds)
    x = x16.astype(np.float32) / 32768.0
    if rng_seed is not None:
        np.random.seed(rng_seed)
    y, taps = qd.process_audio(audio=x, sr=sr, **qd_cases.script_scenario_kwargs(name))
    for got, key in ((y, "y"), (taps["pre_quant"], "pre_quant"), (taps["post_dist"], "post_dist")):
        what = f"{name}/{key} ({cite})"
        assert got.dtype == np.float32 and got.shape == scr.shape(f"{name}/{key}"), what
        got, ref = scr.at(f"{name}/{key}", got)
        err = float(np.max(np.abs(got.astype(np.float64) - ref)))
        assert err <= MAX_ABS, f"{what}: max abs err {err:.3e}"
        assert orc.null_test_db(got, ref) <= NULL_DB, what


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(qd_cases.HARNESS_SCENARIOS))
def test_reference_harness_renders(qd, scr, name, tmp_path):
    """process_file_to_file as scripts/quick_regression_suite.py and tests/test_harness_smoke.py call it: WAV in, WAV
    out, against the PCM16 samples the reference's own harness wrote (1e-4 = 3.3 steps of 16-bit PCM)."""
    from scipy.io import wavfile
    wav, seconds, rng_seed, preset, _ep, cite = qd_cases.HARNESS_SCENARIOS[name]
    x16, sr = _wav_slice(wav, seconds)
    src, dst = tmp_path / f"{name}_in.wav", tmp_path / "processed" / f"{name}_out.wav"
    wavfile.write(str(src), sr, x16)
    if rng_seed is not None:
        np.random.seed(rng_seed)
    qd.process_file_to_file(src, dst, preset=preset, extra_params=qd_cases.harness_extra_params(name))
    sr2, y16 = wavfile.read(str(dst))
    assert sr2 == sr and y16.dtype == np.int16 and y16.shape == scr.shape(f"{name}/y16")
    y16, ref = scr.at(f"{name}/y16", y16)
    d = int(np.max(np.abs(y16.astype(np.int32) - ref.astype(np.int32))))
    assert d <= 4, f"{name} ({cite}): {d} PCM16 steps"
