"""CPU: the autotune_v1 oracle (oracle/qd_autotune.py) against outputs of the LIVE reference stored in
tests/golden/autotune.npz (tests/golden/make_golden.py autotune).  Bit-exact on every stage and on whole renders."""

import numpy as np
import pytest
import scipy.signal

import qd_cases
from oracle import qd_autotune as at


@pytest.fixture(scope="module")
def gold():
    return qd_cases.Golden("autotune")


def test_band_split_and_detector(gold):
    x = gold["st/x"]
    sub, body, air = at.split_sub_body_air(x, 48000, 110.0, 5000.0)
    assert gold.matches("st/sub", sub) and gold.matches("st/body", body) and gold.matches("st/air", air)
    assert np.array_equal(at.detector_sidechain(body, 48000, 110.0, 3000.0), gold["st/det"])


def test_sosfiltfilt_restatement_is_scipy():
    """The sample-level specification the CUDA kernel follows equals scipy.signal.sosfiltfilt."""
    rng = np.random.default_rng(5)
    x = rng.standard_normal(700).astype(np.float32)
    for cutoff, bt in ((110.0, "low"), (5000.0, "high"), (3000.0, "low")):
        sos = at.butter_sos(48000, cutoff, bt)
        assert np.array_equal(at.sosfiltfilt_restated(sos, x), scipy.signal.sosfiltfilt(sos, x))
    with pytest.raises(ValueError):
        at.sosfiltfilt_restated(at.butter_sos(48000, 110.0, "low"), np.zeros(15))


def test_frame_features_and_ratio_track(gold):
    cfg = at.AutotuneConfig()
    centers, rms, flat, pitch, conf = at.frame_features(gold["st/det"], 48000, cfg)
    f = gold["st/features"]
    assert np.array_equal(rms, f[:, 0]) and np.array_equal(flat, f[:, 1])
    assert np.array_equal(pitch, f[:, 2]) and np.array_equal(conf, f[:, 3])
    assert np.array_equal(at.ratio_track(gold["st/det"], 48000, cfg), gold["st/ratio_track"])
    got = np.array([at.nearest_scale_freq(v, "D", "minor") for v in (97.3, 233.1, 440.0, 1234.5)])
    assert np.array_equal(got, gold["st/nearest"])


def test_granular_shifter(gold):
    assert gold.matches("st/corrected", at.granular_pitch_shift(gold["st/body"], gold["st/ratio_track"]))
    assert gold.matches("st/shift_manual", at.granular_pitch_shift(gold["st/body"], gold["st/ratio_manual"]))
    ones = np.ones(100, dtype=np.float32)
    assert np.array_equal(at.granular_pitch_shift(gold["st/body"][:100], ones), gold["st/body"][:100])  # early out, no latency


def test_sub_layer_and_mode_output(gold):
    x = gold["st/x"]
    assert gold.matches("st/env", at.envelope_follow(x, 48000))
    assert gold.matches("st/sub_layer", at.sub_layer(x, 48000, at.AutotuneConfig()))
    assert gold.matches("st/output", at.apply_autotune_v1(x, 48000, at.AutotuneConfig())["output"])


@pytest.mark.parametrize("name", list(qd_cases.AUTOTUNE_CASES))
def test_autotune_pipeline_matches_reference(gold, name):
    kind, seed, n, sr, kw = qd_cases.AUTOTUNE_CASES[name]
    x = qd_cases.make_signal(kind, seed, n, sr)
    assert gold.matches(f"{name}/x", x)
    y, taps = at.process_audio_autotune(x, sr, **{k: v for k, v in kw.items()
                                                  if k not in ("smear", "bin_smoothing", "post_quant")})
    for got, key in ((y, "y"), (taps["pre_quant"], "pre_quant"), (taps["post_dist"], "post_dist")):
        assert gold.matches(f"{name}/{key}", got), f"{name}/{key}: max abs diff {gold.max_abs_err(f'{name}/{key}', got):.3e}"
