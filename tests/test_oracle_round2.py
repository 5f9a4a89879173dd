"""CPU: round-2 fixtures from the live reference (tests/golden/make_golden.py round2 / refwav).

* the oracle against spectral_fx_params overrides, spectral FX at other n_fft, n_fft 8192 with every option,
  autotune_v1 kept on the high band of a multiband render, and UI dicts that stay in autotune_v1 -- bit for bit;
* the north-star's integer gate: the product's np.random replay (tables.replay_fx_table) against scramble indices
  recovered from the reference's own bin_scramble output -- elementwise equal;
* the reference's own audio files (BASELINE configs[0]): literal render_cli default and spectral_bins, plus the
  reference's committed tests/data/processed/*_multiband(.|_bitcrush).wav renders as a loose known-answer test.
"""

import numpy as np
import pytest

import qd_cases
from oracle import qd_autotune as at
from oracle import qd_oracle as orc

_AT_DROP = ("smear", "bin_smoothing", "post_quant", "use_multiband", "crossover_hz", "lowband_drive")


@pytest.fixture(scope="module")
def r2():
    return qd_cases.Golden("round2")


@pytest.fixture(scope="module")
def wav():
    return qd_cases.Golden("refwav")


@pytest.fixture(scope="module")
def renders():
    return qd_cases.Golden("refwav_renders")


@pytest.mark.parametrize("name", list(qd_cases.CASES_R2))
def test_round2_pipeline_cases(r2, name):
    kind, seed, n, sr, n_fft, rng_seed, kw = qd_cases.CASES_R2[name]
    x = qd_cases.make_signal(kind, seed, n, sr)
    assert r2.matches(f"{name}/x", x), "synthetic input drifted from the fixture"
    if rng_seed is not None:
        np.random.seed(rng_seed)
    y, taps = orc.process_audio(x, sr, n_fft=n_fft, **kw)
    for got, key in ((y, "y"), (taps["pre_quant"], "pre_quant"), (taps["post_dist"], "post_dist")):
        err = r2.max_abs_err(f"{name}/{key}", got)
        if n_fft == 8192:
            # SURVEY.md section 8(c): the vectorised restatement is 0.0 off up to n_fft 4096 and ~1.5e-8 at 8192
            # (summation order of 106-source targets); the float32 cast hides it except on isolated samples
            assert err <= 2e-7, f"{name}/{key}"
        else:
            assert r2.matches(f"{name}/{key}", got), f"{name}/{key}: max abs diff {err:.3e}"


@pytest.mark.parametrize("name", list(qd_cases.AT_MB_CASES))
def test_autotune_inside_multiband_snap0(r2, name):
    """dsp/pipeline.py:1326-1327, :1076, :537-601: quantize_mode stays "autotune_v1", multiband stays on."""
    kind, seed, n, sr, kw = qd_cases.AT_MB_CASES[name]
    x = qd_cases.make_signal(kind, seed, n, sr)
    assert r2.matches(f"{name}/x", x)
    y, taps = orc.process_audio(x, sr, quantize_mode="autotune_v1", **kw)
    for got, key in ((y, "y"), (taps["pre_quant"], "pre_quant"), (taps["post_dist"], "post_dist")):
        assert r2.matches(f"{name}/{key}", got), f"{name}/{key}"


def _ui_explicit(cfg, kw):
    """What dsp/pipeline.py:923-1008 makes of a UI dict whose mode stays autotune_v1, as explicit keyword arguments
    of the autotune oracle (multiband is dropped by :1326-1327 because snap_strength > 0)."""
    q = cfg.get("quantization", {})
    out = dict(kw)
    for src, dst in (("key", "key"), ("scale", "scale"), ("sub_enabled", "sub_enabled"), ("sub_source", "sub_source"),
                     ("sub_note", "sub_note"), ("sub_scale_degree", "sub_scale_degree"), ("sub_octave", "sub_octave"),
                     ("sub_level", "sub_level"), ("sub_cut_hz", "sub_cut_hz"), ("air_cut_hz", "air_cut_hz"),
                     ("air_mix", "air_mix")):
        if src in q:
            out[dst] = q[src]
    return out


@pytest.mark.parametrize("name", list(qd_cases.UI_AT_CASES))
def test_ui_dict_autotune_keys(r2, name):
    kind, seed, n, sr, _rng, cfg, kw = qd_cases.UI_AT_CASES[name]
    x = qd_cases.make_signal(kind, seed, n, sr)
    assert r2.matches(f"{name}/x", x)
    y, _ = at.process_audio_autotune(x, sr, **_ui_explicit(cfg, kw))
    assert r2.matches(f"{name}/y", y), "the quantization.* sub-layer keys of the UI dict reach the autotune render"
    # the product's parser resolves the dict to the same C struct as the explicit keywords
    from quantumdistortion_b200.pipeline import _resolve_kwargs
    a, _ = _resolve_kwargs(n, sr, 2048, dict(kw, config=cfg))
    b, _ = _resolve_kwargs(n, sr, 2048, dict(_ui_explicit(cfg, kw), quantize_mode="autotune_v1"))
    assert bytes(a) == bytes(b)


@pytest.mark.parametrize("n_bins", [1025, 257])
def test_scramble_permutations_bit_exact(r2, n_bins):
    """North-star: "scramble permutations must be bit-exact".  Three consecutive frames per mode from one seed."""
    from quantumdistortion_b200 import tables
    for tag, window in (("pick_w9", 9), ("pick_w3", 3), ("pick_w15", 15)):
        np.random.seed(4321)
        got = tables.replay_fx_table(("pick", window // 2), 1, 3, n_bins)
        assert got.dtype == np.int16
        assert np.array_equal(got[0], r2[f"scr/{n_bins}/{tag}"]), tag
        assert np.array_equal(got[1], np.broadcast_to(np.arange(n_bins, dtype=np.int16), (3, n_bins))), "unused pass stays identity"
    np.random.seed(4321)
    got = tables.replay_fx_table(("swap",), 1, 3, n_bins)
    ref = r2[f"scr/{n_bins}/swap"]
    assert np.array_equal(got[0], ref)
    for t in range(3):
        assert np.array_equal(np.sort(ref[t]), np.arange(n_bins)), "swap is a permutation"
    # the strength -> (mode, window) mapping the renders use (dsp/pipeline.py:121-138)
    assert tables.resolve_spectral_fx("bin_scramble", 0.55, {})["rng"] == ("pick", 4)    # window int(3 + 12 * .55^1.2) = 8 -> 9
    assert tables.resolve_spectral_fx("bin_scramble", 0.3, {})["rng"] == ("swap",)
    assert tables.resolve_spectral_fx("bin_scramble", 0.9, {"window": 4})["rng"] == ("pick", 2)
    assert tables.resolve_spectral_fx("bin_scramble", 0.9, {"window": 1, "mode": "swap"})["rng"] == ("swap",)


def test_dispersal_jitter_replay(r2):
    from quantumdistortion_b200 import tables
    np.random.seed(4321)
    got = tables.replay_fx_table(("jitter",), 1, 3, 1025)[0]
    ref = r2["scr/1025/jitter"]            # (rand * 2 - 1) * 1.0 wrapped to [-pi, pi): |jitter| < 1, no wrap
    assert got.dtype == np.float32 and np.array_equal(got, ref.astype(np.float32))


# ---------------------------------------------------------------------------------------------- the reference's own files
def _wav_input(wav, name):
    return wav[f"{name}/x16"].astype(np.float32) / 32768.0, int(wav[f"{name}/sr"])


@pytest.mark.parametrize("name", list(qd_cases.REF_WAVS))
def test_reference_files_spectral_bins(wav, renders, name):
    x, sr = _wav_input(wav, name)
    y, _ = orc.process_audio(x, sr)
    assert renders.matches(f"{name}/y_spectral_bins", y)


@pytest.mark.parametrize("name", ["example_bass", "wobble_bass"])
def test_reference_files_literal_default(wav, renders, name):
    """scripts/render_cli.py:32: process_audio(audio, sr) -- the reference's default mode is autotune_v1."""
    x, sr = _wav_input(wav, name)
    y, _ = at.process_audio_autotune(x, sr)
    assert renders.matches(f"{name}/y_default", y)


@pytest.mark.parametrize("name", [n for n in qd_cases.REF_WAVS if n != "example_bass"])
def test_reference_processed_renders_kat(wav, renders, name):
    """SURVEY.md section 4: the reference's committed *_multiband.wav / *_multiband_bitcrush.wav renders (made by an
    older revision of its code) reproduce to a few PCM16 steps with sub_cut_hz = air_cut_hz = 0."""
    from quantumdistortion_b200.audio_io import float_to_pcm16
    x, sr = _wav_input(wav, name)
    kw = dict(use_multiband=True, crossover_hz=300.0, sub_cut_hz=0.0, air_cut_hz=0.0)
    y, _ = orc.process_audio(x, sr, **kw)
    got, ref = renders.at(f"{name}/kat_multiband", float_to_pcm16(y))
    d = np.abs(got.astype(np.int32) - ref.astype(np.int32))
    assert int(d.max()) <= 6, int(d.max())
    y, _ = orc.process_audio(x, sr, spectral_fx_mode="bitcrush", spectral_fx_strength=0.5, **kw)
    got, ref = renders.at(f"{name}/kat_multiband_bitcrush", float_to_pcm16(y))
    d = np.abs(got.astype(np.int32) - ref.astype(np.int32))
    assert int(d.max()) <= 6, int(d.max())
