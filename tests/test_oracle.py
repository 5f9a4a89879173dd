"""CPU: pin oracle/qd_oracle.py against fixtures produced by the live reference
(tests/golden/make_golden.py) and against the reference's own known-answer tests."""
import os

import numpy as np
import pytest
import scipy.signal

import qd_cases
from oracle import qd_oracle as orc

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def tables():
    return np.load(os.path.join(G, "tables.npz"))


@pytest.fixture(scope="module")
def stages():
    return qd_cases.Golden("stages")


@pytest.fixture(scope="module")
def pipe():
    return qd_cases.Golden("pipeline")


def test_target_bins_and_masks_bit_exact(tables):
    n = 0
    for k in tables.files:
        if k.startswith("tb/") and k != "tb/kat4":
            sr, n_fft, key, scale = k[3:].split("_", 3)
            freqs = np.fft.rfftfreq(int(n_fft), d=1.0 / int(sr))
            assert np.array_equal(orc.target_bins_for_freqs(freqs, key, scale), tables[k]), k
            assert np.array_equal(orc.quantize_band_mask(freqs, 110.0, 5000.0), tables["mask/" + k[3:]]), k
            n += 1
    assert n == 10
    freqs = np.fft.rfftfreq(2048, d=1.0 / 48000)
    assert np.array_equal(orc.quantize_band_mask(freqs, 0.0, 0.0), tables["mask/wide"])
    for f0 in (55.0, 110.0, 441.3):
        assert np.array_equal(orc.harmonic_target_bins(freqs, f0), tables[f"htb/{f0}"])


def test_reference_quantizer_kats(tables):
    # reference tests/test_quantizer.py:10-23
    freqs = np.array([0.0, 430.0, 440.0, 450.0])
    tb = orc.target_bins_for_freqs(freqs, "A", "minor")
    assert list(tb) == [0, 2, 2, 2] and np.array_equal(tb, tables["tb/kat4"])
    mags = np.array([0.0, 1.0, 0.0, 0.0])
    ph = np.zeros(4)
    # :26-49 energy moves 1 -> 2, phases unchanged
    nm, nph = orc.quantize_frames(mags, ph, tb, None, 1.0, 0.0, False)
    assert np.isclose(nm[1], 0.0) and np.isclose(nm[2], 1.0) and np.isclose(nm.sum(), 1.0)
    assert np.allclose(nph, ph)
    # :52-84 smear radius 1
    nm, _ = orc.quantize_frames(mags, ph, tb, None, 1.0, 0.8, False, smear_radius=1)
    assert 0.0 < nm[1] < 0.5 and nm[2] > nm[1] and nm[3] > 0.0
    # :87-107 smoothing only conserves interior energy shape
    nm, _ = orc.quantize_frames(np.array([0.0, 1.0, 0.0, 0.0]), ph, tb, None, 0.0, 0.0, True)
    assert np.allclose(nm, [0.25, 0.5, 0.25, 0.0])
    # :110-131 active mask keeps masked bins
    nm, _ = orc.quantize_frames(mags, ph, tb, np.array([False, False, True, True]), 1.0, 0.0, False)
    assert np.allclose(nm, mags)
    with pytest.raises(ValueError):
        orc.note_name_to_pitch_class("H")
    with pytest.raises(KeyError):
        orc.scale_notes("C", "lydian", 20.0, 2000.0)


def test_quantize_frames_matches_reference(stages):
    freqs = np.fft.rfftfreq(2048, d=1.0 / 48000)
    tb = orc.target_bins_for_freqs(freqs, "D", "minor")
    mask = orc.quantize_band_mask(freqs, 110.0, 5000.0)
    cfg = {"default": (1.0, 0.1, True, mask), "growl": (0.9, 0.3, True, mask),
           "nosmooth": (0.75, 0.4, False, mask), "nomask": (1.0, 0.1, True, None),
           "smear0": (1.0, 0.0, True, mask), "smear1": (0.5, 1.0, True, mask)}
    for tag, (snap, smear, smooth, m) in cfg.items():
        nm, nph = orc.quantize_frames(stages["q/mags"], stages["q/phases"], tb, m, snap, smear, smooth)
        assert stages.matches(f"q/{tag}/mags", nm), tag
        assert stages.matches(f"q/{tag}/phases", nph), tag


def test_stft_istft_matches_reference(stages):
    x = stages["stft/x"]
    for nf in (512, 2048):
        S, _ = orc.stft(x, 48000, n_fft=nf)
        assert stages.matches(f"stft/{nf}/S", S)
        assert stages.matches(f"stft/{nf}/y", orc.istft(S, 48000, n_fft=nf, length=len(x)))


def test_spectral_fx_matches_reference(stages):
    fm, fp = stages["fx/mag"], stages["fx/phase"]
    cfg = {"bitcrush05": ("bitcrush", 0.5), "bitcrush03": ("bitcrush", 0.3), "bitcrush08": ("bitcrush", 0.8),
           "disp06": ("phase_dispersal", 0.6), "disp03": ("phase_dispersal", 0.3),
           "scr055": ("bin_scramble", 0.55), "scr03": ("bin_scramble", 0.3), "scr09": ("bin_scramble", 0.9)}
    for tag, (mode, s) in cfg.items():
        np.random.seed(99)
        frames = [orc.apply_spectral_fx(fm.copy(), fp.copy(), mode, s, {}) for t in range(3)]
        assert stages.matches(f"fx/{tag}/mag", np.array([a for a, _ in frames])), tag
        assert stages.matches(f"fx/{tag}/phase", np.array([b for _, b in frames])), tag
    a, _ = orc.fx_bitcrush(fm, fp, method="uniform", step=0.07, threshold=0.01)
    assert stages.matches("fx/uniform/mag", a)


def test_formant_shift_matches_reference(stages):
    fm = stages["fx/mag"]
    for st in (3.0, -5.0, 12.0, -0.5):
        assert stages.matches(f"fx/formant/{st}", orc.formant_shift_frame(fm, st)), st
        assert stages.matches(f"fx/formant/zeros/{st}", orc.formant_shift_frame(stages["fx/formant/zeros_in"], st)), st
        assert stages.matches(f"fx/formant/257/{st}", orc.formant_shift_frame(stages["fx/formant/in257"], st)), st
    assert np.array_equal(orc.formant_shift_frame(fm, 0.0), fm)


def test_time_domain_stages_match_reference(stages):
    x = stages["td/x"]
    assert np.array_equal(orc.apply_distortion(x, "wavefold", fold_amount=5.0, bias=0.1), stages["td/wavefold"])
    assert np.array_equal(orc.apply_distortion(x, "tube", drive=4.0, warmth=0.7), stages["td/tube"])
    with pytest.raises(ValueError):
        orc.apply_distortion(x, "fuzz")
    for sr in (48000, 44100):
        y, g = orc.peak_limiter(x, sr, ceiling_db=-1.0, lookahead_ms=5.0, release_ms=30.0)
        assert np.array_equal(y, stages[f"td/lim/{sr}/y"]) and np.array_equal(g, stages[f"td/lim/{sr}/g"])
    assert orc.limiter_constants(44100, -1.0, 5.0, 30.0)[1] == 220  # round-half-even (SURVEY C.7)
    lo, hi = orc.linkwitz_riley_split(x, 48000, 300.0)
    assert np.array_equal(lo, stages["td/xo/low"]) and np.array_equal(hi, stages["td/xo/high"])
    sl, sh = orc.linkwitz_riley_sos(48000, 300.0)
    assert np.array_equal(sl, stages["td/xo/sos_low"]) and np.array_equal(sh, stages["td/xo/sos_high"])
    assert np.array_equal(orc.saturate_lowband(lo, drive=2.5), stages["td/sat"])
    with pytest.raises(ValueError):
        orc.linkwitz_riley_sos(48000, 24000.0)


def test_sosfilt_matches_scipy():
    rng = np.random.default_rng(3)
    x = rng.standard_normal(5000)
    sl, sh = orc.linkwitz_riley_sos(44100, 180.0)
    for sos in (sl, sh):
        assert np.array_equal(orc.sosfilt(sos, x), scipy.signal.sosfilt(sos, x))


@pytest.mark.parametrize("name", list(qd_cases.CASES))
def test_pipeline_matches_reference(pipe, name):
    kind, seed, n, sr, n_fft, rng_seed, kw = qd_cases.CASES[name]
    x = qd_cases.make_signal(kind, seed, n, sr)
    assert pipe.matches(f"{name}/x", x), "synthetic input drifted from the fixture"
    if rng_seed is not None:
        np.random.seed(rng_seed)
    y, taps = orc.process_audio(x, sr, n_fft=n_fft, **kw)
    assert y.dtype == np.float32 and y.shape == x.shape
    for got, key in ((y, "y"), (taps["pre_quant"], "pre_quant"), (taps["post_dist"], "post_dist")):
        err = pipe.max_abs_err(f"{name}/{key}", got)
        assert pipe.matches(f"{name}/{key}", got), f"{name}/{key}: max abs diff {err:.3e}"


def test_null_test_definition():
    a = np.zeros(100, dtype=np.float32)
    assert orc.null_test_db(a, a) == -200.0
    assert abs(orc.null_test_db(a + 0.1, a) + 20.0) < 1e-4


@pytest.mark.parametrize("name", list(qd_cases.ANALYSIS_CASES))
def test_cents_metric_matches_reference(name):
    """avg_cents_offset_from_scale (dsp/analyses.py:53-142): oracle and the host cents table vs the live reference."""
    g = qd_cases.Golden("analysis")
    kind, seed, n, sr, key, scale, kw = qd_cases.ANALYSIS_CASES[name]
    x = qd_cases.make_signal(kind, seed, n, sr)
    assert g.matches(f"{name}/x", x)
    avg, per, bins = orc.avg_cents_offset_from_scale(x, sr, key, scale, return_bins=True, **kw)
    assert np.array_equal(per, g[f"{name}/per_peak"])
    assert (np.isnan(avg) and np.isnan(g[f"{name}/avg"])) or avg == float(g[f"{name}/avg"])
    # the product's per-bin table reproduces the per-peak values from the chosen bins
    from quantumdistortion_b200.analyses import scale_cents_table
    table = scale_cents_table(np.fft.rfftfreq(kw.get("frame_length", 2048), d=1.0 / sr), key, scale)
    flat = bins.reshape(-1)
    assert np.array_equal(table[flat[flat >= 0]], per)
