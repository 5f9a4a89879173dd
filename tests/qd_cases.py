"""Named pipeline cases used by make_golden.py (live reference) and the parity tests.

Every case is (signal kind, seed, n_samples, sr, n_fft, np.random seed or None, kwargs for
process_audio).  quantize_mode="spectral_bins" is always passed (SURVEY.md section 0.1).
"""
from __future__ import annotations

import fnmatch
import hashlib
import os

import numpy as np

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# ---------------------------------------------------------------- fixture files (tests/golden/*.npz)
# Whole renders of every case would make the fixtures tens of megabytes.  An array larger than GOLDEN_SAMPLE elements is
# therefore stored as the SHA-256 digest of the whole array (exact comparisons stay exact) plus its values at
# GOLDEN_SAMPLE fixed positions drawn with a seed (toleranced comparisons); the positions are stored too, one set per
# array size.  Arrays the tests feed back into the code as inputs are kept whole (GOLDEN_WHOLE).
GOLDEN_SAMPLE = 1024
GOLDEN_WHOLE = {
    "tables": ("*",),
    "refwav": ("*",),                                     # the reference's own WAV files: cannot be regenerated
    "stages": ("q/mags", "q/phases", "fx/mag", "fx/phase", "fx/formant/zeros_in", "fx/formant/in257", "stft/x", "td/*"),
    "autotune": ("st/x", "st/body", "st/det", "st/ratio_track", "st/ratio_manual"),
    "round2": ("scr/*",),
    "pipeline": ("sb_wide_mask/post_dist",),
    "scenarios": ("formant_six/*",),
}


def _digest(a: np.ndarray) -> str:
    a = np.ascontiguousarray(a)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()


def save_golden(name: str, arrays: dict) -> str:
    """Write tests/golden/<name>.npz in the form Golden reads."""
    whole = GOLDEN_WHOLE.get(name, ())
    out = {}
    for key, a in arrays.items():
        a = np.asarray(a)
        if a.size <= GOLDEN_SAMPLE or any(fnmatch.fnmatchcase(key, p) for p in whole):
            out[key] = a
            continue
        ik = f"#idx/{a.size}"
        if ik not in out:
            out[ik] = np.sort(np.random.default_rng(a.size).choice(a.size, GOLDEN_SAMPLE, replace=False)).astype(np.uint32)
        out[f"{key}#sha"] = np.array(_digest(a))
        out[f"{key}#shape"] = np.array(a.shape, dtype=np.int64)
        out[f"{key}#v"] = a.reshape(-1)[out[ik]]
    path = os.path.join(GOLDEN_DIR, f"{name}.npz")
    np.savez_compressed(path, **out)
    return path


class Golden:
    """One fixture file: `g[key]` is an array stored whole; `matches` compares a whole array exactly, `at` returns the
    values to compare at the stored positions."""

    def __init__(self, name: str):
        self._z = np.load(os.path.join(GOLDEN_DIR, f"{name}.npz"))
        self._files = set(self._z.files)

    def __getitem__(self, key):
        if key not in self._files:
            raise KeyError(f"{key} is not stored whole (use Golden.matches / Golden.at)")
        return self._z[key]

    def shape(self, key):
        return self._z[key].shape if key in self._files else tuple(int(s) for s in self._z[f"{key}#shape"])

    def matches(self, key, got) -> bool:
        """np.array_equal(got, <the whole fixture array>)."""
        got = np.asarray(got)
        if key in self._files:
            return bool(np.array_equal(got, self._z[key]))
        v = self._z[f"{key}#v"]
        if got.shape != self.shape(key):
            return False
        cast = got.astype(v.dtype)
        return bool(np.array_equal(cast, got)) and _digest(cast) == str(self._z[f"{key}#sha"])

    def at(self, key, got):
        """(got, fixture) at the stored positions, after checking that `got` has the fixture's shape."""
        got = np.asarray(got)
        assert got.shape == self.shape(key), (key, got.shape, self.shape(key))
        if key in self._files:
            return got, self._z[key]
        idx = self._z[f"#idx/{int(np.prod(got.shape))}"]
        return got.reshape(-1)[idx], self._z[f"{key}#v"]

    def max_abs_err(self, key, got) -> float:
        a, b = self.at(key, got)
        return float(np.max(np.abs(a.astype(np.result_type(a, np.float64)) - b))) if b.size else 0.0

    def input(self, name, x):
        """`x`, regenerated from its seed, after checking that it is the input of the fixture's case `name`."""
        assert self.matches(f"{name}/x", x), f"{name}: input drifted from the fixture"
        return x


GROWL = dict(key="F", scale="minor", snap_strength=0.9, smear=0.3, bin_smoothing=True,
             pre_quant=True, post_quant=True, distortion_mode="wavefold",
             distortion_params={"fold_amount": 5.0, "bias": 0.1, "drive": 1.0, "warmth": 0.5},
             limiter_on=True, limiter_ceiling_db=-1.0, dry_wet=1.0)
CLANG = dict(key="D", scale="minor", snap_strength=0.75, smear=0.4, bin_smoothing=True,
             pre_quant=True, post_quant=True, distortion_mode="tube",
             distortion_params={"fold_amount": 1.0, "bias": 0.0, "drive": 4.0, "warmth": 0.7},
             limiter_on=True, limiter_ceiling_db=-2.0, dry_wet=1.0)
GLUE = dict(key="C", scale="major", snap_strength=0.4, smear=0.2, bin_smoothing=True,
            pre_quant=True, post_quant=False, distortion_mode="tube",
            distortion_params={"fold_amount": 1.0, "bias": 0.0, "drive": 2.0, "warmth": 0.3},
            limiter_on=True, limiter_ceiling_db=-1.0, dry_wet=0.7)

N = 12000  # 0.25 s @ 48 kHz -> 24 frames at n_fft 2048

# name: (kind, seed, n, sr, n_fft, rng_seed, kwargs)
CASES = {
    "sb_default_bass": ("bass", 0, N, 48000, 2048, None, {}),
    "sb_default_noise": ("noise", 1, N, 48000, 2048, None, {}),
    "sb_default_loud": ("loud", 2, N, 48000, 2048, None, {}),
    "sb_default_441": ("bass", 3, 11025, 44100, 2048, None, {}),
    "sb_ragged_len": ("bass", 4, 5003, 48000, 2048, None, {}),
    "sb_short": ("noise", 5, 700, 48000, 2048, None, {}),
    "sb_passthrough": ("bass", 6, N, 48000, 2048, None, {"passthrough_test": True}),
    "sb_growl": ("loud", 7, N, 48000, 2048, None, dict(GROWL)),
    "sb_clang_tube": ("bass", 8, N, 48000, 2048, None, dict(CLANG)),
    "sb_glue_pre_only_drywet": ("bass", 9, N, 48000, 2048, None, dict(GLUE)),
    "sb_post_only": ("bass", 10, N, 48000, 2048, None, {"pre_quant": False}),
    "sb_no_quant": ("bass", 11, N, 48000, 2048, None, {"snap_strength": 0.0}),
    "sb_no_limiter_trim_delta": ("loud", 12, N, 48000, 2048, None,
                                 {"limiter_on": False, "output_trim_db": -3.0, "delta_listen": True,
                                  "dry_wet": 0.5}),
    "sb_no_smooth_no_smear": ("noise", 13, N, 48000, 2048, None, {"bin_smoothing": False, "smear": 0.0}),
    "sb_wide_mask": ("noise", 14, N, 48000, 2048, None, {"sub_cut_hz": 0.0, "air_cut_hz": 0.0,
                                                          "key": "A", "scale": "pentatonic"}),
    "sb_harmonic_lock": ("bass", 15, N, 48000, 2048, None, {"harmonic_lock_hz": 55.0}),
    "mb_default": ("bass", 20, N, 48000, 2048, None, {"use_multiband": True, "crossover_hz": 300.0}),
    "mb_loud_drive": ("loud", 21, N, 48000, 2048, None, {"use_multiband": True, "crossover_hz": 300.0,
                                                          "lowband_drive": 2.5, "dry_wet": 0.8}),
    "mb_growl_bitcrush": ("loud", 22, N, 48000, 2048, 1234,
                          dict(GROWL, use_multiband=True, spectral_fx_mode="bitcrush",
                               spectral_fx_strength=0.5)),
    "mb_growl_bitcrush_lo": ("bass", 23, N, 48000, 2048, 1234,
                             dict(GROWL, use_multiband=True, spectral_fx_mode="bitcrush",
                                  spectral_fx_strength=0.3)),
    "mb_growl_dispersal": ("loud", 24, N, 48000, 2048, 1234,
                           dict(GROWL, use_multiband=True, spectral_fx_mode="phase_dispersal",
                                spectral_fx_strength=0.6)),
    "mb_growl_dispersal_det": ("bass", 25, N, 48000, 2048, 1234,
                               dict(GROWL, use_multiband=True, spectral_fx_mode="phase_dispersal",
                                    spectral_fx_strength=0.3)),
    "mb_growl_scramble_pick": ("loud", 26, N, 48000, 2048, 1234,
                               dict(GROWL, use_multiband=True, spectral_fx_mode="bin_scramble",
                                    spectral_fx_strength=0.55)),
    "mb_growl_scramble_swap": ("bass", 27, N, 48000, 2048, 1234,
                               dict(GROWL, use_multiband=True, spectral_fx_mode="bin_scramble",
                                    spectral_fx_strength=0.3)),
    "sb_freeze": ("bass", 28, N, 48000, 2048, None, {"spectral_freeze": True}),
    "mb_freeze_bitcrush": ("loud", 29, N, 48000, 2048, 1234,
                           dict(GROWL, use_multiband=True, spectral_freeze=True, spectral_fx_mode="bitcrush",
                                spectral_fx_strength=0.5)),
    "sb_formant_up": ("bass", 34, N, 48000, 2048, None, {"formant_shift": 3.0}),
    "sb_formant_down_growl": ("loud", 35, N, 48000, 2048, None, dict(GROWL, formant_shift=-5.0)),
    "mb_formant_bitcrush": ("loud", 36, N, 48000, 2048, 1234,
                            dict(GROWL, use_multiband=True, formant_shift=2.0, spectral_fx_mode="bitcrush",
                                 spectral_fx_strength=0.5)),
    "sb_formant_freeze": ("bass", 37, N, 48000, 2048, None, {"formant_shift": 7.0, "spectral_freeze": True}),
    "nfft1024_formant": ("bass", 38, 6000, 48000, 1024, None, {"formant_shift": -2.0}),
    "nfft512": ("bass", 30, 6000, 48000, 512, None, {}),
    "nfft1024": ("bass", 31, 6000, 48000, 1024, None, {}),
    "nfft4096": ("bass", 32, N, 48000, 4096, None, {}),
    "nfft8192": ("bass", 33, 20000, 48000, 8192, None, {}),
}

# Round-2 additions (fixtures in tests/golden/round2.npz; same tuple layout plus an optional `precision`):
# spectral_fx_params overrides, uniform bitcrush, spectral FX away from n_fft 2048, the float64 FX kernels,
# n_fft 8192 with every option, and autotune_v1 kept on the high band of a multiband render (snap_strength = 0).
_MB = dict(GROWL, use_multiband=True)
CASES_R2 = {
    "mb_bitcrush_uniform": ("loud", 100, N, 48000, 2048, 1234,
                            dict(_MB, spectral_fx_mode="bitcrush", spectral_fx_strength=0.5,
                                 spectral_fx_params={"method": "uniform"})),
    "mb_bitcrush_uniform_step_thr": ("bass", 101, N, 48000, 2048, 1234,
                                     dict(_MB, spectral_fx_mode="bitcrush", spectral_fx_strength=0.3,
                                          spectral_fx_params={"method": "uniform", "step": 0.004, "threshold": 0.003})),
    "mb_bitcrush_log_stepdb_thr": ("loud", 102, N, 48000, 2048, 1234,
                                   dict(_MB, spectral_fx_mode="bitcrush", spectral_fx_strength=0.7,
                                        spectral_fx_params={"step_db": 3.0, "threshold": 0.02})),
    "mb_bitcrush_unknown_method": ("bass", 103, N, 48000, 2048, 1234,
                                   dict(_MB, spectral_fx_mode="bitcrush", spectral_fx_strength=0.6,
                                        spectral_fx_params={"method": "cubic"})),
    "mb_dispersal_thresh_det": ("loud", 104, N, 48000, 2048, 1234,
                                dict(_MB, spectral_fx_mode="phase_dispersal", spectral_fx_strength=0.6,
                                     spectral_fx_params={"thresh": 0.05, "randomized": False})),
    "mb_dispersal_forced_random": ("bass", 105, N, 48000, 2048, 1234,
                                   dict(_MB, spectral_fx_mode="phase_dispersal", spectral_fx_strength=0.2,
                                        spectral_fx_params={"randomized": True, "rand_amt": 0.4, "amount": 1.1,
                                                            "thresh": 0.0})),
    "mb_scramble_window_swap": ("loud", 106, N, 48000, 2048, 1234,
                                dict(_MB, spectral_fx_mode="bin_scramble", spectral_fx_strength=0.7,
                                     spectral_fx_params={"window": 9, "mode": "swap"})),
    "mb_scramble_window_pick": ("bass", 107, N, 48000, 2048, 1234,
                                dict(_MB, spectral_fx_mode="bin_scramble", spectral_fx_strength=0.2,
                                     spectral_fx_params={"window": 4, "mode": "random_pick"})),
    "mb_scramble_unknown_mode": ("bass", 108, N, 48000, 2048, 1234,
                                 dict(_MB, spectral_fx_mode="bin_scramble", spectral_fx_strength=0.5,
                                      spectral_fx_params={"mode": "shuffle"})),
    "nfft512_bitcrush": ("loud", 110, 6000, 48000, 512, 1234,
                         dict(_MB, spectral_fx_mode="bitcrush", spectral_fx_strength=0.5)),
    "nfft512_scramble_pick": ("bass", 111, 6000, 48000, 512, 1234,
                              dict(_MB, spectral_fx_mode="bin_scramble", spectral_fx_strength=0.55)),
    "nfft1024_dispersal": ("loud", 112, 6000, 48000, 1024, 1234,
                           dict(_MB, spectral_fx_mode="phase_dispersal", spectral_fx_strength=0.6)),
    "nfft4096_bitcrush": ("loud", 113, N, 48000, 4096, 1234,
                          dict(_MB, spectral_fx_mode="bitcrush", spectral_fx_strength=0.5)),
    "nfft4096_dispersal": ("bass", 114, N, 48000, 4096, 1234,
                           dict(_MB, spectral_fx_mode="phase_dispersal", spectral_fx_strength=0.6)),
    "nfft4096_scramble_pick": ("loud", 115, N, 48000, 4096, 1234,
                               dict(_MB, spectral_fx_mode="bin_scramble", spectral_fx_strength=0.55)),
    "nfft4096_scramble_swap": ("bass", 116, N, 48000, 4096, 1234,
                               dict(_MB, spectral_fx_mode="bin_scramble", spectral_fx_strength=0.3)),
    "nfft4096_formant": ("bass", 117, N, 48000, 4096, None, {"formant_shift": 4.0}),
    "nfft8192_bitcrush": ("loud", 120, 20000, 48000, 8192, 1234,
                          dict(_MB, spectral_fx_mode="bitcrush", spectral_fx_strength=0.5)),
    "nfft8192_dispersal": ("bass", 121, 20000, 48000, 8192, 1234,
                           dict(_MB, spectral_fx_mode="phase_dispersal", spectral_fx_strength=0.6)),
    "nfft8192_scramble_pick": ("loud", 122, 20000, 48000, 8192, 1234,
                               dict(_MB, spectral_fx_mode="bin_scramble", spectral_fx_strength=0.55)),
    "nfft8192_scramble_swap": ("bass", 123, 20000, 48000, 8192, 1234,
                               dict(_MB, spectral_fx_mode="bin_scramble", spectral_fx_strength=0.3)),
    "nfft8192_freeze": ("bass", 124, 20000, 48000, 8192, None, {"spectral_freeze": True}),
    "nfft8192_formant": ("bass", 125, 20000, 48000, 8192, None, {"formant_shift": 3.0}),
    "nfft8192_multiband": ("loud", 126, 20000, 48000, 8192, None, {"use_multiband": True}),
}
# cases of CASES / CASES_R2 that are ALSO rendered with precision="float64" against the same fixture
F64_CASES = ("mb_growl_bitcrush", "mb_growl_dispersal", "mb_growl_scramble_pick", "nfft4096_bitcrush",
             "nfft4096_dispersal", "nfft4096_scramble_pick", "nfft4096_scramble_swap", "nfft4096_formant",
             "nfft512_scramble_pick")

# quantize_mode left at the reference default ("autotune_v1") with snap_strength = 0 inside a multiband render:
# the only combination that keeps both (dsp/pipeline.py:1326-1327, :1076, :537-601)
AT_MB_CASES = {
    "at_mb_snap0": ("loud", 130, N, 48000, {"snap_strength": 0.0, "use_multiband": True, "lowband_drive": 1.7}),
    "at_mb_snap0_tube": ("bass", 131, 11025, 44100, dict(CLANG, snap_strength=0.0, use_multiband=True, crossover_hz=180.0,
                                                          dry_wet=0.6, output_trim_db=-1.5, delta_listen=True)),
}

# the reference's own audio files (BASELINE configs[0]): name -> path below /root/reference
REF_WAVS = {
    "example_bass": "examples/example_bass.wav",
    "sub_sweep": "tests/data/sub_sweep.wav",
    "wobble_bass": "tests/data/wobble_bass.wav",
    "kick_sub_combo": "tests/data/kick_sub_combo.wav",
    "midrange_growl_like": "tests/data/midrange_growl_like.wav",
}


def make_signal(kind: str, seed: int, n: int, sr: int):
    from quantumdistortion_b200 import synth as signals
    if kind == "bass":
        return signals.bass_clip(seed, n, sr)
    if kind == "noise":
        return signals.noise_clip(seed, n)
    if kind == "loud":
        return signals.loud_clip(seed, n, sr)
    if kind == "tone":
        return signals.tone_clip(seed, n, sr)
    raise KeyError(kind)


# quantize_mode="autotune_v1" (dsp/autotune.py, dsp/pipeline.py:537-601): name -> (kind, seed, n, sr, kwargs)
AT_N = 24000  # 0.5 s @ 48 kHz -> 47 detector frames
AUTOTUNE_CASES = {
    "at_tone_default": ("tone", 0, AT_N, 48000, {}),
    "at_tone_half_strength_441": ("tone", 1, 22050, 44100, {"snap_strength": 0.5, "key": "F", "scale": "major"}),
    "at_bass_growl_nosub": ("bass", 80, AT_N, 48000, dict(GROWL, sub_enabled=False)),
    "at_tone_tube_drywet": ("tone", 2, AT_N, 48000, dict(CLANG, dry_wet=0.6, sub_source="scale_degree",
                                                          sub_scale_degree=4, sub_octave=1, sub_level=0.5,
                                                          air_mix=0.5, output_trim_db=-2.0)),
    "at_noise": ("noise", 81, 9000, 48000, {"sub_source": "manual", "sub_note": "G", "delta_listen": True}),
    "at_no_prequant": ("tone", 3, 9000, 48000, {"pre_quant": False}),
    "at_ragged_short": ("tone", 4, 5003, 48000, {"sub_cut_hz": 0.0, "air_cut_hz": 8000.0}),
}

# avg_cents_offset_from_scale (dsp/analyses.py:53-142): name -> (kind, seed, n, sr, key, scale, kwargs)
ANALYSIS_CASES = {
    "an_bass_dminor": ("bass", 60, N, 48000, "D", "minor", {}),
    "an_noise_top5": ("noise", 61, 6000, 48000, "A", "pentatonic", {"topn_peaks": 5, "min_db": -20.0}),
    "an_loud_1024": ("loud", 62, 9000, 44100, "F#", "dorian", {"frame_length": 1024}),
    "an_quiet": ("bass", 63, 6000, 48000, "C", "major", {"min_db": 40.0}),
}

# Streamlit V2 UI dicts (dsp/pipeline.py:923-1008): name -> (kind, seed, n, sr, rng_seed, config dict, extra kwargs)
UI_CASES = {
    "ui_full": ("loud", 50, N, 48000, 77,
                {"quantization": {"key": "E", "scale": "dorian", "sub_cut_hz": 90.0, "air_cut_hz": 6000.0},
                 "crossover_freq": 250.0,
                 "low_band": {"saturation_amount": 0.5, "mono_strength": 0.6, "output_trim_db": -1.5},
                 "high_band": {"bin_scrambling": 0.0, "phase_dispersal": 0.45, "mag_decimation": 0.7, "output_trim_db": -2.0},
                 "delta_listen": False}, {"snap_strength": 0.8}),
    "ui_defaults_scramble": ("bass", 51, N, 48000, 78, {"high_band": {}, "quantum_fx": {"fundamental_hz": 0.0}}, {}),
    "ui_bitcrush_delta": ("loud", 52, N, 48000, 79,
                          {"high_band": {"bin_scrambling": 0.0, "phase_dispersal": 0.0, "mag_decimation": 0.6},
                           "delta_listen": True}, {}),
}
# UI dicts that keep quantize_mode="autotune_v1" (no high_band / quantum_fx section, so no FX switches the mode):
# the quantization.* sub-layer keys must reach the autotune render (dsp/pipeline.py:964-977)
UI_AT_CASES = {
    "ui_at_sub_keys": ("tone", 53, AT_N, 48000, None,
                       {"quantization": {"mode": "autotune_v1", "key": "G", "scale": "major", "sub_enabled": True,
                                         "sub_source": "scale_degree", "sub_scale_degree": 2, "sub_octave": 1,
                                         "sub_level": 0.6, "sub_cut_hz": 95.0, "air_cut_hz": 7000.0, "air_mix": 0.4},
                        "crossover_freq": 200.0}, {}),
    "ui_at_manual_sub": ("tone", 54, AT_N, 48000, None,
                         {"quantization": {"sub_source": "manual", "sub_note": "A", "sub_level": 0.8},
                          "low_band": {"saturation_amount": 0.2}}, {"snap_strength": 0.7}),
}


# ---------------------------------------------------------------- the reference's own pipeline-level test scenarios
# Every process_audio call the reference's test suite makes at pipeline level (tests/test_pipeline.py,
# test_passthrough_null.py, test_multiband_alignment.py, test_pipeline_multiband_identity.py, test_m12_quantum_fx.py,
# test_quantization_integration.py), with the reference's own signals and arguments -- quantize_mode is left at the
# reference default wherever the reference test leaves it there.  name -> (signal, sr, rng_seed, kwargs, property, cite).
# `property` names the assertion of the reference test, repeated on OUR output by tests/test_gpu_ref_scenarios.py.
def scenario_signal(spec, sr):
    kind = spec[0]
    if kind == "sine":        # (kind, freq, seconds, amp): amp * sin(2 pi f t), t = linspace(0, s, int(sr s), endpoint=False)
        _, f, sec, amp = spec
        t = np.linspace(0.0, sec, int(sr * sec), endpoint=False)
        return (amp * np.sin(2.0 * np.pi * f * t)).astype(np.float32)
    if kind == "sweep_t":     # instantaneous "frequency" f0 + (f1 - f0) t / s inside sin(2 pi f t)  (test_pipeline.py:65-71)
        _, f0, f1, sec, amp = spec
        t = np.linspace(0.0, sec, int(sr * sec), endpoint=False)
        return (amp * np.sin(2.0 * np.pi * (f0 + (f1 - f0) * t / sec) * t)).astype(np.float32)
    if kind == "sweep_phase":  # phase = 2 pi cumsum(f) / sr  (test_passthrough_null.py:33-45)
        _, f0, f1, sec, amp = spec
        t = np.linspace(0.0, sec, int(sr * sec), endpoint=False)
        return (amp * np.sin(2.0 * np.pi * np.cumsum(f0 + (f1 - f0) * t / sec) / sr)).astype(np.float32)
    if kind == "click":       # single-sample spike in the middle (test_multiband_alignment.py:14-20)
        n = int(sr * spec[1])
        x = np.zeros(n, dtype=np.float32)
        x[n // 2] = 1.0
        return x
    if kind == "harmonic":    # sum_h (0.1 / h) sin(2 pi f0 h t), h = 1..5  (test_m12_quantum_fx.py:34-40)
        _, f0, sec = spec
        t = np.linspace(0, sec, int(sr * sec), endpoint=False)
        s = np.zeros_like(t)
        for h in range(1, 6):
            s += (0.1 / h) * np.sin(2 * np.pi * f0 * h * t)
        return s.astype(np.float32)
    if kind == "two_tone":    # 0.2 sin(80 Hz) + 0.2 sin(2 kHz)  (test_pipeline_multiband_identity.py:72-76)
        t = np.linspace(0.0, spec[1], int(sr * spec[1]), endpoint=False)
        return (0.2 * np.sin(2.0 * np.pi * 80.0 * t) + 0.2 * np.sin(2.0 * np.pi * 2000.0 * t)).astype(np.float32)
    if kind == "refwav":      # first `seconds` of one of the reference's WAV files (tests/golden/refwav.npz)
        d = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "refwav.npz"))
        x = d[f"{spec[1]}/x16"].astype(np.float32) / 32768.0
        return x[: int(int(d[f"{spec[1]}/sr"]) * spec[2])]
    raise KeyError(kind)


_NEUTRAL = dict(snap_strength=0.0, pre_quant=False, post_quant=False, distortion_mode="wavefold", limiter_on=False, dry_wet=1.0)
_FXI = dict(use_multiband=True, crossover_hz=300.0, snap_strength=0.5, pre_quant=True, post_quant=False, limiter_on=False)
A4_35_CENTS_SHARP = 440.0 * 2.0 ** (0.35 / 12.0)
REF_SCENARIOS = {
    "taps_shapes": (("sine", 220.0, 0.2, 0.1), 44100, None,
                    dict(snap_strength=0.0, pre_quant=False, post_quant=False, limiter_on=False),
                    "taps", "test_pipeline.py:16-35"),
    "neutral_passthrough": (("sine", 220.0, 0.2, 0.1), 44100, None,
                            dict(key="C", scale="major", snap_strength=0.0, smear=0.0, bin_smoothing=False, pre_quant=False,
                                 post_quant=False, distortion_mode="wavefold",
                                 distortion_params={"fold_amount": 1.0, "bias": 0.0}, limiter_on=False, dry_wet=1.0),
                            "allclose_input_1e-3", "test_pipeline.py:38-62"),
    "fx_baseline": (("sweep_t", 440.0, 880.0, 0.1, 0.1), 44100, None,
                    dict(_FXI, spectral_fx_mode=None, spectral_fx_strength=0.0), "shape", "test_pipeline.py:79-90"),
    "fx_bitcrush": (("sweep_t", 440.0, 880.0, 0.1, 0.1), 44100, None,
                    dict(_FXI, spectral_fx_mode="bitcrush", spectral_fx_strength=0.3), "differs:fx_baseline",
                    "test_pipeline.py:94-113"),
    "fx_phase_dispersal": (("sweep_t", 440.0, 880.0, 0.1, 0.1), 44100, 11,
                           dict(_FXI, spectral_fx_mode="phase_dispersal", spectral_fx_strength=0.3), "differs:fx_baseline",
                           "test_pipeline.py:94-113"),
    "fx_bin_scramble": (("sweep_t", 440.0, 880.0, 0.1, 0.1), 44100, 12,
                        dict(_FXI, spectral_fx_mode="bin_scramble", spectral_fx_strength=0.3), "differs:fx_baseline",
                        "test_pipeline.py:94-113"),
    "passthrough_sweep": (("sweep_phase", 100.0, 2000.0, 0.5, 0.1), 44100, None, dict(passthrough_test=True),
                          "delta_rms_below_-80dB", "test_passthrough_null.py:56-109"),
    "passthrough_sine": (("sine", 440.0, 0.2, 0.1), 44100, None, dict(passthrough_test=True),
                         "delta_rms_below_-80dB", "test_passthrough_null.py:112-150"),
    "click_single": (("click", 0.1), 44100, None,
                     dict(_NEUTRAL, distortion_params={"fold_amount": 1.0, "bias": 0.0}, use_multiband=False),
                     "peak_above_0.1", "test_multiband_alignment.py:22-33"),
    "click_multi": (("click", 0.1), 44100, None,
                    dict(_NEUTRAL, distortion_params={"fold_amount": 1.0, "bias": 0.0}, use_multiband=True, crossover_hz=300.0,
                         lowband_drive=0.0),
                    "argmax_within_50_of:click_single", "test_multiband_alignment.py:35-63"),
    **{f"click_xover_{int(c)}": (("click", 0.1), 44100, None,
                                 dict(_NEUTRAL, distortion_params={"fold_amount": 1.0}, use_multiband=True, crossover_hz=c,
                                      lowband_drive=0.0),
                                 "argmax_within_1200_of_click", "test_multiband_alignment.py:80-119")
       for c in (200.0, 500.0, 1000.0)},
    "wobble_multiband": (("refwav", "wobble_bass", 0.5), 48000, None,   # the file's own rate (load_audio)
                         dict(snap_strength=0.5, pre_quant=True, post_quant=True, distortion_mode="wavefold",
                              distortion_params={"fold_amount": 1.0, "bias": 0.0}, limiter_on=False, dry_wet=1.0,
                              use_multiband=True, crossover_hz=300.0, lowband_drive=1.0),
                         "taps", "test_pipeline_multiband_identity.py:9-64"),
    **{f"two_tone_xover_{int(c)}": (("two_tone", 0.3), 44100, None,
                                    dict(snap_strength=0.3, pre_quant=True, post_quant=False, distortion_mode="wavefold",
                                         distortion_params={"fold_amount": 1.0}, limiter_on=False, dry_wet=1.0,
                                         use_multiband=True, crossover_hz=c),
                                    "taps", "test_pipeline_multiband_identity.py:67-103")
       for c in (200.0, 500.0, 1000.0)},
    "mb_passthrough_null": (("sine", 200.0, 0.5, 0.1), 44100, None,
                            dict(passthrough_test=True, use_multiband=True, crossover_hz=300.0, lowband_drive=1.0),
                            "delta_rms_below_-10dB_and_audible", "test_m12_quantum_fx.py:57-88"),
    "freeze_on": (("harmonic", 110.0, 0.5), 44100, None,
                  dict(spectral_freeze=True, snap_strength=0.0, pre_quant=True, post_quant=False), "shape",
                  "test_m12_quantum_fx.py:96-103"),
    "freeze_off": (("harmonic", 110.0, 0.5), 44100, None,
                   dict(spectral_freeze=False, snap_strength=0.0, pre_quant=True, post_quant=False), "shape",
                   "test_m12_quantum_fx.py:104-115"),
    "freeze_multiband": (("sine", 440.0, 0.3, 0.1), 44100, None, dict(use_multiband=True, spectral_freeze=True), "shape",
                         "test_m12_quantum_fx.py:119-127"),
    "formant_multiband": (("sine", 440.0, 0.3, 0.1), 44100, None, dict(formant_shift=3.0, use_multiband=True), "shape",
                          "test_m12_quantum_fx.py:151-159"),
    "formant_zero": (("harmonic", 110.0, 0.3), 44100, None, dict(formant_shift=0.0), "shape", "test_m12_quantum_fx.py:163-164"),
    "formant_six": (("harmonic", 110.0, 0.3), 44100, None, dict(formant_shift=6.0), "differs_1e-6:formant_zero",
                    "test_m12_quantum_fx.py:165-167"),
    "harmonic_lock": (("harmonic", 110.0, 0.3), 44100, None, dict(harmonic_lock_hz=110.0), "shape",
                      "test_m12_quantum_fx.py:198-205"),
    "delta_off": (("sine", 440.0, 0.3, 0.1), 44100, None, dict(delta_listen=False), "shape", "test_m12_quantum_fx.py:237"),
    "delta_on": (("sine", 440.0, 0.3, 0.1), 44100, None, dict(delta_listen=True), "is_input_minus:delta_off",
                 "test_m12_quantum_fx.py:240-250"),
    "autotune_detuned_a4": (("sine", A4_35_CENTS_SHARP, 1.0, 0.2), 48000, None,
                            dict(key="A", scale="minor", quantize_mode="autotune_v1", snap_strength=1.0, smear=0.0,
                                 bin_smoothing=False, pre_quant=True, post_quant=False, distortion_mode="wavefold",
                                 distortion_params={"fold_amount": 1.0, "bias": 0.0, "drive": 1.0, "warmth": 0.5},
                                 limiter_on=False, dry_wet=1.0, sub_enabled=False),
                            "dominant_freq_moves_to_440", "test_quantization_integration.py:46-74"),
}

# Tolerance of the final output where the REFERENCE ITSELF is ill-conditioned (taps before the ill-conditioned stage keep
# 1e-4).  formant_six: the second quantised pass takes log(max(|X|, 1e-12)) of every bin of the wavefolded first-pass
# output, whose inter-harmonic bins hold nothing but that signal's float32 rounding noise -- moving the reference's own
# pass-2 input by 1e-9 (a seventh of its float32 ulp) moves the reference's output by 2e-4
# (tests/test_oracle_ref_scenarios.py::test_reference_formant_second_pass_is_ill_conditioned), so a single differently
# rounded sample of the first pass is enough.  The float64 kernels reproduce each pass to 7.5e-9 (same test file, emulator).
REF_SCENARIO_Y_TOL = {"formant_six": 1e-3}


def _rms_db(v):
    r = float(np.sqrt(np.mean(np.asarray(v, dtype=np.float64) ** 2)))
    return -np.inf if r == 0.0 else 20.0 * np.log10(r)


def _dominant_freq(a, sr, lo=80.0, hi=1200.0, t0=0.25, t1=0.85):
    seg = np.asarray(a[int(t0 * sr): min(len(a), int(t1 * sr))], dtype=np.float64)
    spec = np.abs(np.fft.rfft(seg * np.hanning(len(seg))))
    fr = np.fft.rfftfreq(len(seg), d=1.0 / sr)
    m = (fr >= lo) & (fr <= hi)
    return float(fr[m][int(np.argmax(spec[m]))])


def check_scenario_property(name, x, y, other_output):
    """The assertion the reference's own test makes on this scenario, on the output `y` of any implementation;
    `other_output(name)` returns the same implementation's output of another scenario."""
    spec, sr, _seed, _kw, prop, cite = REF_SCENARIOS[name]
    what = f"{name} ({cite}): {prop}"
    assert y.shape == x.shape and y.dtype == np.float32, what
    assert np.all(np.isfinite(y)), what
    arg = prop.split(":", 1)[1] if ":" in prop else None
    if prop == "allclose_input_1e-3":
        assert np.allclose(y, x, atol=1e-3), what
    elif prop == "delta_rms_below_-80dB":
        assert _rms_db(y - x) < -80.0, what
    elif prop == "delta_rms_below_-10dB_and_audible":
        assert _rms_db(x - y) < -10.0 and _rms_db(y) > -60.0, what
    elif prop == "peak_above_0.1":
        assert np.max(np.abs(y)) > 0.1, what
    elif prop.startswith("argmax_within_50_of"):
        o = other_output(arg)
        assert abs(int(np.argmax(np.abs(y))) - int(np.argmax(np.abs(o)))) < 50 and np.max(np.abs(y)) > 0.1, what
    elif prop == "argmax_within_1200_of_click":
        assert abs(int(np.argmax(np.abs(y))) - len(x) // 2) < 1200, what
    elif prop.startswith("differs_1e-6"):
        assert not np.allclose(other_output(arg), y, atol=1e-6), what
    elif prop.startswith("differs"):
        assert float(np.sqrt(np.mean((y - other_output(arg)) ** 2))) > 0.0, what
    elif prop.startswith("is_input_minus"):
        np.testing.assert_allclose(y, x - other_output(arg), atol=1e-6, err_msg=what)
    elif prop == "dominant_freq_moves_to_440":
        fi, fo = _dominant_freq(x, sr), _dominant_freq(y, sr)
        assert abs(fo - 440.0) < abs(fi - 440.0) and abs(fo - 440.0) < 6.0, what
    else:
        assert prop in ("taps", "shape"), prop


# ---------------------------------------------------------------- the reference's scripts as scenarios
# The process_audio / process_file_to_file calls of the reference's scripts/ on the first second of its own WAV files.
# SCRIPT_SCENARIOS: direct process_audio calls, name -> (wav, seconds, rng_seed, kwargs, cite).
# HARNESS_SCENARIOS: file-to-file renders, name -> (wav, seconds, rng_seed, preset, extra_params, cite); compared as PCM16.
_DP3 = {"fold_amount": 3.0, "bias": 0.0, "drive": 1.0, "warmth": 0.5}
_PRESET_ARGS = ("key", "scale", "snap_strength", "smear", "bin_smoothing", "pre_quant", "post_quant", "distortion_mode",
                "distortion_params", "limiter_on", "limiter_ceiling_db", "dry_wet")   # scripts/render_preset.py:50-81


def _preset_kwargs(name):
    from quantumdistortion_b200.presets import get_preset
    p = get_preset(name)
    return {k: p[k] for k in _PRESET_ARGS}


SCRIPT_SCENARIOS = {
    "validate_metrics_main": ("midrange_growl_like", 1.0, None,
                              dict(key="D", scale="minor", snap_strength=0.8, smear=0.4, bin_smoothing=True, pre_quant=True,
                                   post_quant=True, distortion_mode="wavefold", distortion_params=_DP3, limiter_on=True,
                                   limiter_ceiling_db=-1.0, dry_wet=1.0), "scripts/validate_dsp_metrics.py:59-74"),
    "validate_metrics_quantizer_only": ("midrange_growl_like", 1.0, None,
                                        dict(key="D", scale="minor", snap_strength=1.0, smear=0.0, bin_smoothing=False,
                                             pre_quant=True, post_quant=True, distortion_mode="wavefold",
                                             distortion_params={"fold_amount": 1.0, "bias": 0.0, "drive": 1.0, "warmth": 0.5},
                                             limiter_on=False, limiter_ceiling_db=-1.0, dry_wet=1.0),
                                        "scripts/validate_dsp_metrics.py:92-107"),
    "profile_pipeline": ("kick_sub_combo", 1.0, None,
                         dict(key="C", scale="minor", snap_strength=0.8, smear=0.3, bin_smoothing=True, pre_quant=True,
                              post_quant=True, distortion_mode="wavefold", distortion_params=_DP3, limiter_on=True,
                              limiter_ceiling_db=-1.0, dry_wet=1.0), "scripts/profile_pipeline.py:35-50"),
    **{f"render_preset_{n.split()[0].lower()}": ("wobble_bass", 1.0, None, n, "scripts/render_preset.py:67-82")
       for n in ("Chordal Noise Wash", "Controlled Dubstep Growl", "Perc To Tonal Clang", "Subtle Tube Glue")},
}


def script_scenario_kwargs(name):
    kw = SCRIPT_SCENARIOS[name][3]
    return _preset_kwargs(kw) if isinstance(kw, str) else dict(kw)


_MB = {"use_multiband": True, "crossover_hz": 300.0}
HARNESS_SCENARIOS = {
    "qrs_single": ("sub_sweep", 1.0, None, None, {"use_multiband": False}, "scripts/quick_regression_suite.py:148-153"),
    "qrs_multiband_baseline": ("sub_sweep", 1.0, None, None, dict(_MB, spectral_fx_mode=None, spectral_fx_strength=0.0),
                               "scripts/quick_regression_suite.py:158-168"),
    "qrs_single_growl_preset": ("wobble_bass", 1.0, None, "Controlled Dubstep Growl", {"use_multiband": False},
                                "scripts/quick_regression_suite.py:148-153 --preset"),
    **{f"qrs_fxpreset_{p}": ("wobble_bass", 1.0, 300 + i, None, ("fx_preset", p), "scripts/quick_regression_suite.py:198-209")
       for i, p in enumerate(("sub_safe_glue", "digital_growl", "laser_zap", "grainy_top"))},
    **{f"qrs_fx_{m}": ("kick_sub_combo", 1.0, 400 + i, None, dict(_MB, spectral_fx_mode=m, spectral_fx_strength=0.5),
                       "scripts/quick_regression_suite.py:237-247")
       for i, m in enumerate(("bitcrush", "phase_dispersal", "bin_scramble"))},
    "harness_extra_params": ("sub_sweep", 1.0, None, None,
                             {"snap_strength": 0.0, "pre_quant": False, "post_quant": False, "limiter_on": False, "dry_wet": 1.0},
                             "tests/test_harness_smoke.py:50-70"),
}


def harness_extra_params(name):
    ep = HARNESS_SCENARIOS[name][4]
    if isinstance(ep, tuple):   # a spectral-FX preset applied like scripts/quick_regression_suite.py:65-84, 198-209
        from quantumdistortion_b200.presets import spectral_fx_preset_kwargs
        return dict(_MB, **spectral_fx_preset_kwargs(ep[1]))
    return dict(ep)


def flatness_interval(frame, rtol: float = 1e-4):
    """Where a float32 FFT may put the spectral flatness of one detector frame (dsp/autotune.py:130-137, symmetric
    Hann): every bin of a float32 FFT of length N may move by up to delta = eps32 log2(N) ||frame * window||_2, so the
    flatness lies between that of max(|X| - delta, 0) and that of |X| + delta (float64 |X|), widened by rtol for the
    float32 logarithm and sums.  On a frame whose spectrum sits well above delta everywhere this is rtol itself; on a
    band-limited, tonal frame (the detector band above 3 kHz) the stopband bins hold only the FFT's rounding noise and
    the flatness is that noise's: a float32 FFT moves it by up to 160 % (4.6e-6 -> 1.1e-5 measured on the B200)."""
    frame = np.asarray(frame, dtype=np.float64)
    xw = frame * np.hanning(len(frame))
    mag = np.abs(np.fft.rfft(xw))
    delta = float(np.finfo(np.float32).eps) * np.log2(len(frame)) * float(np.linalg.norm(xw))

    def flat(m):
        spec = m + 1e-8
        ari = float(np.mean(spec))
        return 1.0 if ari <= 1e-8 else float(np.exp(np.mean(np.log(spec)))) / ari
    return flat(np.maximum(mag - delta, 0.0)) * (1.0 - rtol), flat(mag + delta) * (1.0 + rtol)
