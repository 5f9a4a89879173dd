"""CPU: every autotune_v1 kernel after the band split, single-stepped through tests/emu/cuda_emu.h and compared with
oracle/qd_autotune.py fed the SAME input the kernel got, at the tightest bound its arithmetic allows.  The whole-render
checks compare at 1e-4; a wrong value at an edge (the clamped last frame centre, the last lag of a ballot group, the
latency trim, a short clip, a silent gap) moves a few samples by less than that and shows up only here.

  frame stats   at_frame_stats_kernel<2048> vs frame_features: rms rtol 1e-5, flatness rtol 1e-4 where every bin lies
                above the float32 FFT's rounding (qd_cases.flatness_interval on a band-limited frame), flag exact
  YIN pick      at_yin_pick_kernel vs yin_pick on hand-built difference functions: pitch and confidence exact
  note hold     at_target_kernel + at_hold_kernel vs note_hold_ratios: 1e-12 relative
  shifter       at_tap_sums / at_tap_scan / at_shift_kernel vs granular_pitch_shift: ratio track and flag bit-identical,
                corrected within 1 float32 ulp (the Hann weight's cos)
  envelope      at_env_kernel / at_env_seg_kernel vs envelope_follow: bit-identical, env_max too
  mix           at_mix_kernel vs sub_layer + the apply_autotune_v1 sum: layer within 2 ulp of sub_level (sinf), sum exact
"""
import math
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

import qd_cases
from oracle import qd_autotune as at
from oracle import qd_oracle as orc
from test_emu_ragged_autotune import emu_at, TIMEOUT  # noqa: F401  (fixture)

SR = 48000
CFG = at.AutotuneConfig()
FS, HOP, HALF = 4096, 512, 2048
MIN_FREQ, MAX_FREQ = max(60.0, CFG.detector_low_hz * 0.65), max(CFG.detector_high_hz, 400.0)
MAX_TAU = min(int(SR / MIN_FREQ), max(2, FS // 2 - 1))     # 671
MIN_TAU = max(2, int(SR / MAX_FREQ))                       # 16
STRIDE = (MAX_TAU + 2) & ~1
MAX_DELAY, BUF = 1024, 4096


def _run(*cmd):
    subprocess.run([str(c) for c in cmd], check=True, timeout=TIMEOUT, stdout=subprocess.DEVNULL)


def _f(v):
    """A number for the driver's command line, exact through strtod."""
    return repr(float(v))


def _ulps(a, b):
    """Distance in float32 units in the last place, elementwise."""
    def key(v):
        i = np.asarray(v, dtype=np.float32).view(np.int32).astype(np.int64)
        return np.where(i < 0, -(i & 0x7FFFFFFF), i)
    return np.abs(key(a) - key(b))


def _frames(x):
    """The zero-padded detector frames of frame_features."""
    out = []
    for s in range(0, len(x), HOP):
        fr = x[s:s + FS]
        out.append(np.pad(fr, (0, FS - len(fr))) if len(fr) < FS else fr)
    return out


# ------------------------------------------------------------------------------------------------ frame stats
def _signal(kind, n, seed):
    rng = np.random.default_rng(seed)
    t = np.arange(n) / SR
    if kind == "silent":
        return np.zeros(n, np.float32)
    if kind == "tiny":          # below the 1e-6 silence threshold
        return (9e-7 * np.clip(rng.standard_normal(n), -1, 1)).astype(np.float32)
    if kind == "tonal":         # a harmonic tone over a -60 dB floor: every bin sits above the float32 FFT's noise
        x = sum(0.4 / k * np.sin(2 * np.pi * 196.0 * k * t + k) for k in range(1, 6))
        return (x + 1e-3 * rng.standard_normal(n)).astype(np.float32)
    return (0.3 * rng.standard_normal(n)).astype(np.float32)


def _stats(exe, d, x):
    x.astype(np.float32).tofile(os.path.join(d, "x"))
    _run(exe, "stats", HOP, MIN_TAU, MAX_TAU, os.path.join(d, "x"), "-", "-", os.path.join(d, "feat"))
    return np.fromfile(os.path.join(d, "feat")).reshape(-1, 4)


@pytest.mark.parametrize("n", [1, 511, 512, 4095, 4096, 4097, 20000])
def test_emu_frame_stats_vs_oracle(emu_at, n):
    with tempfile.TemporaryDirectory() as d:
        for i, kind in enumerate(("silent", "tiny", "tonal", "noise", "detector band")):
            if kind == "detector band":
                if n <= 15:
                    continue
                x = at.detector_sidechain(_signal("tonal", n, 100 * n + i), SR, CFG.detector_low_hz, CFG.detector_high_hz)
            else:
                x = _signal(kind, n, 100 * n + i)
            got = _stats(emu_at, d, x)
            frames = _frames(x)
            assert got.shape == (len(frames), 4)
            rms = np.array([float(np.sqrt(np.mean(fr * fr))) for fr in frames])
            flat = np.array([at.spectral_flatness(fr) for fr in frames])
            loud = np.array([not (np.max(np.abs(fr.astype(np.float64))) < 1e-6) for fr in frames])
            assert np.allclose(got[:, 0], rms, rtol=1e-5, atol=0.0), (kind, n)
            if kind == "detector band":   # band-limited and tonal: the stopband bins hold the float32 FFT's rounding
                lo, hi = np.array([qd_cases.flatness_interval(fr) for fr in frames]).T
                assert ((lo <= got[:, 1]) & (got[:, 1] <= hi)).all(), (kind, n)
            else:                         # every bin above the float32 FFT's rounding: the flatness to 1e-4
                assert np.allclose(got[:, 1], flat, rtol=1e-4, atol=0.0), (kind, n, np.max(np.abs(got[:, 1] / flat - 1)))
            assert np.array_equal(got[:, 2], loud.astype(np.float64)), (kind, n)
            assert (got[:, 3] == 0.0).all()


# ------------------------------------------------------------------------------------------------ YIN pick
def _cmnd(diff):
    """The oracle's sequential cumulative-mean normalisation (yin_tables)."""
    cm = np.ones(MAX_TAU + 1)
    run = 0.0
    for tau in range(1, MAX_TAU + 1):
        run += diff[tau]
        if run > 0.0:
            cm[tau] = diff[tau] * tau / run
    return cm


def _pick(exe, d, diffs, flags, min_freq=MIN_FREQ, max_freq=MAX_FREQ):
    diff = np.full((len(diffs), STRIDE), np.nan)
    for r, v in enumerate(diffs):
        diff[r, :MAX_TAU + 1] = v
        diff[r, 0] = np.nan       # lag 0 is never read
    feat = np.zeros((len(diffs), 4))
    feat[:, 2] = flags
    feat[:, 3] = -5.0
    diff.tofile(os.path.join(d, "diff"))
    feat.tofile(os.path.join(d, "feat"))
    _run(exe, "pick", SR, MIN_TAU, MAX_TAU, _f(min_freq), _f(max_freq), _f(0.15), os.path.join(d, "diff"),
         os.path.join(d, "feat"), os.path.join(d, "out"))
    return np.fromfile(os.path.join(d, "out")).reshape(-1, 4)


def _dips(base=1000.0, **lags):
    v = np.full(MAX_TAU + 1, base)
    for t, val in lags.items():
        v[int(t[1:])] = val
    return v


def _hand_built():
    """Integer-valued difference functions, so that any summation order gives the same running sums and the kernel's
    normalised difference equals the oracle's bit for bit: then the pick itself must agree exactly."""
    g31 = MIN_TAU + 32 + 31                                   # lane 31 of the second ballot group
    cases = {
        "dip at min_tau": _dips(**{f"t{MIN_TAU}": 10.0}),
        "dip at min_tau + 1, walk": _dips(**{f"t{MIN_TAU + 1}": 100.0, f"t{MIN_TAU + 2}": 40.0}),
        "lane 31, walk into the next group": _dips(**{f"t{g31}": 100.0, f"t{g31 + 1}": 60.0, f"t{g31 + 2}": 30.0}),
        "lane 0 of a group after a miss": _dips(**{f"t{g31 + 1}": 50.0}),
        "dip only at max_tau": _dips(**{f"t{MAX_TAU}": 5.0}),
        "walk ends at max_tau": _dips(**{f"t{MAX_TAU - 2}": 60.0, f"t{MAX_TAU - 1}": 30.0, f"t{MAX_TAU}": 10.0}),
        "flat bottom stops the walk": _dips(**{"t200": 0.0, "t201": 0.0, "t202": 0.0}),
        "never below the threshold": _dips(),
        "zero leading lags (running sum 0)": np.concatenate([np.zeros(40), _dips(**{"t300": 20.0})[40:]]),
    }
    # |den| <= 1e-12: cm[est - 1] ~ 1e-13 above cm[est] = cm[est + 1] = 0 (no parabola), and the same just above it
    big = _dips(base=1e13, t150=1.0, t151=0.0, t152=0.0)
    cases["|den| <= 1e-12"] = big
    cases["|den| just above 1e-12"] = _dips(base=1e13, t150=10.0, t151=0.0, t152=0.0)
    rng = np.random.default_rng(7)
    for k in range(24):                                       # random integer difference functions with a few dips
        v = rng.integers(200, 5000, MAX_TAU + 1).astype(np.float64)
        for t in rng.integers(MIN_TAU - 4, MAX_TAU + 1, rng.integers(0, 6)):
            v[t] = float(rng.integers(0, 60))
        cases[f"random {k}"] = v
    return cases


def _oracle_pick(v, min_freq=MIN_FREQ, max_freq=MAX_FREQ):
    return at.yin_pick(_cmnd(v), MIN_TAU, MAX_TAU, SR, min_freq, max_freq, 0.15)


def test_emu_yin_pick_hand_built(emu_at):
    cases = _hand_built()
    names = list(cases)
    for v in cases.values():
        assert np.array_equal(np.cumsum(v[1:]), np.cumsum(v[1:].astype(np.int64)).astype(np.float64))   # exact sums
    with tempfile.TemporaryDirectory() as d:
        for flag in (1.0, 0.0):
            got = _pick(emu_at, d, [cases[k] for k in names], [flag] * len(names))
            voiced = 0
            for r, name in enumerate(names):
                p, c = _oracle_pick(cases[name]) if flag else (0.0, 0.0)
                voiced += p > 0
                assert (got[r, 2] > 0) == (p > 0), name
                assert abs(got[r, 2] - p) <= 1e-12 * p, (name, got[r, 2], p)
                assert abs(got[r, 3] - c) <= 1e-12, (name, got[r, 3], c)
            assert voiced >= (len(names) // 2 if flag else 0)
        # the sharp dips resolve where they were built (the cases above are what they say they are)
        e = {k: _oracle_pick(v) for k, v in cases.items()}
        assert e["dip at min_tau"][0] == SR / MIN_TAU and e["dip only at max_tau"][0] == SR / MAX_TAU
        assert e["never below the threshold"] == (0.0, 0.0)
        assert e["flat bottom stops the walk"][0] == SR / 200.5
        assert e["|den| <= 1e-12"][0] == SR / 151 and e["|den| just above 1e-12"][0] != SR / 151


def test_emu_yin_pick_refined_pitch_at_the_range_edges(emu_at):
    """The range check uses the refined pitch: just inside / just outside [min_freq, max_freq] on both sides."""
    v = _dips(t200=100.0, t201=20.0, t202=60.0)
    p, _ = _oracle_pick(v, 1.0, 1e9)
    assert p != SR / 201 and p > 0
    lo_out, hi_out = np.nextafter(p, np.inf), np.nextafter(p, -np.inf)
    with tempfile.TemporaryDirectory() as d:
        for fmin, fmax in ((p, 1e9), (lo_out, 1e9), (1.0, p), (1.0, hi_out)):
            got = _pick(emu_at, d, [v], [1.0], fmin, fmax)
            ref = _oracle_pick(v, fmin, fmax)
            assert (got[0, 2], got[0, 3]) == ref, (fmin, fmax)
            assert (ref[0] > 0) == (fmin <= p <= fmax)


def test_emu_detector_real_frames_vs_detect_pitch_yin(emu_at):
    """stats + the sliding difference function + pick on real detector frames against detect_pitch_yin: the bar of
    DESIGN section 9 (pitch 1e-9 relative; the difference function sums in another order than the oracle's np.dot)."""
    n = 12000
    t = np.arange(n) / SR
    f0 = 220.0 * 2.0 ** (np.sin(2 * np.pi * 3 * t) / 12)       # vibrato
    x = (0.5 * np.sin(2 * np.pi * np.cumsum(f0) / SR) + 0.2 * np.sin(4 * np.pi * np.cumsum(f0) / SR)).astype(np.float32)
    x[5000:5200] = 0.0
    x[-1500:] *= 1e-7                                           # a quiet tail
    with tempfile.TemporaryDirectory() as d:
        feat = _stats(emu_at, d, x)
        _run(emu_at, "yin", FS, HOP, MAX_TAU, 42, os.path.join(d, "x"), "-", "-", os.path.join(d, "diff"))
        feat.tofile(os.path.join(d, "feat"))
        _run(emu_at, "pick", SR, MIN_TAU, MAX_TAU, _f(MIN_FREQ), _f(MAX_FREQ), _f(0.15), os.path.join(d, "diff"),
             os.path.join(d, "feat"), os.path.join(d, "out"))
        got = np.fromfile(os.path.join(d, "out")).reshape(-1, 4)
    ref = np.array([at.detect_pitch_yin(fr, SR, MIN_FREQ, MAX_FREQ) for fr in _frames(x)])
    assert np.array_equal(got[:, 2] > 0, ref[:, 0] > 0)
    assert (ref[:, 0] > 0).sum() >= len(ref) // 2
    assert np.allclose(got[:, 2], ref[:, 0], rtol=1e-9, atol=0.0)
    assert np.allclose(got[:, 3], ref[:, 1], rtol=0.0, atol=1e-9)


# ------------------------------------------------------------------------------------------------ note hold
SCALES = [("D", "minor"), ("C", "major"), ("F#", "dorian"), ("A#", "harmonic_minor"), ("E", "pentatonic")]


def _scale(key, scale):
    return orc.note_name_to_pitch_class(key), orc.SCALE_INTERVALS[scale]


def _feature_sequence(seed, frames, cfg):
    """Seeded features that walk through every branch of the state machine: held notes with a few cents of jitter,
    note changes that confirm after confirm_frames, blips that a third note or a return resets, candidates more than
    20 cents apart, gaps inside and beyond release_frames, each voiced gate failing alone, pitches far enough from
    the held note for the 0.5 / 2.0 clamp."""
    rng = np.random.default_rng(seed)
    rms = np.full(frames, 0.1)
    flat = np.full(frames, 0.2)
    conf = np.full(frames, 0.9)
    pitch = np.zeros(frames)
    note = 220.0
    i = 0
    while i < frames:
        ev = rng.integers(0, 10)
        m = int(rng.integers(1, 6))
        for j in range(i, min(frames, i + m)):
            cents = rng.uniform(-15, 15)
            if ev == 0:                                    # a new note, long enough to confirm (or not)
                note = float(rng.uniform(70, 1400)) if j == i else note
            elif ev == 1 and j == i:                       # a step of 45-60 cents: a candidate > 20 cents from the last
                note = note * 2 ** (rng.choice([-1, 1]) * rng.uniform(45, 60) / 1200)
            elif ev == 2:                                  # unvoiced
                pitch[j] = 0.0
                continue
            elif ev == 3:                                  # one gate fails
                which = rng.integers(0, 3)
                if which == 0:
                    rms[j] = cfg.detector_rms_threshold * rng.uniform(0.5, 0.999)
                elif which == 1:
                    flat[j] = cfg.detector_flatness_threshold + rng.uniform(1e-6, 0.3)
                else:
                    conf[j] = cfg.detector_min_confidence * rng.uniform(0.5, 0.999)
            elif ev == 4:                                  # far from the held note: the clamp
                pitch[j] = note * rng.choice([0.3, 0.45, 2.2, 3.5])
                continue
            elif ev == 5:                                  # exactly at the gates
                rms[j], flat[j], conf[j] = cfg.detector_rms_threshold, cfg.detector_flatness_threshold, cfg.detector_min_confidence
            pitch[j] = note * 2 ** (cents / 1200)
        i += m
    return rms, flat, pitch, conf


def _hold(exe, d, feats, n, cfg, starts="-", lengths="-"):
    root, iv = _scale(cfg.key, cfg.scale)
    feats.tofile(os.path.join(d, "feat"))
    _run(exe, "hold", n, HOP, root, ",".join(str(v) for v in iv), _f(cfg.strength), _f(cfg.detector_rms_threshold),
         _f(cfg.detector_flatness_threshold), _f(cfg.detector_min_confidence), _f(cfg.note_change_cents),
         cfg.note_confirm_frames, cfg.note_release_frames, os.path.join(d, "feat"), starts, lengths,
         os.path.join(d, "ratio"))
    return np.fromfile(os.path.join(d, "ratio"))


def _hold_lines_hit(fn):
    """Line numbers of note_hold_ratios that ran during fn() (the test asserts that every branch did)."""
    code = at.note_hold_ratios.__code__
    hit = set()

    def tracer(frame, event, arg):
        if frame.f_code is code:
            if event == "line":
                hit.add(frame.f_lineno)
            return tracer
        return None
    old = sys.gettrace()
    sys.settrace(tracer)
    try:
        fn()
    finally:
        sys.settrace(old)
    return hit, code


def test_emu_note_hold_vs_oracle(emu_at):
    import dis
    runs = []
    with tempfile.TemporaryDirectory() as d:
        for k, (key, scale) in enumerate(SCALES):
            for strength in (1.0, 0.6):
                cfg = at.AutotuneConfig(key=key, scale=scale, strength=strength)
                frames = 700
                rms, flat, pitch, conf = _feature_sequence(31 * k + int(10 * strength), frames, cfg)
                feats = np.stack([rms, flat, pitch, conf], axis=1)
                n = frames * HOP - 100
                got = _hold(emu_at, d, feats, n, cfg)
                runs.append((got, (rms, flat, pitch, conf), cfg))

    def oracle_all():
        return [at.note_hold_ratios(*f, cfg) for _, f, cfg in runs]
    hit, code = _hold_lines_hit(oracle_all)
    refs = oracle_all()
    body = {ln for _, ln in dis.findlinestarts(code) if ln is not None and ln > code.co_firstlineno + 1}
    assert body - hit == set(), f"note_hold_ratios lines never reached: {sorted(body - hit)}"
    clamped = 0
    for (got, _, cfg), ref in zip(runs, refs):
        assert got.shape == ref.shape
        assert np.allclose(got, ref, rtol=1e-12, atol=0.0), (cfg.key, cfg.scale, cfg.strength)
        clamped += int(np.sum((ref == 0.5) | (ref == 2.0)))
    assert clamped > 0


# ------------------------------------------------------------------------------------------------ shifter
def _ratios_for(kind, frames, rng):
    k = np.arange(frames)
    if kind == "glide up":
        return 0.5 + 1.5 * k / max(1, frames - 1)
    if kind == "glide down":
        return 2.0 - 1.5 * k / max(1, frames - 1)
    if kind == "pinned":
        return np.where(k % 6 < 3, 0.5, 2.0) * np.where(k % 4 == 0, 1.2, 1.0)     # 0.5, 0.6, 2.0, 2.4: the clamp
    if kind == "flat":
        return 1.0 + rng.uniform(-9e-4, 9e-4, frames)
    if kind == "just not flat":
        r = 1.0 + rng.uniform(-9e-4, 9e-4, frames)
        r[frames // 2] = 1.0 + 1.02e-3
        return r
    return np.exp(rng.uniform(np.log(0.55), np.log(1.9), frames))                     # random per frame


def _body(n, seed):
    rng = np.random.default_rng(seed)
    t = np.arange(n)
    return (0.4 * np.sin(2 * np.pi * t / 97.0) + 0.2 * rng.standard_normal(n)).astype(np.float32)


def _shift(exe, d, body, ratios, hop=HOP, half=HALF, starts="-", lengths="-"):
    body.tofile(os.path.join(d, "body"))
    np.asarray(ratios, np.float64).tofile(os.path.join(d, "ratio"))
    _run(exe, "shift", hop, half, MAX_DELAY, BUF, os.path.join(d, "body"), starts, lengths, os.path.join(d, "ratio"),
         os.path.join(d, "out"), os.path.join(d, "track"), os.path.join(d, "flag"))
    return (np.fromfile(os.path.join(d, "out"), np.float32), np.fromfile(os.path.join(d, "track"), np.float32),
            np.fromfile(os.path.join(d, "flag"), np.int32))


def _shift_oracle(body, ratios, hop=HOP, half=HALF):
    n = len(body)
    centers = np.minimum(n - 1, np.arange(len(ratios)) * hop + half).astype(np.float64)
    track = np.interp(np.arange(n, dtype=np.float64), centers, ratios).astype(np.float32)
    flat = int(n == 0 or np.allclose(track, 1.0, atol=1e-3))
    return at.granular_pitch_shift(body, track, 1024, 4096), track, flat


SHIFT_CASES = [(1, "random"), (511, "random"), (512, "glide up"), (513, "glide down"), (2049, "pinned"),
               (4095, "random"), (4097, "glide up"), (8191, "pinned"), (8193, "random"), (6000, "flat"),
               (6000, "just not flat"), (7000, "random"), (7001, "pinned"), (40000, "glide down"),
               (104001, "glide up")]


@pytest.mark.parametrize("n,kind", SHIFT_CASES)
def test_emu_shifter_vs_oracle(emu_at, n, kind):
    """Glides wrap the taps many times both ways; 2049 samples clamp the first centre; n = 7000 / 7001 put the last
    four / five centres on the clamped sample n - 1 with different ratios (r_last); 512 / 513 sit at the latency trim."""
    rng = np.random.default_rng(n)
    frames = -(-n // HOP)
    ratios = _ratios_for(kind, frames, rng)
    body = _body(n, n + 1)
    with tempfile.TemporaryDirectory() as d:
        out, track, flag = _shift(emu_at, d, body, ratios)
    ref, rtrack, rflat = _shift_oracle(body, ratios)
    assert np.array_equal(track, rtrack)
    assert int(flag[0]) == rflat
    assert rflat == (kind == "flat")
    u = _ulps(out, ref)
    assert u.max(initial=0) <= 1, (n, kind, int(u.max()))
    print(f"shifter n={n} {kind}: {int(np.count_nonzero(u))} of {n} samples differ (max {int(u.max(initial=0))} ulp)")


def test_emu_shifter_unaligned_interp_path(emu_at):
    """hop 480, half 2000: not multiples of the 512-sample tile, so every sample takes at_ratio_at."""
    n, hop, half = 9000, 480, 2000
    rng = np.random.default_rng(3)
    ratios = _ratios_for("random", -(-n // hop), rng)
    body = _body(n, 4)
    with tempfile.TemporaryDirectory() as d:
        out, track, flag = _shift(emu_at, d, body, ratios, hop, half)
    ref, rtrack, rflat = _shift_oracle(body, ratios, hop, half)
    assert np.array_equal(track, rtrack) and int(flag[0]) == rflat == 0
    assert _ulps(out, ref).max() <= 1


# ------------------------------------------------------------------------------------------------ envelope
def env_coeffs(sr, attack_ms=8.0, release_ms=90.0):
    att = float(np.float32(np.exp(-1.0 / max(1.0, attack_ms * 0.001 * sr))))
    rel = float(np.float32(np.exp(-1.0 / max(1.0, release_ms * 0.001 * sr))))
    return att, rel


def env_halo(att, rel, tile):
    """at_render: halo with max(att, rel)^halo < 1e-10 (multiple of 32), seg_min = 4 tiles when halo <= 8 tiles."""
    c = max(att, rel)
    halo = (math.ceil(math.log(1e-10) / math.log(c)) + 31) // 32 * 32
    return halo, (4 * tile if halo <= 8 * tile else 2 ** 62)


def run_env(exe, d, x, att, rel, tile, halo, seg_min, starts="-", lengths="-"):
    x.astype(np.float32).tofile(os.path.join(d, "x"))
    _run(exe, "env", _f(att), _f(rel), tile, halo, seg_min, os.path.join(d, "x"), starts, lengths,
         os.path.join(d, "env"), os.path.join(d, "emax"))
    return np.fromfile(os.path.join(d, "env"), np.float32), np.fromfile(os.path.join(d, "emax"), np.float32)


def _env_signal(n, seed, silent=None):
    rng = np.random.default_rng(seed)
    t = np.arange(n)
    x = (np.sin(2 * np.pi * t / 211.0) * (0.2 + 0.8 * (np.sin(2 * np.pi * t / 9000.0) > 0)) * 0.6
         + 0.05 * rng.standard_normal(n)).astype(np.float32)
    if silent is not None:
        x[silent[0]:silent[1]] = 0.0
    return x


# (release_ms, attack_ms) of 0.2 / 0.05 ms: coefficients 0.90 / 0.66, halo 224: the segment kernel on small tiles
SMALL = dict(attack_ms=0.05, release_ms=0.2)


@pytest.mark.parametrize("case", ["one warp", "segments, small tiles", "segments, production tiles"])
def test_emu_envelope_vs_oracle(emu_at, case):
    if case == "segments, production tiles":
        att, rel = env_coeffs(SR)
        tile = 16384
        halo, seg_min = env_halo(att, rel, tile)
        lengths, kw = [65536, 70001], {}
    else:
        kw = SMALL if case == "segments, small tiles" else {}
        att, rel = env_coeffs(SR, **kw)
        tile = 256
        halo, seg_min = env_halo(att, rel, tile)
        lengths = [1024, 5000, 40000] if kw else [1, 511, 513, 3000]
        if not kw:
            seg_min = 2 ** 62
    with tempfile.TemporaryDirectory() as d:
        for n in lengths:
            x = _env_signal(n, n)
            env, emax = run_env(emu_at, d, x, att, rel, tile, halo, seg_min)
            ref = at.envelope_follow(x, SR, **kw)
            assert np.array_equal(env, ref), (case, n, int(np.count_nonzero(env != ref)))
            assert emax[0] == np.max(ref), (case, n)


@pytest.mark.parametrize("production", [False, True])
def test_emu_envelope_across_digital_silence(emu_at, production):
    """A silent stretch longer than the warm-up: the sequential follower decays into float32 subnormals and stops
    where rel * cur rounds back to cur; a tile that warms up inside the silence starts from 0 and stays there.  The
    segment follower is then off by at most that subnormal floor (<= 1e-10 of the maximum, as DESIGN states)."""
    kw = {} if production else SMALL
    att, rel = env_coeffs(SR, **kw)
    tile = 16384 if production else 256
    halo, seg_min = env_halo(att, rel, tile)
    n, gap = (240000, (60000, 180000)) if production else (12000, (3000, 6000))
    x = _env_signal(n, 5, gap)
    with tempfile.TemporaryDirectory() as d:
        env, emax = run_env(emu_at, d, x, att, rel, tile, halo, seg_min)
    ref = at.envelope_follow(x, SR, **kw)
    assert emax[0] == np.max(ref)
    err = float(np.max(np.abs(env.astype(np.float64) - ref)))
    assert err <= 1e-10 * float(np.max(ref))
    print(f"envelope across {gap[1] - gap[0]} silent samples (halo {halo}): max abs diff {err:.3e}, "
          f"{int(np.count_nonzero(env != ref))} samples differ")


# ------------------------------------------------------------------------------------------------ mix
def mix_params(cfg, sr=SR):
    f = at.sub_frequency(cfg)
    layer_on = int(cfg.sub_enabled and cfg.sub_level > 0.0 and f > 0.0)
    att, rel = env_coeffs(sr)
    return dict(sub_enabled=int(cfg.sub_enabled), layer_on=layer_on, att=att, rel=rel,
                level=float(np.float32(cfg.sub_level)), preserve=float(np.float32(cfg.sub_preserve_mix)),
                air_mix=float(np.float32(cfg.air_mix)), phase_k=float(np.float32(2.0 * np.pi * f)), sr=float(sr))


def run_mix(exe, d, x, sub, air, corr, prm, tile=16384, starts="-", lengths="-"):
    halo, seg_min = env_halo(prm["att"], prm["rel"], tile)
    for name, v in (("x", x), ("sub", sub), ("air", air), ("corr", corr)):
        v.astype(np.float32).tofile(os.path.join(d, name))
    _run(exe, "mix", prm["sub_enabled"], prm["layer_on"], _f(prm["att"]), _f(prm["rel"]), tile, halo, seg_min,
         _f(prm["level"]), _f(prm["preserve"]), _f(prm["air_mix"]), _f(prm["phase_k"]), _f(prm["sr"]),
         *[os.path.join(d, k) for k in ("x", "sub", "air", "corr")], starts, lengths, os.path.join(d, "y"),
         os.path.join(d, "layer"))
    return np.fromfile(os.path.join(d, "y"), np.float32), np.fromfile(os.path.join(d, "layer"), np.float32)


def mix_bands(n, seed, scale=1.0):
    rng = np.random.default_rng(seed)
    x = (scale * (0.5 * np.sin(np.arange(n) / 40.0) + 0.1 * rng.standard_normal(n))).astype(np.float32)
    sub, air, corr = (rng.standard_normal((3, n)) * 0.3).astype(np.float32)
    return x, sub, air, corr


MIX_CASES = {
    "default": dict(),
    "sub off": dict(sub_enabled=False),
    "layer off": dict(sub_level=0.0),
    "octave 0": dict(sub_octave=0, key="A", air_mix=0.7),
    "octave 6": dict(sub_octave=6, key="G#", sub_level=0.8),
}


@pytest.mark.parametrize("name", list(MIX_CASES) + ["quiet input"])
def test_emu_mix_vs_oracle(emu_at, name):
    cfg = at.AutotuneConfig(**MIX_CASES.get(name, {}))
    n = 6000
    x, sub, air, corr = mix_bands(n, 11)
    if name == "quiet input":
        x = (x / np.max(np.abs(x)) * 9e-7).astype(np.float32)    # envelope max <= 1e-6: no normalisation
    prm = mix_params(cfg)
    with tempfile.TemporaryDirectory() as d:
        y, layer = run_mix(emu_at, d, x, sub, air, corr, prm)
    ref_layer = at.sub_layer(x, SR, cfg)
    bound = 2 * float(np.spacing(np.float32(cfg.sub_level))) if cfg.sub_level > 0 else 0.0
    assert float(np.max(np.abs(layer.astype(np.float64) - ref_layer))) <= bound, name
    if not prm["layer_on"]:
        assert (layer == 0).all()
    low = (cfg.sub_preserve_mix * sub) + layer if cfg.sub_enabled else sub   # the apply_autotune_v1 sum, same layer
    assert np.array_equal(y, (low + corr + (cfg.air_mix * air)).astype(np.float32)), name
    if name == "quiet input":
        assert float(np.max(at.envelope_follow(x, SR))) <= 1e-6 and np.max(np.abs(layer)) < 1e-6
