"""GPU (B200): every autotune_v1 stage after the band split against the oracle fed the GPU's OWN input to that stage
(AutotuneRenderer.render_device(..., debug=True)), so that a stage's error is not mixed with the error of the stages
before it and the bounds can be as tight as the stage's arithmetic:

  features     rms rtol 1e-5 vs frame_features(det); flatness inside what a float32 FFT can do to it
               (qd_cases.flatness_interval: rtol 1e-4 where the spectrum lies above the FFT's rounding, wider on the
               tonal frames of the band-limited detector signal), flatness gate exact; pitch 1e-9 relative and
               confidence 1e-9 vs detect_pitch_yin (DESIGN section 9); voiced decisions exact
  ratio_track  bit-identical to np.interp(note_hold_ratios(features)) as float32
  corrected    within 1 float32 ulp of granular_pitch_shift(body, ratio_track) (the Hann weight's cos)
  sub_layer    within 4 ulp of sub_level of sub_layer(x) (the device sinf is a 2-ulp function)
  pre_quant    bit-identical to the oracle's sum of the GPU's sub, air, corrected and sub_layer

Each case prints its per-stage worst error."""
import numpy as np
import pytest

import qd_cases
from oracle import qd_autotune as at

CFG = at.AutotuneConfig()


@pytest.fixture(scope="module")
def qd():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import quantumdistortion_b200 as q
    return q


def _ulps(a, b):
    def key(v):
        i = np.asarray(v, dtype=np.float32).view(np.int32).astype(np.int64)
        return np.where(i < 0, -(i & 0x7FFFFFFF), i)
    return np.abs(key(a) - key(b))


def _frames(det):
    """The zero-padded detector frames of frame_features."""
    return [np.pad(det[s:s + 4096], (0, max(0, s + 4096 - len(det)))) for s in range(0, len(det), 512)]


def _voice(f0, sr, seed):
    """A voice-like tone on the frequency track f0 (Hz per sample) over a -60 dB noise floor."""
    rng = np.random.default_rng(seed)
    ph = 2 * np.pi * np.cumsum(f0) / sr
    x = sum(0.35 / k * np.sin(k * ph + 0.3 * k) for k in range(1, 5))
    return (x + 1e-3 * rng.standard_normal(len(f0))).astype(np.float32)


def _case(name):
    sr = 96000 if name == "96 kHz" else 48000
    if name.startswith("n="):
        n = int(name[2:])
        t = np.arange(n) / sr
        return _voice(240.0 * 2 ** (0.4 * np.sin(2 * np.pi * 1.3 * t) / 12), sr, n), sr
    if name == "96 kHz":
        n = 100000
        return _voice(np.full(n, 311.0), sr, 1), sr
    if name == "3 s silence between tones":
        a, b = _voice(np.full(sr, 190.0), sr, 2), _voice(np.full(sr, 290.0), sr, 3)
        return np.concatenate([a, np.zeros(3 * sr, np.float32), b]), sr
    if name == "two-octave glide":
        n = 3 * sr
        return _voice(110.0 * 4.0 ** (np.arange(n) / n), sr, 4), sr
    if name == "flat ratio track":                        # A4 is in D minor: the correction stays within 1e-3 of 1
        return _voice(np.full(30000, 440.0), sr, 5), sr
    raise KeyError(name)


CASES = ["n=513", "n=2049", "n=4097", "n=65535", "n=65536", "n=480000", "96 kHz", "3 s silence between tones",
         "two-octave glide", "flat ratio track"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_autotune_stage_on_gpu_upstream(qd, name):
    import torch
    from quantumdistortion_b200 import make_renderer
    x, sr = _case(name)
    n = len(x)
    r = make_renderer(n, sr, quantize_mode="autotune_v1", limiter_on=False)
    y, taps, dbg = r.render_device(torch.from_numpy(x[None, :]).cuda(), want_taps=True, debug=True)
    d = {k: v[0].cpu().numpy() for k, v in dbg.items()}
    pre = taps["pre_quant"][0].cpu().numpy()
    worst = {}

    # features: the oracle's frame features of the GPU's detector band
    feat = d["features"]
    centers, rms, flat, pitch, conf = at.frame_features(d["det"], sr, CFG)
    assert feat.shape == (len(centers), 4)
    assert np.allclose(feat[:, 0], rms, rtol=1e-5, atol=0.0)
    lo, hi = np.array([qd_cases.flatness_interval(fr) for fr in _frames(d["det"])]).T
    assert ((lo <= feat[:, 1]) & (feat[:, 1] <= hi)).all(), np.flatnonzero((feat[:, 1] < lo) | (feat[:, 1] > hi))
    thr = CFG.detector_flatness_threshold
    clear = (hi < thr) | (lo > thr)                          # frames whose interval does not straddle the gate
    assert np.array_equal(feat[clear, 1] <= thr, flat[clear] <= thr)
    assert np.array_equal(feat[:, 2] > 0, pitch > 0)
    assert np.allclose(feat[:, 2], pitch, rtol=1e-9, atol=0.0)
    assert np.allclose(feat[:, 3], conf, rtol=0.0, atol=1e-9)
    v = pitch > 0
    worst["rms rel"] = float(np.max(np.abs(feat[:, 0] / np.where(rms > 0, rms, 1) - np.where(rms > 0, 1, 0))))
    worst["flatness rel"] = float(np.max(np.abs(feat[:, 1] / flat - 1)))
    worst["flatness rel (flatness > 1e-3)"] = float(np.max(np.abs(feat[:, 1] / flat - 1)[flat > 1e-3], initial=0.0))
    worst["pitch rel"] = float(np.max(np.abs(feat[v, 2] / pitch[v] - 1), initial=0.0))
    worst["conf abs"] = float(np.max(np.abs(feat[:, 3] - conf)))

    # ratio track: the oracle's note hold and interpolation of the GPU's features
    ratios = at.note_hold_ratios(feat[:, 0], feat[:, 1], feat[:, 2], feat[:, 3], CFG)
    track = np.interp(np.arange(n, dtype=np.float64), centers, ratios).astype(np.float32)
    assert np.array_equal(d["ratio_track"], track)
    flat_track = bool(np.allclose(track, 1.0, atol=1e-3))    # the shifter's early-out: corrected = body
    if name in ("flat ratio track", "n=2049", "two-octave glide"):
        assert flat_track == (name == "flat ratio track")
    worst["flat track"] = int(flat_track)

    # shifter on the GPU's body and ratio track
    ref = at.granular_pitch_shift(d["body"], d["ratio_track"], CFG.grain_size, CFG.buffer_size)
    u = _ulps(d["corrected"], ref)
    assert u.max() <= 1, int(u.max())
    worst["corrected ulp"] = int(u.max())
    worst["corrected samples differing"] = int(np.count_nonzero(u))

    # sub layer from the input
    layer = at.sub_layer(x, sr, CFG)
    lerr = float(np.max(np.abs(d["sub_layer"].astype(np.float64) - layer)))
    assert lerr <= 4 * float(np.spacing(np.float32(CFG.sub_level))), lerr
    worst["sub_layer abs"] = lerr

    # the mix of the GPU's bands
    low = (CFG.sub_preserve_mix * d["sub"]) + d["sub_layer"]
    assert np.array_equal(pre, (low + d["corrected"] + (CFG.air_mix * d["air"])).astype(np.float32))
    print(f"{name} (n={n}, sr={sr}): " + ", ".join(f"{k} {v:.3g}" if isinstance(v, float) else f"{k} {v}"
                                                    for k, v in worst.items()))
