"""GPU: the scale-alignment metric on ragged batches (spectral_peak_bins / avg_cents_offset_batch on a list of clips of
different lengths, one qd_spectral_peaks_device_varlen call).  Every clip must get exactly what it gets alone."""
import numpy as np
import pytest

import qd_cases
from oracle import qd_oracle as orc
from quantumdistortion_b200 import synth

pytestmark = pytest.mark.gpu

SR = 48000
SMALL = 4096     # clips per reference call past the grid limit


def _lengths(n_fft, rng):
    hop = n_fft // 4
    around = [k * hop + d for k in (1, 2, 5) for d in (-1, 0, 1)]
    return [0, 1, hop - 1, n_fft] + around + [int(v) for v in rng.integers(2, 3 * SR, 3)] + [0]


def _clips(lengths, seed):
    return [(0.6 * synth.bass_clip(seed + i, n, SR) + 0.05 * synth.noise_clip(seed + i, n)).astype(np.float32)
            if n >= 2 else np.full(n, 0.5, np.float32) for i, n in enumerate(lengths)]


def _container(clips, kind):
    import torch
    if kind == "numpy":
        return clips
    if kind == "numpy64":
        return [c.astype(np.float64) for c in clips]
    ts = [torch.from_numpy(c) for c in clips]
    return [t.cuda() for t in ts] if kind == "cuda" else ts


def _np(b):
    return b.cpu().numpy() if hasattr(b, "cpu") else np.asarray(b)


@pytest.mark.parametrize("name", list(qd_cases.ANALYSIS_CASES))
def test_ragged_metric_matches_reference_fixtures(name):
    """each fixture input in a list among clips of random lengths from 0 to 3 s, with that case's parameters"""
    from quantumdistortion_b200 import analyses
    g = qd_cases.Golden("analysis")
    kind, seed, n, sr, key, scale, kw = qd_cases.ANALYSIS_CASES[name]
    x = g.input(name, qd_cases.make_signal(kind, seed, n, sr)).astype(np.float32)
    rng = np.random.default_rng(seed)
    others = _clips([int(v) for v in rng.integers(0, 3 * sr, 6)] + [0], seed + 100)
    at = int(rng.integers(0, len(others) + 1))
    batch = others[:at] + [x] + others[at:]
    avgs, per = analyses.avg_cents_offset_batch(batch, sr, key, scale, **kw)
    assert len(per) == len(batch) and avgs.shape == (len(batch),)
    assert np.array_equal(per[at], g[f"{name}/per_peak"]), name
    ref = float(g[f"{name}/avg"])
    assert (np.isnan(ref) and np.isnan(avgs[at])) or avgs[at] == ref


@pytest.mark.parametrize("precision", ["float64", "float32"])
@pytest.mark.parametrize("n_fft", [512, 1024, 2048, 4096, 8192])
def test_ragged_bins_match_clips_alone(n_fft, precision):
    import torch
    from quantumdistortion_b200 import analyses
    rng = np.random.default_rng(n_fft + (precision == "float32"))
    clips = _clips(_lengths(n_fft, rng), n_fft)
    hop = n_fft // 4
    for topn, min_db in [(1, -60.0), (3, -30.0), (8, -60.0)]:
        kw = dict(n_fft=n_fft, topn=topn, min_db=min_db, precision=precision)
        alone = [analyses.spectral_peak_bins(c[None, :], **kw)[0] if len(c) else np.full((1, topn), -1, np.int16)
                 for c in clips]
        assert any((a >= 0).any() for a in alone)
        for kind in ("numpy", "numpy64", "cpu", "cuda"):
            got = analyses.spectral_peak_bins(_container(clips, kind), **kw)
            assert isinstance(got, list) and len(got) == len(clips)
            for i, (b, a) in enumerate(zip(got, alone)):
                if kind.startswith("numpy"):
                    assert isinstance(b, np.ndarray)
                else:
                    assert isinstance(b, torch.Tensor) and b.is_cuda == (kind == "cuda")
                assert b.dtype in (np.int16, torch.int16) and tuple(b.shape) == (1 + len(clips[i]) // hop, topn)
                assert np.array_equal(_np(b), a), (kind, topn, min_db, i, len(clips[i]))


def test_ragged_metric_equals_per_clip_calls_on_renders():
    """The motivating flow (scripts/validate_dsp_metrics.py:59-105 on a sample library): render a list of clips of
    different lengths in one call, then measure the list in one call."""
    import quantumdistortion_b200 as qd
    from quantumdistortion_b200 import analyses
    lengths = [24000, 9000, 30011, 4097, 18000]
    x = [synth.bass_clip(70 + i, n, SR).astype(np.float32) for i, n in enumerate(lengths)]
    ys, _ = qd.process_batch(x, SR, quantize_mode="spectral_bins", limiter_on=False)
    wet, wper = analyses.avg_cents_offset_batch(ys, SR, "D", "minor")
    dry, dper = analyses.avg_cents_offset_batch(x, SR, "D", "minor")
    for sig, avgs, per in ((ys, wet, wper), (x, dry, dper)):
        for i, s in enumerate(sig):
            a, p = analyses.avg_cents_offset_from_scale(s, SR, "D", "minor")
            assert np.array_equal(per[i], p) and avgs[i] == a, i
            oa, op = orc.avg_cents_offset_from_scale(s, SR, "D", "minor")
            assert np.array_equal(per[i], op) and avgs[i] == oa, i
    assert np.mean(wet) < np.mean(dry)


def test_ragged_list_validation_on_the_device():
    import torch
    from quantumdistortion_b200 import analyses
    with pytest.raises(ValueError, match="all CUDA or all CPU"):
        analyses.spectral_peak_bins([torch.zeros(100).cuda(), torch.zeros(100)])
    with pytest.raises(ValueError, match="1-D"):
        analyses.avg_cents_offset_batch([torch.zeros(100).cuda(), torch.zeros(2, 100).cuda()], SR, "D", "minor")
    got = analyses.spectral_peak_bins([np.zeros(0, np.float32)] * 3, topn=2)
    assert len(got) == 3 and all(np.array_equal(b, np.full((1, 2), -1, np.int16)) for b in got)
    avgs, per = analyses.avg_cents_offset_batch([np.zeros(0, np.float32)], SR, "D", "minor")
    assert np.isnan(avgs[0]) and per[0].size == 0


def test_ragged_peak_bins_past_grid_limit():
    import torch
    from quantumdistortion_b200 import analyses
    rng = np.random.default_rng(6)
    lengths = rng.integers(0, 3000, 65_600)
    lengths[::997] = 0
    flat = torch.from_numpy((0.5 * synth.noise_clip(6, int(lengths.sum()))).astype(np.float32)).cuda()
    ends = np.cumsum(lengths)
    clips = [flat[e - n:e] for e, n in zip(ends, lengths)]
    kw = dict(n_fft=2048, topn=3, precision="float32")
    got = analyses.spectral_peak_bins(clips, **kw)
    ref = []
    for b0 in range(0, len(clips), SMALL):
        ref += analyses.spectral_peak_bins(clips[b0:b0 + SMALL], **kw)
    assert [tuple(b.shape) for b in got] == [tuple(b.shape) for b in ref]
    assert torch.equal(torch.cat(got), torch.cat(ref))
