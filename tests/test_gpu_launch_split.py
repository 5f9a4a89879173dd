"""GPU: batches past the grid limit.  A launch holds at most 65 535 CTA rows on gridDim.y (131 070 clips for the
two-group spectral kernel); past that the library splits the batch into several launches (qd::for_each_launch), each
advancing the clip index clip0.  Every batch here is large enough to split and must come out bit-identical, output and
taps, to the same clips rendered in batches of a few thousand.  The clips are short (a few hundred samples) so that the
batches stay cheap."""
import ctypes as C

import numpy as np
import pytest

from quantumdistortion_b200 import synth

pytestmark = pytest.mark.gpu

SR = 48000
SMALL = 4096     # clips per reference batch


def _batch(b, n, seed=0, gain=0.6):
    import torch
    rng = np.random.default_rng(seed)
    base = np.stack([synth.bass_clip(seed + i, n, SR) for i in range(16)]).astype(np.float32)
    x = base[rng.integers(0, 16, b)] * rng.uniform(0.2, 1.0, (b, 1)).astype(np.float32) * np.float32(gain)
    x += (0.01 * rng.standard_normal((b, n))).astype(np.float32)   # every clip differs
    return torch.from_numpy(x).cuda()


def _check_uniform(x, seeds=None, **kw):
    import torch
    import quantumdistortion_b200 as qd
    y, taps = qd.process_batch(x, SR, return_taps=True, seeds=seeds, **kw)
    for b0 in range(0, x.shape[0], SMALL):
        s = None if seeds is None else seeds[b0:b0 + SMALL]
        ry, rt = qd.process_batch(x[b0:b0 + SMALL], SR, return_taps=True, seeds=s, **kw)
        assert torch.equal(y[b0:b0 + SMALL], ry), b0
        for k in ("pre_quant", "post_dist"):
            assert torch.equal(taps[k][b0:b0 + SMALL], rt[k]), (k, b0)
    return y


def test_headline_kernel_past_two_group_limit():
    """defaults at n_fft 2048, float32: the NG = 2 kernel splits at 65 535 * 2 clips"""
    _check_uniform(_batch(131_100, 300), quantize_mode="spectral_bins", n_fft=2048, precision="float32")


def test_team_kernel_past_grid_limit():
    _check_uniform(_batch(65_600, 400, seed=1), quantize_mode="spectral_bins", n_fft=4096, precision="float32")


def test_multiband_freeze_fx_limiter_past_grid_limit():
    """crossover, freeze magnitudes, per-clip FX-table rows and the per-clip peaks that let the limiter skip quiet clips,
    all across the split"""
    b = 65_600
    x = _batch(b, 300, seed=2, gain=3.0)   # loud: the limiter works on these clips
    x[1::3] *= 0.01                        # quiet: the limiter skips them by their peak
    _check_uniform(x, seeds=[1000 + i for i in range(b)], quantize_mode="spectral_bins", n_fft=2048,
                   precision="float32", use_multiband=True, crossover_hz=300.0, spectral_freeze=True,
                   spectral_fx_mode="bin_scramble", spectral_fx_strength=0.6)


def test_ragged_device_past_grid_limit():
    import torch
    import quantumdistortion_b200 as qd
    rng = np.random.default_rng(3)
    lengths = rng.integers(100, 500, 65_600)
    lengths[::1000] = 0
    flat = _batch(1, int(lengths.sum()), seed=3)[0]
    ends = np.cumsum(lengths)
    clips = [flat[e - n:e] for e, n in zip(ends, lengths)]
    kw = dict(quantize_mode="spectral_bins", n_fft=2048, precision="float32")
    ys, _ = qd.process_batch(clips, SR, **kw)
    for b0 in range(0, len(clips), SMALL):
        ref, _ = qd.process_batch(clips[b0:b0 + SMALL], SR, **kw)
        for i, r in enumerate(ref):
            assert torch.equal(ys[b0 + i], r), (b0 + i, int(lengths[b0 + i]))


def test_autotune_uniform_past_grid_limit():
    """autotune_v1 renders chunk_clips clips per call (default 2048, which never splits); 70 000 in one call does"""
    import torch
    import quantumdistortion_b200 as qd
    from quantumdistortion_b200 import autotune
    x = _batch(70_000, 300, seed=4)
    p = qd.make_renderer(300, SR, quantize_mode="autotune_v1").params
    y, taps, _, _ = autotune.render_device(p, x, want_taps=True, chunk_clips=70_000)
    ry, rtaps, _, _ = autotune.render_device(p, x, want_taps=True, chunk_clips=SMALL)
    assert torch.equal(y, ry)
    for k in ("pre_quant", "post_dist"):
        assert torch.equal(taps[k], rtaps[k]), k


def test_autotune_ragged_past_grid_limit():
    import torch
    import quantumdistortion_b200 as qd
    rng = np.random.default_rng(5)
    lengths = rng.integers(17, 500, 65_600)
    lengths[::1000] = 0
    flat = _batch(1, int(lengths.sum()), seed=5)[0]
    ends = np.cumsum(lengths)
    clips = [flat[e - n:e] for e, n in zip(ends, lengths)]
    ys, taps = qd.process_batch(clips, SR, return_taps=True, quantize_mode="autotune_v1")
    for b0 in range(0, len(clips), SMALL):
        ref, rtaps = qd.process_batch(clips[b0:b0 + SMALL], SR, return_taps=True, quantize_mode="autotune_v1")
        for i, r in enumerate(ref):
            assert torch.equal(ys[b0 + i], r), (b0 + i, int(lengths[b0 + i]))
            for k in ("pre_quant", "post_dist"):
                assert torch.equal(taps[k][b0 + i], rtaps[k][i]), (k, b0 + i)


def test_spectral_peak_bins_past_grid_limit():
    import torch
    from quantumdistortion_b200 import analyses
    x = _batch(65_600, 2048, seed=6)
    bins = analyses.spectral_peak_bins(x, n_fft=2048, topn=3, precision="float32")
    for b0 in range(0, x.shape[0], SMALL):
        assert torch.equal(bins[b0:b0 + SMALL], analyses.spectral_peak_bins(x[b0:b0 + SMALL], n_fft=2048, topn=3,
                                                                             precision="float32")), b0


def test_render_device_rejects_batches_past_int32():
    import torch
    import quantumdistortion_b200 as qd
    from quantumdistortion_b200 import _lib
    r = qd.make_renderer(300, SR, quantize_mode="spectral_bins")
    buf = torch.zeros(1024, device="cuda")
    rc = r._lib.qd_render_device(r._plan, buf.data_ptr(), buf.data_ptr(), 2 ** 31, None, buf.data_ptr(),
                                 buf.numel() * 4, C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == -1 and b"2^31" in _lib.load().qd_last_error()
