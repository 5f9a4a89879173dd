"""GPU: ragged batches (process_batch on a list of clips of different lengths).  Every clip must come out bit-identical
to the same clip rendered alone through the uniform path (process_batch on [1, n_c]), on every transport."""
import numpy as np
import pytest

from oracle import qd_oracle as orc
from quantumdistortion_b200 import synth

pytestmark = pytest.mark.gpu

SR = 48000


def _lengths(n_fft):
    hop = n_fft // 4
    # empty, one sample, shorter than a hop, shorter than a frame, odd, ~4k not a multiple of the hop, 10 s
    return [0, 1, hop - 5, n_fft - 3, 4097, 4000 + hop // 2 + 1, 10 * SR]


def _clips(lengths, seed=0):
    return [(0.6 * synth.bass_clip(seed + i, n, SR)).astype(np.float32) if n else np.zeros(0, np.float32)
            for i, n in enumerate(lengths)]


def _alone(clip, seeds=None, **kw):
    import torch
    import quantumdistortion_b200 as qd
    y, taps = qd.process_batch(torch.from_numpy(clip[None, :]).cuda(), SR, seeds=seeds, **kw)
    return y[0].cpu().numpy(), None if taps is None else {k: v[0].cpu().numpy() for k, v in taps.items()}


def _check_against_alone(clips, kw, seeds=None, return_taps=False):
    import torch
    import quantumdistortion_b200 as qd
    ys, taps = qd.process_batch([torch.from_numpy(c).cuda() for c in clips], SR, seeds=seeds,
                                return_taps=return_taps, **kw)
    torch.cuda.synchronize()
    assert len(ys) == len(clips)
    for i, c in enumerate(clips):
        got = ys[i].cpu().numpy()
        assert got.shape == c.shape
        if len(c) == 0:
            continue
        s = seeds[i] if isinstance(seeds, list) else seeds
        ref, rtaps = _alone(c, seeds=s, return_taps=return_taps, **kw)
        assert np.array_equal(got, ref), (kw, i, len(c), float(np.max(np.abs(got - ref))))
        if return_taps:
            for k in ("pre_quant", "post_dist"):
                assert np.array_equal(taps[k][i].cpu().numpy(), rtaps[k]), (k, i)


@pytest.mark.parametrize("precision", ["float32", "float64"])
@pytest.mark.parametrize("n_fft", [512, 1024, 2048, 4096, 8192])
def test_ragged_bit_identical_to_single(n_fft, precision):
    _check_against_alone(_clips(_lengths(n_fft)), dict(quantize_mode="spectral_bins", n_fft=n_fft, precision=precision))


CONFIGS = {
    "single_band": {},
    "multiband": {"use_multiband": True, "crossover_hz": 300.0},
    "tube": {"distortion_mode": "tube", "distortion_params": {"drive": 2.0, "warmth": 0.4}},
    "wavefold_bias": {"distortion_params": {"fold_amount": 1.7, "bias": 0.05}},
    "delta_listen": {"delta_listen": True},
    "passthrough": {"passthrough_test": True, "use_multiband": True},
    "freeze": {"spectral_freeze": True},
    "formant": {"formant_shift": 3.0},
    "bitcrush": {"use_multiband": True, "spectral_fx_mode": "bitcrush", "spectral_fx_strength": 0.5},
}


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_ragged_configs(name):
    kw = dict(quantize_mode="spectral_bins", n_fft=2048, precision="float32", **CONFIGS[name])
    _check_against_alone(_clips(_lengths(2048), seed=10), kw, return_taps=name in ("single_band", "multiband"))


@pytest.mark.parametrize("mode", ["bin_scramble", "phase_dispersal"])
@pytest.mark.parametrize("seeds", ["list", "int"])
def test_ragged_random_fx(mode, seeds):
    lengths = _lengths(2048)
    sd = [11 + i for i in range(len(lengths))] if seeds == "list" else 5
    kw = dict(quantize_mode="spectral_bins", n_fft=2048, precision="float32", use_multiband=True,
              spectral_fx_mode=mode, spectral_fx_strength=0.6)
    _check_against_alone(_clips(lengths, seed=20), kw, seeds=sd)


def test_ragged_random_fx_global_state_matches_loop():
    """seeds=None: clip after clip from the global state, like a loop of single-clip renders."""
    import torch
    import quantumdistortion_b200 as qd
    clips = _clips([3000, 0, 9001, 700], seed=30)
    kw = dict(quantize_mode="spectral_bins", n_fft=2048, precision="float32", use_multiband=True,
              spectral_fx_mode="bin_scramble", spectral_fx_strength=0.4)
    np.random.seed(99)
    ys, _ = qd.process_batch(clips, SR, **kw)
    after = np.random.get_state()[1].copy()
    np.random.seed(99)
    for c, y in zip(clips, ys):
        if len(c):
            ref, _ = qd.process_batch(c[None, :], SR, **kw)
            assert np.array_equal(y, ref[0])
    assert np.array_equal(np.random.get_state()[1], after)
    torch.cuda.synchronize()


def test_ragged_against_oracle():
    import quantumdistortion_b200 as qd
    clips = _clips([24000, 5001, 700], seed=40)
    for kw in ({}, {"use_multiband": True, "crossover_hz": 300.0}):
        ys, _ = qd.process_batch(clips, SR, quantize_mode="spectral_bins", **kw)
        for c, y in zip(clips, ys):
            ref, _ = orc.process_audio(c, SR, **kw)
            err = float(np.max(np.abs(y.astype(np.float64) - ref)))
            assert err <= 1e-4 and orc.null_test_db(y, ref) <= -80.0, (kw, len(c), err)


def test_ragged_transports_agree():
    """Device path, packed pinned host path, pageable host buffers through the library's staging ring, and PCM16 --
    with chunk budgets smaller than one clip and smaller than the batch."""
    import torch
    import quantumdistortion_b200 as qd
    from quantumdistortion_b200.pipeline import make_renderer, pack_layout
    lengths = [48000, 0, 1, 30001, 2047, 96000, 5]
    clips = _clips(lengths, seed=50)
    kw = dict(quantize_mode="spectral_bins", use_multiband=True, precision="float32")
    dev, _ = qd.process_batch([torch.from_numpy(c).cuda() for c in clips], SR, **kw)
    dev = [y.cpu().numpy() for y in dev]
    host_np, _ = qd.process_batch(clips, SR, **kw)
    host_t, _ = qd.process_batch([torch.from_numpy(c) for c in clips], SR, **kw)
    for a, b, c in zip(dev, host_np, host_t):
        assert np.array_equal(a, b) and np.array_equal(a, c.numpy())
    live = [c for c in clips if len(c)]
    n_live = np.array([len(c) for c in live])
    starts, span = pack_layout(n_live, 4)
    x = torch.zeros(span, dtype=torch.float32)
    for s, c in zip(starts, live):
        x[s:s + len(c)] = torch.from_numpy(c)
    r = make_renderer(int(n_live.max()), SR, ragged=True, **kw)
    ref = np.concatenate([y for y in dev if len(y)])
    for budget in (10000, 60000, int(span) // 2, 0):   # < one clip, < the batch, default
        for pinned in (False, True):
            xx = x.pin_memory() if pinned else x
            y = torch.empty_like(xx)
            r.render_host_varlen(xx, y, starts, n_live, chunk_samples=budget)
            got = np.concatenate([y[s:s + n].numpy() for s, n in zip(starts, n_live)])
            assert np.array_equal(got, ref), (budget, pinned)
    # PCM16 on the link: the same as converting the float32 result with save_audio's rule
    pcm = [np.round(c * 32767.0).astype(np.int16) for c in clips]
    y16, _ = qd.process_batch(pcm, SR, **kw)
    for c16, y in zip(pcm, y16):
        assert y.dtype == np.int16 and y.shape == c16.shape
        if len(c16):
            ref32, _ = qd.process_batch((c16.astype(np.float32) / 32768.0)[None, :], SR, **kw)
            want = np.clip(np.rint(ref32[0].astype(np.float64) * 32767.0), -32768, 32767).astype(np.int16)
            assert np.array_equal(y, want)


def test_ragged_host_validation():
    import torch
    from quantumdistortion_b200 import _lib
    from quantumdistortion_b200.pipeline import make_renderer
    r = make_renderer(1000, SR, ragged=True, quantize_mode="spectral_bins")
    x = torch.zeros(4000, dtype=torch.float32)
    y = torch.empty_like(x)
    for starts, lengths in (([0, 1004], [1000, 1001]),      # longer than the plan
                            ([0, 500], [600, 100]),         # overlap
                            ([0, 8], [4, -1])):             # negative length
        with pytest.raises(_lib.QdError):
            r.render_host_varlen(x, y, np.array(starts, np.int64), np.array(lengths, np.int32))


@pytest.mark.parametrize("extra", [{"quantize_mode": "spectral_bins", "use_multiband": True}, None])
def test_process_files_mixed_lengths(tmp_path, extra):
    from quantumdistortion_b200.audio_io import save_audio
    from quantumdistortion_b200.harness import process_file_to_file, process_files
    lengths = [24000, 0, 7001, 24000, 1500, 50000]
    pairs = []
    for i, n in enumerate(lengths):
        src = tmp_path / f"in{i}.wav"
        save_audio(src, (0.5 * synth.bass_clip(60 + i, n, SR)).astype(np.float32) if n else np.zeros(0, np.float32), SR)
        pairs.append((src, tmp_path / f"batch{i}.wav"))
    assert process_files(pairs, extra_params=extra) == len(pairs)
    for i, (src, out) in enumerate(pairs):
        one = tmp_path / f"one{i}.wav"
        process_file_to_file(src, one, extra_params=extra)
        assert out.read_bytes() == one.read_bytes(), i
