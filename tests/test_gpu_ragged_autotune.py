"""GPU: ragged batches in quantize_mode="autotune_v1" (process_batch on a list of clips of different lengths).  Every
clip must come out bit-identical to the same clip rendered alone through the uniform path (process_batch on [1, n_c]),
output and taps, on every transport."""
import numpy as np
import pytest

from oracle import qd_oracle as orc
from quantumdistortion_b200 import synth

pytestmark = pytest.mark.gpu

SR = 48000
HOP = 512
# empty, just past the filter padding, one hop -/+ 1, one detector frame -1/0/+1, the envelope-follower switch
# (four 16384-sample tiles) -1/0, an odd length near 1 s, 10 s + 1
LENGTHS = [0, 16, 17, HOP - 1, HOP + 1, 4095, 4096, 4097, 65535, 65536, SR - 1, 10 * SR + 1]


def _clips(lengths, seed=0):
    return [(0.6 * synth.bass_clip(seed + i, n, SR)).astype(np.float32) if n else np.zeros(0, np.float32)
            for i, n in enumerate(lengths)]


def _alone(clip, return_taps=False, **kw):
    import torch
    import quantumdistortion_b200 as qd
    y, taps = qd.process_batch(torch.from_numpy(clip[None, :]).cuda(), SR, return_taps=return_taps, **kw)
    return y[0].cpu().numpy(), None if taps is None else {k: v[0].cpu().numpy() for k, v in taps.items()}


CONFIGS = {
    "defaults": {},
    "no_sub": {"sub_enabled": False},
    "tail_only": {"snap_strength": 0.0},
    "tube": {"distortion_mode": "tube", "distortion_params": {"drive": 2.0, "warmth": 0.7}},
    "delta_listen": {"delta_listen": True},
    "half_wet": {"dry_wet": 0.5},
    "d_minor": {"key": "D", "scale": "minor"},
}


@pytest.mark.parametrize("name", list(CONFIGS))
def test_ragged_autotune_bit_identical_to_single(name):
    import torch
    import quantumdistortion_b200 as qd
    kw = CONFIGS[name]
    clips = _clips(LENGTHS)
    ys, taps = qd.process_batch([torch.from_numpy(c).cuda() for c in clips], SR, return_taps=True, **kw)
    torch.cuda.synchronize()
    assert len(ys) == len(clips)
    for i, c in enumerate(clips):
        got = ys[i].cpu().numpy()
        assert got.shape == c.shape
        if len(c) == 0:
            assert taps["pre_quant"][i].numel() == 0 and taps["post_dist"][i].numel() == 0
            continue
        ref, rtaps = _alone(c, return_taps=True, **kw)
        assert np.array_equal(got, ref), (name, i, len(c), float(np.max(np.abs(got - ref))))
        for k in ("pre_quant", "post_dist"):
            assert np.array_equal(taps[k][i].cpu().numpy(), rtaps[k]), (name, k, i, len(c))


def test_ragged_autotune_transports():
    """CUDA tensors, NumPy (pinned packing), CPU tensors, pageable host buffers straight into the renderer, PCM16, and
    host chunk budgets smaller than one clip and smaller than the batch: all the same bits."""
    import torch
    import quantumdistortion_b200 as qd
    from quantumdistortion_b200.pipeline import make_renderer, pack_layout
    lengths = [4097, 0, 30000, 17, 96001, 5000, 65536]
    clips = _clips(lengths, seed=20)
    ref = [_alone(c)[0] if len(c) else c for c in clips]
    ys, _ = qd.process_batch([torch.from_numpy(c).cuda() for c in clips], SR)
    for i in range(len(clips)):
        assert np.array_equal(ys[i].cpu().numpy(), ref[i]), ("cuda", i)
    for chunk in (128, 1, 3):   # default; smaller than the longest clip; smaller than the batch
        got, _ = qd.process_batch(clips, SR, chunk_clips=chunk)
        for i in range(len(clips)):
            assert np.array_equal(got[i], ref[i]), ("numpy", chunk, i)
    got, _ = qd.process_batch([torch.from_numpy(c) for c in clips], SR, chunk_clips=2)
    for i in range(len(clips)):
        assert np.array_equal(got[i].numpy(), ref[i]), ("cpu tensor", i)
    # pageable (not pinned) host buffers handed to the renderer directly
    live = [c for c in clips if len(c)]
    n = np.array([len(c) for c in live], np.int64)
    starts, span = pack_layout(n, 4)
    x = np.zeros(span, np.float32)
    for s, c in zip(starts, live):
        x[s:s + len(c)] = c
    xt, yt = torch.from_numpy(x), torch.zeros(span, dtype=torch.float32)
    r = make_renderer(int(n.max()), SR, ragged=True)
    r.render_host_varlen(xt, yt, starts, n.astype(np.int32), chunk_samples=40000)
    k = 0
    for i, c in enumerate(clips):
        if len(c):
            assert np.array_equal(yt.numpy()[starts[k]:starts[k] + len(c)], ref[i]), ("pageable", i)
            k += 1
    # PCM16 in, PCM16 out
    pcm = [np.clip(np.rint(c.astype(np.float64) * 32767.0), -32768, 32767).astype(np.int16) for c in clips]
    got16, _ = qd.process_batch(pcm, SR, chunk_clips=2)
    for i, c in enumerate(pcm):
        assert got16[i].dtype == np.int16 and got16[i].shape == c.shape
        if len(c):
            one, _ = qd.process_batch(c[None, :], SR)
            assert np.array_equal(got16[i], one[0]), ("pcm16", i)


def test_ragged_autotune_short_clip_raises():
    import quantumdistortion_b200 as qd
    clips = _clips([4096, 5, 20000])
    with pytest.raises(ValueError, match="padlen"):
        qd.process_batch(clips, SR)
    with pytest.raises(ValueError, match="padlen"):
        qd.process_batch(clips[1][None, :], SR)
    # the tail-only render has no zero-phase filters: short clips are fine there
    ys, _ = qd.process_batch(clips, SR, snap_strength=0.0)
    assert [len(y) for y in ys] == [4096, 5, 20000]


def test_ragged_autotune_against_oracle():
    import quantumdistortion_b200 as qd
    from oracle import qd_autotune as at
    clips = [synth.tone_clip(i, n, SR) for i, n in enumerate([12000, 9001, 4097])]
    ys, _ = qd.process_batch(clips, SR)
    for i, c in enumerate(clips):
        ref, _ = at.process_audio_autotune(c, SR)
        err = float(np.max(np.abs(ys[i].astype(np.float64) - ref)))
        assert err <= 1e-4 and orc.null_test_db(ys[i], ref) <= -80.0, (i, err)


def test_process_files_default_config_mixed_lengths_and_formats(tmp_path):
    from scipy.io import wavfile
    from quantumdistortion_b200.audio_io import save_audio
    from quantumdistortion_b200.harness import process_file_to_file, process_files
    lengths = [24000, 0, 7001, 50000, 1500, 24000, 33333]
    pairs = []
    for i, n in enumerate(lengths):
        src = tmp_path / f"in{i}.wav"
        x = (0.5 * synth.bass_clip(80 + i, n, SR)).astype(np.float32) if n else np.zeros(0, np.float32)
        if i % 2:
            wavfile.write(str(src), SR, x)   # float WAV
        else:
            save_audio(src, x, SR)           # 16-bit PCM WAV
        pairs.append((src, tmp_path / f"batch{i}.wav"))
    assert process_files(pairs) == len(pairs)
    for i, (src, out) in enumerate(pairs):
        one = tmp_path / f"one{i}.wav"
        process_file_to_file(src, one)
        assert out.read_bytes() == one.read_bytes(), i
