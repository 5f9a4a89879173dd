"""CPU: host logic of ragged batches -- packing, layout validation, per-clip FX replay tables, the C declarations."""
import os
import re

import numpy as np
import pytest

from quantumdistortion_b200 import _lib, tables
from quantumdistortion_b200.pipeline import check_layout, fx_tables, pack_layout

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("itemsize", [4, 2])
def test_pack_layout_aligns_every_start(itemsize):
    lengths = [0, 1, 7, 4, 4099, 0, 3, 16000]
    starts, span = pack_layout(lengths, itemsize)
    align = 16 // itemsize
    assert starts.dtype == np.int64 and starts[0] == 0
    assert np.all(starts % align == 0)
    assert span == starts[-1] + lengths[-1]
    ends = starts + np.asarray(lengths)
    assert np.all(starts[1:] >= ends[:-1])                   # no overlap
    assert np.all(starts[1:] - ends[:-1] < align)            # gaps only for alignment
    check_layout(starts, lengths, max(lengths))


def test_pack_layout_empty_and_negative():
    s, span = pack_layout([])
    assert s.size == 0 and span == 0
    with pytest.raises(ValueError):
        pack_layout([3, -1])


@pytest.mark.parametrize("starts,lengths,why", [
    ([0, 8], [5, 9], "longer than the renderer"),      # max_samples = 8
    ([0, 4], [5, 3], "overlap"),
    ([8, 0], [3, 3], "non-decreasing"),
    ([0, 8], [3, -1], ">= 0"),
])
def test_check_layout_rejects(starts, lengths, why):
    with pytest.raises(ValueError, match=why):
        check_layout(np.array(starts, np.int64), np.array(lengths, np.int32), 8)


def test_check_layout_accepts_gaps_and_empty_clips():
    check_layout(np.array([0, 100, 100, 104]), np.array([3, 0, 4, 8]), 8)


def _resolved(mode, n_samples=20000, n_fft=2048):
    r = tables.resolve(sr=48000, n_samples=n_samples, n_fft=n_fft, key="D", scale="minor", snap_strength=1.0,
                       smear=0.1, bin_smoothing=True, pre_quant=True, post_quant=True, distortion_mode="wavefold",
                       distortion_params={}, limiter_on=True, limiter_ceiling_db=-1.0, dry_wet=1.0, use_multiband=True,
                       crossover_hz=300.0, lowband_drive=1.0, passthrough_test=False, harmonic_lock_hz=0.0,
                       delta_listen=False, mono_strength=1.0, output_trim_db=0.0, low_trim_db=0.0, sub_cut_hz=0.0,
                       air_cut_hz=0.0, spectral_fx_mode=mode, spectral_fx_strength=0.5, spectral_fx_params={},
                       precision="float32", spectral_freeze=False, formant_shift=0.0, no_spectral=False)
    assert r.fx_rng, mode
    return r


@pytest.mark.parametrize("mode", ["bin_scramble", "phase_dispersal"])
@pytest.mark.parametrize("seeds", [None, 7, [3, 1, 4, 1]])
def test_fx_tables_per_clip_frames(mode, seeds):
    """Each clip's table is a single-clip replay over its own frames (padded to the plan's), and the global
    np.random state afterwards is that of a loop of single-clip replays."""
    r = _resolved(mode)
    hop = 512
    lengths = [20000, 1, 5000, 700]
    frames = [1 + n // hop for n in lengths]
    np.random.seed(1234)
    tabs = fx_tables(r, len(lengths), seeds, frames=frames)
    after = np.random.get_state()[1].copy()
    np.random.seed(1234)
    for c, t in enumerate(frames):
        if isinstance(seeds, int):
            np.random.seed(seeds)
        elif seeds is not None:
            np.random.seed(seeds[c])
        one = tables.replay_fx_table(r.fx_rng, r.fx_passes, t, r.n_bins)
        assert tabs[c].shape == (2, r.n_frames, r.n_bins)
        assert np.array_equal(tabs[c][:, :t], one)
    assert np.array_equal(np.random.get_state()[1], after)


def test_fx_tables_ragged_rejects_bad_frames_and_shard():
    r = _resolved("bin_scramble")
    with pytest.raises(ValueError):
        fx_tables(r, 2, None, frames=[1, r.n_frames + 1])
    with pytest.raises(ValueError):
        fx_tables(r, 2, [1], frames=[1, 2])
    with pytest.raises(ValueError):
        fx_tables(r, 2, None, shard=(0, 2, 4), frames=[1, 2])


def test_varlen_symbols_declared():
    header = open(os.path.join(ROOT, "include", "qd_b200.h")).read()
    assert re.search(r"#define QD_ABI_VERSION 6\b", header)
    assert _lib.QD_ABI_VERSION == 6
    src = open(os.path.join(ROOT, "quantumdistortion_b200", "_lib.py")).read()
    for name in ("qd_plan_workspace_bytes_varlen", "qd_render_device_varlen", "qd_render_host_varlen"):
        assert name + "(" in header, name
        assert f"lib.{name}.argtypes" in src, name
    assert "lib.qd_plan_workspace_bytes_varlen.restype = C.c_size_t" in src


def test_process_batch_list_rejects_shard_and_out():
    from quantumdistortion_b200 import process_batch
    clips = [np.zeros(10, np.float32), np.zeros(20, np.float32)]
    with pytest.raises(ValueError, match="shard"):
        process_batch(clips, 48000, shard=(0, 2, 4), quantize_mode="spectral_bins")
    with pytest.raises(ValueError, match="out"):
        process_batch(clips, 48000, out=np.zeros(30, np.float32), quantize_mode="spectral_bins")
