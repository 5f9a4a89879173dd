"""CPU: autotune_v1 kernels on a ragged batch (per-clip starts / lengths, packed with gaps), single-stepped through
tests/emu/cuda_emu.h.  Every clip of the packed batch must come out bit-identical to the same clip run alone through
the uniform path: the YIN difference function (frame rows at floor(start / hop) + clip) and the zero-phase filter
sweeps with a clip short enough to get a halved filter tile next to one that keeps the full tile."""
import os
import subprocess
import tempfile

import numpy as np
import pytest
from scipy.signal import butter, sosfilt_zi

from quantumdistortion_b200.pipeline import pack_layout

HERE = os.path.dirname(os.path.abspath(__file__))
EMU_DIR = os.path.join(HERE, "emu")
CSRC = os.path.join(os.path.dirname(HERE), "quantumdistortion_b200", "csrc")
TIMEOUT = 900


@pytest.fixture(scope="module")
def emu_at():
    exe = os.path.join(tempfile.gettempdir(), f"qd_emu_at_ragged_{os.getuid()}")
    srcs = [os.path.join(EMU_DIR, f) for f in ("emu_at_ragged.cpp", "cuda_emu.h", "cuda_emu_at.h")]
    srcs += [os.path.join(CSRC, f) for f in ("qd_autotune.cuh", "qd_yin.cuh", "qd_common.cuh", "qd_spec.cuh",
                                             "qd_spec_team.cuh", "qd_time.cuh", "qd_host_time.hpp")]
    if not os.path.exists(exe) or any(os.path.getmtime(s) > os.path.getmtime(exe) for s in srcs):
        tmp = f"{exe}.{os.getpid()}"
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-DQD_EMU", "-I", EMU_DIR, "-o", tmp,
                               os.path.join(EMU_DIR, "emu_at_ragged.cpp"), "-lpthread"], timeout=TIMEOUT)
        os.replace(tmp, exe)
    return exe


def _run(cmd):
    subprocess.run(cmd, check=True, timeout=TIMEOUT, stdout=subprocess.DEVNULL)


def _clip(seed, n):
    t = np.arange(n)
    rng = np.random.default_rng(seed)
    return (0.5 * np.sin(2 * np.pi * t / (30.0 + seed)) + 0.1 * rng.standard_normal(n)).astype(np.float32)


def _packed(d, clips, gap_value=7.0):
    """Packed input with wider gaps than the packer's, filled with junk that no kernel may read."""
    lengths = np.array([len(c) for c in clips], dtype=np.int64)
    starts, _ = pack_layout(lengths, 4)
    starts = starts + 3 * np.arange(len(clips), dtype=np.int64) * 4
    span = int(starts[-1] + lengths[-1])
    x = np.full(span, gap_value, dtype=np.float32)
    for s, c in zip(starts, clips):
        x[s:s + len(c)] = c
    x.tofile(os.path.join(d, "x"))
    starts.tofile(os.path.join(d, "starts"))
    lengths.astype(np.int32).tofile(os.path.join(d, "lengths"))
    return starts, lengths


def test_emu_ragged_yin_difference_function(emu_at):
    frame, hop, max_tau, cols = 512, 64, 100, 3    # two lag CTAs per clip
    stride = (max_tau + 2) & ~1
    clips = [_clip(i, n) for i, n in enumerate([1500, 0, 63, 700, 65, 1023])]
    with tempfile.TemporaryDirectory() as d:
        starts, lengths = _packed(d, clips)
        _run([emu_at, "yin", str(frame), str(hop), str(max_tau), str(cols), os.path.join(d, "x"),
              os.path.join(d, "starts"), os.path.join(d, "lengths"), os.path.join(d, "diff")])
        got = np.fromfile(os.path.join(d, "diff")).reshape(-1, stride)
        for i, c in enumerate(clips):
            frames = -(-len(c) // hop)
            if frames == 0:
                continue
            c.tofile(os.path.join(d, "one"))
            _run([emu_at, "yin", str(frame), str(hop), str(max_tau), str(cols), os.path.join(d, "one"), "-", "-",
                  os.path.join(d, "ref")])
            ref = np.fromfile(os.path.join(d, "ref")).reshape(-1, stride)[:frames, 1:max_tau + 1]
            r0 = int((starts[i] - starts[0]) // hop) + i
            assert (ref >= 0).all()
            assert np.array_equal(got[r0:r0 + frames, 1:max_tau + 1], ref), (i, len(c))


def _bank(sr, cutoffs):
    sos, zi = [], []
    for hz, btype in cutoffs:
        s = butter(4, hz / (sr / 2.0), btype=btype, output="sos")
        sos.append(s)
        zi.append(sosfilt_zi(s))
    return np.array(sos, np.float64), np.array(zi, np.float64)


def _tile_of(sos):
    """qd_host::segment_tiling: the warm-up and the full tile of a filter, from its largest pole radius."""
    r = 0.0
    for a1, a2 in sos[:, 4:6]:
        disc = a1 * a1 - 4 * a2
        r = max(r, np.sqrt(max(a2, 0)) if disc < 0 else max(abs((-a1 + np.sqrt(disc)) / 2), abs((-a1 - np.sqrt(disc)) / 2)))
    halo = (int(np.ceil(44.0 / (1.0 - r))) + 31) & ~31
    t = 4096
    while t < 2 * halo:
        t *= 2
    return t, halo


def _halved(tile, halo, m):
    """qd::at_filt_tile"""
    while tile // 2 >= max(4096, halo) and -(-m // tile) < 32:
        tile //= 2
    return tile


def test_emu_ragged_filter_sweeps_per_clip_tile(emu_at):
    """A 400 Hz high-pass at 48 kHz warms up over 2240 samples: full tile 8192, halved to 4096 while a clip has fewer
    than 32 tiles.  The 262000-sample clip keeps 8192, the shorter ones get 4096, in one launch; the 5 kHz low-pass
    keeps 4096 everywhere.  Both sweeps, bit for bit against each clip alone."""
    sos, zi = _bank(48000, [(400.0, "high"), (5000.0, "low")])
    lengths = [70000, 16, 262000, 0, 20000, 4097]
    tile, halo = _tile_of(sos[0])
    assert tile == 8192 and _halved(tile, halo, 262000 + 30) == 8192 and _halved(tile, halo, 70000 + 30) == 4096
    clips = [_clip(10 + i, n) for i, n in enumerate(lengths)]
    with tempfile.TemporaryDirectory() as d:
        sos.tofile(os.path.join(d, "sos"))
        zi.tofile(os.path.join(d, "zi"))
        starts, _ = _packed(d, clips)
        _run([emu_at, "filt", os.path.join(d, "sos"), os.path.join(d, "zi"), os.path.join(d, "x"),
              os.path.join(d, "starts"), os.path.join(d, "lengths"), os.path.join(d, "y")])
        got = np.fromfile(os.path.join(d, "y"), dtype=np.float32).reshape(2, -1)
        for i, c in enumerate(clips):
            if len(c) == 0:
                continue
            c.tofile(os.path.join(d, "one"))
            _run([emu_at, "filt", os.path.join(d, "sos"), os.path.join(d, "zi"), os.path.join(d, "one"), "-", "-",
                  os.path.join(d, "ref")])
            ref = np.fromfile(os.path.join(d, "ref"), dtype=np.float32).reshape(2, -1)
            o = int(starts[i] - starts[0])
            for j in range(2):
                assert np.array_equal(got[j, o:o + len(c)], ref[j]), (i, j, len(c))
