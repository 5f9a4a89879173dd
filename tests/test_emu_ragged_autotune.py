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


# ------------------------------------------------------------------------------------------------ the later stages
# Each stage on a packed batch next to the same clip alone, bit for bit: clips of 0, 1, 511 and 513 samples, and the
# per-clip tables (frame rows at floor(start / hop) + clip, tap tiles at floor(start / 512) + clip) with junk in every
# row and sample that no clip owns.
HOP = 512
RAGGED = [4097, 0, 1, 511, 513, 9000, 2049]


def _rows(starts, lengths, unit):
    span = int(starts[-1] - starts[0] + lengths[-1])
    return span // unit + len(lengths), [int((s - starts[0]) // unit) + i for i, s in enumerate(starts)]


def _gaps_untouched(got, starts, lengths, fill):
    mask = np.ones(len(got), bool)
    for s, n in zip(starts - starts[0], lengths):
        mask[s:s + n] = False
    assert (got[mask] == fill).all()


def test_emu_ragged_frame_stats(emu_at):
    clips = [_clip(20 + i, n) for i, n in enumerate(RAGGED)]
    clips[5][3000:] = 0.0                                         # silent frames at a clip's end
    with tempfile.TemporaryDirectory() as d:
        starts, lengths = _packed(d, clips)
        _run([emu_at, "stats", str(HOP), "16", "671", os.path.join(d, "x"), os.path.join(d, "starts"),
              os.path.join(d, "lengths"), os.path.join(d, "feat")])
        got = np.fromfile(os.path.join(d, "feat")).reshape(-1, 4)
        _, r0 = _rows(starts, lengths, HOP)
        for i, c in enumerate(clips):
            if len(c) == 0:
                continue
            c.tofile(os.path.join(d, "one"))
            _run([emu_at, "stats", str(HOP), "16", "671", os.path.join(d, "one"), "-", "-", os.path.join(d, "ref")])
            ref = np.fromfile(os.path.join(d, "ref")).reshape(-1, 4)
            assert np.array_equal(got[r0[i]:r0[i] + len(ref)], ref), (i, len(c))


def _hold_cmd(emu_at, d, n, feat, starts="-", lengths="-"):
    feat.tofile(os.path.join(d, "feat"))
    _run([emu_at, "hold", str(n), str(HOP), "2", "0,2,3,5,7,8,10", "0.8", "0.01", "0.55", "0.72", "40.0", "3", "2",
          os.path.join(d, "feat"), starts, lengths, os.path.join(d, "ratio")])
    return np.fromfile(os.path.join(d, "ratio"))


def _features(seed, frames):
    rng = np.random.default_rng(seed)
    notes = rng.choice([110.0, 147.0, 233.0, 440.0, 460.0, 700.0], frames)
    pitch = notes * 2 ** (rng.uniform(-10, 10, frames) / 1200) * (rng.uniform(0, 1, frames) > 0.15)
    return np.stack([rng.uniform(0.005, 0.2, frames), rng.uniform(0.1, 0.6, frames), pitch,
                     rng.uniform(0.6, 1.0, frames)], axis=1)


def test_emu_ragged_note_hold(emu_at):
    lengths = np.array([30000, 0, 1, 511, 513, 70000, 2049], dtype=np.int64)
    with tempfile.TemporaryDirectory() as d:
        starts, _ = _packed(d, [np.zeros(n, np.float32) for n in lengths])
        rows, r0 = _rows(starts, lengths, HOP)
        feat = np.tile([0.1, 0.1, 300.0, 0.9], (rows, 1))          # voiced junk in the rows no clip owns
        per = [_features(i, -(-int(n) // HOP)) for i, n in enumerate(lengths)]
        for i, f in enumerate(per):
            feat[r0[i]:r0[i] + len(f)] = f
        got = _hold_cmd(emu_at, d, 0, feat, os.path.join(d, "starts"), os.path.join(d, "lengths"))
        for i, f in enumerate(per):
            if len(f) == 0:
                continue
            ref = _hold_cmd(emu_at, d, int(lengths[i]), f)
            assert np.array_equal(got[r0[i]:r0[i] + len(f)], ref), (i, int(lengths[i]))


def test_emu_ragged_shifter(emu_at):
    lengths = [9000, 0, 1, 511, 513, 4097, 2049, 6000]
    clips = [_clip(40 + i, n) for i, n in enumerate(lengths)]
    rng = np.random.default_rng(5)
    with tempfile.TemporaryDirectory() as d:
        starts, lens = _packed(d, clips)
        rows, r0 = _rows(starts, lens, HOP)
        ratio = np.full(rows, 1.7)
        per = []
        for i, n in enumerate(lengths):
            r = np.exp(rng.uniform(np.log(0.5), np.log(2.0), -(-n // HOP)))
            if i == 7:
                r = 1.0 + rng.uniform(-5e-4, 5e-4, len(r))          # a flat clip next to shifted ones
            ratio[r0[i]:r0[i] + len(r)] = r
            per.append(r)
        os.rename(os.path.join(d, "x"), os.path.join(d, "body"))
        ratio.tofile(os.path.join(d, "ratio"))
        args = [str(HOP), "2048", "1024", "4096"]
        _run([emu_at, "shift", *args, os.path.join(d, "body"), os.path.join(d, "starts"), os.path.join(d, "lengths"),
              os.path.join(d, "ratio"), os.path.join(d, "out"), os.path.join(d, "track"), os.path.join(d, "flag")])
        out = np.fromfile(os.path.join(d, "out"), np.float32)
        track = np.fromfile(os.path.join(d, "track"), np.float32)
        flag = np.fromfile(os.path.join(d, "flag"), np.int32)
        _gaps_untouched(out, starts, lens, -7.0)
        _gaps_untouched(track, starts, lens, -7.0)
        assert list(flag) == [0, 1, 0, 0, 0, 0, 0, 1]
        for i, c in enumerate(clips):
            if len(c) == 0:
                continue
            c.tofile(os.path.join(d, "one"))
            per[i].tofile(os.path.join(d, "r1"))
            _run([emu_at, "shift", *args, os.path.join(d, "one"), "-", "-", os.path.join(d, "r1"),
                  os.path.join(d, "o1"), os.path.join(d, "t1"), os.path.join(d, "f1")])
            o = int(starts[i] - starts[0])
            assert np.array_equal(out[o:o + len(c)], np.fromfile(os.path.join(d, "o1"), np.float32)), (i, len(c))
            assert np.array_equal(track[o:o + len(c)], np.fromfile(os.path.join(d, "t1"), np.float32)), (i, len(c))
            assert flag[i] == np.fromfile(os.path.join(d, "f1"), np.int32)[0]


ENV_LENGTHS = [70000, 0, 1, 511, 513, 3000]        # 70000: the segment follower (>= 65536 at 48 kHz), the rest one warp


def _env_args():
    att = float(np.float32(np.exp(-1.0 / (8.0 * 0.001 * 48000))))
    rel = float(np.float32(np.exp(-1.0 / (90.0 * 0.001 * 48000))))
    halo = (int(np.ceil(np.log(1e-10) / np.log(max(att, rel)))) + 31) // 32 * 32
    return [repr(att), repr(rel), "16384", str(halo), str(4 * 16384)]


def test_emu_ragged_envelope(emu_at):
    clips = [_clip(60 + i, n) for i, n in enumerate(ENV_LENGTHS)]
    with tempfile.TemporaryDirectory() as d:
        starts, lens = _packed(d, clips)
        _run([emu_at, "env", *_env_args(), os.path.join(d, "x"), os.path.join(d, "starts"), os.path.join(d, "lengths"),
              os.path.join(d, "env"), os.path.join(d, "emax")])
        env = np.fromfile(os.path.join(d, "env"), np.float32)
        emax = np.fromfile(os.path.join(d, "emax"), np.float32)
        _gaps_untouched(env, starts, lens, -7.0)
        assert emax[1] == 0.0
        for i, c in enumerate(clips):
            if len(c) == 0:
                continue
            c.tofile(os.path.join(d, "one"))
            _run([emu_at, "env", *_env_args(), os.path.join(d, "one"), "-", "-", os.path.join(d, "e1"), os.path.join(d, "m1")])
            o = int(starts[i] - starts[0])
            assert np.array_equal(env[o:o + len(c)], np.fromfile(os.path.join(d, "e1"), np.float32)), (i, len(c))
            assert emax[i] == np.fromfile(os.path.join(d, "m1"), np.float32)[0], i


def test_emu_ragged_mix(emu_at):
    clips = [_clip(80 + i, n) for i, n in enumerate(ENV_LENGTHS)]
    rng = np.random.default_rng(9)
    bands = [(rng.standard_normal((3, len(c))) * 0.3).astype(np.float32) for c in clips]
    env = _env_args()
    mix = ["1", "1", env[0], env[1], env[2], env[3], env[4], repr(float(np.float32(0.35))),
           repr(float(np.float32(0.15))), "1.0", repr(float(np.float32(2 * np.pi * 73.41619197935188))), "48000.0"]
    with tempfile.TemporaryDirectory() as d:
        starts, lens = _packed(d, clips)
        for k, name in enumerate(("sub", "air", "corr")):
            _packed(d, [b[k] for b in bands])
            os.rename(os.path.join(d, "x"), os.path.join(d, name))
        _packed(d, clips)
        files = [os.path.join(d, k) for k in ("x", "sub", "air", "corr")]
        _run([emu_at, "mix", *mix, *files, os.path.join(d, "starts"), os.path.join(d, "lengths"), os.path.join(d, "y"),
              os.path.join(d, "layer")])
        y = np.fromfile(os.path.join(d, "y"), np.float32)
        layer = np.fromfile(os.path.join(d, "layer"), np.float32)
        _gaps_untouched(y, starts, lens, -7.0)
        for i, c in enumerate(clips):
            if len(c) == 0:
                continue
            one = [os.path.join(d, k + "1") for k in ("x", "sub", "air", "corr")]
            for f, v in zip(one, [c, *bands[i]]):
                v.tofile(f)
            _run([emu_at, "mix", *mix, *one, "-", "-", os.path.join(d, "y1"), os.path.join(d, "l1")])
            o = int(starts[i] - starts[0])
            assert np.array_equal(y[o:o + len(c)], np.fromfile(os.path.join(d, "y1"), np.float32)), (i, len(c))
            assert np.array_equal(layer[o:o + len(c)], np.fromfile(os.path.join(d, "l1"), np.float32)), (i, len(c))
