"""CPU: launch splits, single-stepped through tests/emu/cuda_emu.h.  The library cuts a batch into launches at the grid
limit (qd::for_each_launch, 65 535 clips on gridDim.y); every launch advances the clip index clip0, for uniform and
ragged batches alike.  Real batches that reach the limit are too large for the emulator, so the drivers split small
batches into launches of 1, 2 and 3 clips (2, 4 and 6 for the two-group spectral kernel) through the same helper, and
every output must be bit-identical to one launch: samples, the spectral pass's per-clip peaks, and the per-clip tables
of the autotune_v1 stages.  Gaps between ragged clips and rows no clip owns keep their fill value."""
import os
import subprocess
import tempfile

import numpy as np
import pytest
from scipy.signal import butter, sosfilt_zi

from oracle import qd_oracle as orc
from quantumdistortion_b200 import synth
from quantumdistortion_b200.pipeline import pack_layout

HERE = os.path.dirname(os.path.abspath(__file__))
EMU_DIR = os.path.join(HERE, "emu")
CSRC = os.path.join(os.path.dirname(HERE), "quantumdistortion_b200", "csrc")
TIMEOUT = 900
FILL = -777.0   # emu_ragged's initial output value
AT_FILL = -7.0  # emu_at_ragged's


def _build(name, src, headers):
    exe = os.path.join(tempfile.gettempdir(), f"qd_{name}_{os.getuid()}")
    srcs = [os.path.join(EMU_DIR, f) for f in (src, "cuda_emu.h", "cuda_emu_at.h")]
    srcs += [os.path.join(CSRC, f) for f in headers]
    if not os.path.exists(exe) or any(os.path.getmtime(s) > os.path.getmtime(exe) for s in srcs):
        tmp = f"{exe}.{os.getpid()}"
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-DQD_EMU", "-I", EMU_DIR, "-o", tmp,
                               os.path.join(EMU_DIR, src), "-lpthread"], timeout=TIMEOUT)
        os.replace(tmp, exe)
    return exe


@pytest.fixture(scope="module")
def emu_ragged():
    return _build("emu_ragged", "emu_ragged.cpp", ("qd_spec.cuh", "qd_spec_team.cuh", "qd_common.cuh",
                                                    "qd_host_tables.hpp", "qd_time.cuh", "qd_host_time.hpp"))


@pytest.fixture(scope="module")
def emu_at():
    return _build("emu_at_ragged", "emu_at_ragged.cpp", ("qd_autotune.cuh", "qd_yin.cuh", "qd_common.cuh",
                                                          "qd_spec.cuh", "qd_time.cuh", "qd_host_time.hpp"))


def _run(cmd):
    subprocess.run(cmd, check=True, timeout=TIMEOUT, stdout=subprocess.DEVNULL)


def _synth(fn, seed, n, gain=1.0):
    return (gain * fn(seed, n)).astype(np.float32) if n else np.zeros(0, np.float32)


class Batch:
    """x and the layout arguments of a uniform batch ("u<B>", B clips of n samples) or of a ragged one packed with gaps
    (filled with junk that no kernel may read).  The same clips in the same order either way."""

    def __init__(self, d, clips, ragged, name="x"):
        self.d, self.ragged = d, ragged
        self.lengths = np.array([len(c) for c in clips], dtype=np.int64)
        if ragged:
            starts, _ = pack_layout(self.lengths, 4)
            self.starts = starts + 3 * np.arange(len(clips), dtype=np.int64) * 4
        else:
            assert len(set(self.lengths)) == 1
            self.starts = np.arange(len(clips), dtype=np.int64) * self.lengths[0]
        span = int(self.starts[-1] + self.lengths[-1])
        x = np.full(span, 7.0, dtype=np.float32)
        for s, c in zip(self.starts, clips):
            x[s:s + len(c)] = c
        self.x = self.path(name)
        x.tofile(self.x)
        if ragged:
            self.starts.tofile(self.path("starts"))
            self.lengths.astype(np.int32).tofile(self.path("lengths"))
            self.layout = [self.path("starts"), self.path("lengths")]
        else:
            self.layout = ["u%d" % len(clips), "-"]

    def path(self, f):
        return os.path.join(self.d, f)

    def gaps(self, n):
        """mask of the samples of an n-sample buffer that no clip owns"""
        m = np.ones(n, bool)
        for s, k in zip(self.starts, self.lengths):
            m[s:s + k] = False
        return m


def _splits(exe, batch, cmd, outputs, per_launch=(1, 2, 3), dtypes=None):
    """Run cmd (output files "@<name>" for each name of `outputs`) in one launch and split into launches of
    per_launch clips; every output must match the single launch bit for bit.  Returns the single launch's outputs."""
    dtypes = dtypes or [np.float32] * len(outputs)

    def go(opt, tag):
        paths = [batch.path(o + tag) for o in outputs]
        _run([exe] + opt + [paths[outputs.index(a[1:])] if a[:1] == "@" else a for a in cmd])
        return [np.fromfile(p, dtype=t) for p, t in zip(paths, dtypes)]

    ref = go([], "_one")
    for k in per_launch:
        got = go(["-p", str(k)], "_p%d" % k)
        for name, g, r in zip(outputs, got, ref):
            assert np.array_equal(g, r), (k, name)
    return ref


# ------------------------------------------------------------------------------------------------ spectral pass
def _quant_tables(d, n_fft, sr=48000):
    freqs = np.fft.rfftfreq(n_fft, d=1.0 / sr)
    orc.target_bins_for_freqs(freqs, "D", "minor").astype(np.int32).tofile(os.path.join(d, "tb"))
    orc.quantize_band_mask(freqs, 110.0, 5000.0).astype(np.uint8).tofile(os.path.join(d, "mask"))


# (name, prec, n_fft, nw, tile, options, clips per launch, uniform n, ragged lengths).  nw = 16 is the NG = 2 kernel of
# the headline shape: splits in whole CTA rows.  -x: the FX kernel with per-clip scramble tables and the spectral freeze.
SPEC_CASES = [
    ("ng2", "f32", 2048, 16, 3, [], (2, 4, 6), 2500, [9000, 700, 0, 5003, 1, 2500, 640]),
    ("ng1", "f32", 1024, 4, 5, [], (1, 2, 3), 1500, [3000, 1, 0, 1500, 257]),
    ("fx", "f32", 1024, 4, 5, ["-x"], (1, 2, 3), 1500, [3000, 1, 0, 1500, 257]),
    ("team", "f32", 1024, 801, 4, [], (1, 2, 3), 2000, [2500, 0, 333, 4100]),
]


@pytest.mark.parametrize("ragged", [False, True], ids=["uniform", "ragged"])
@pytest.mark.parametrize("name,prec,n_fft,nw,tile,opts,per,n,lengths", SPEC_CASES, ids=[c[0] for c in SPEC_CASES])
def test_emu_split_spec(emu_ragged, ragged, name, prec, n_fft, nw, tile, opts, per, n, lengths):
    lengths = lengths if ragged else [n] * 5
    clips = [_synth(synth.bass_clip, i, k, 0.5) for i, k in enumerate(lengths)]
    with tempfile.TemporaryDirectory() as d:
        _quant_tables(d, n_fft)
        b = Batch(d, clips, ragged)
        cmd = opts + ["spec", prec, str(n_fft), str(nw), str(tile), "1", b.x] + b.layout + [b.path("tb"), b.path("mask"), "@y"]
        y, = _splits(emu_ragged, b, cmd, ["y"], per)
        ref_peak = np.fromfile(b.path("y_one.peak"), np.float32)
        for k in per:
            assert np.array_equal(np.fromfile(b.path("y_p%d.peak" % k), np.float32), ref_peak), k
        assert np.all(y[b.gaps(len(y))] == FILL)
        assert np.all(ref_peak[len(clips):] == 0.0)   # rows no clip owns
        for i, (s, k) in enumerate(zip(b.starts, b.lengths)):   # the peak of each clip is its own
            assert ref_peak[i] == (np.max(np.abs(y[s:s + k])) if k else 0.0), i


# ------------------------------------------------------------------------------------------------ limiter, crossover
@pytest.mark.parametrize("ragged", [False, True], ids=["uniform", "ragged"])
def test_emu_split_limiter_clip_peak(emu_ragged, ragged):
    """-q: per-clip peaks mark the odd clips quiet, so a peak read at the wrong clip changes the output."""
    _, L, _ = orc.limiter_constants(48000, -1.0, 5.0, 30.0)
    lengths = [6000, 0, 2049, 13, 5000] if ragged else [3000] * 5
    clips = [_synth(synth.noise_clip, i + 1, k, 2.0) for i, k in enumerate(lengths)]
    with tempfile.TemporaryDirectory() as d:
        b = Batch(d, clips, ragged)
        y, = _splits(emu_ragged, b, ["-q", "limiter", str(L), b.x] + b.layout + ["@y"], ["y"])
        assert np.all(y[b.gaps(len(y))] == FILL)
        for i, (s, k) in enumerate(zip(b.starts, b.lengths)):
            if k > 100:   # quiet clips pass through, loud ones are limited
                assert np.array_equal(y[s:s + k], clips[i]) == (i % 2 == 1), i


@pytest.mark.parametrize("ragged", [False, True], ids=["uniform", "ragged"])
def test_emu_split_crossover(emu_ragged, ragged):
    lengths = [6000, 100, 0, 5003, 1500] if ragged else [2000] * 5
    clips = [_synth(synth.loud_clip, i + 3, k) for i, k in enumerate(lengths)]
    sl, sh = orc.linkwitz_riley_sos(48000, 300.0)
    with tempfile.TemporaryDirectory() as d:
        sl.astype(np.float64).tofile(os.path.join(d, "lp"))
        sh.astype(np.float64).tofile(os.path.join(d, "hp"))
        b = Batch(d, clips, ragged)
        cmd = ["crossover", "300", b.path("lp"), b.path("hp"), "256", "1632", b.x] + b.layout + ["@lo", "@hi"]
        for out in _splits(emu_ragged, b, cmd, ["lo", "hi"]):
            assert np.all(out[b.gaps(len(out))] == FILL)


# ------------------------------------------------------------------------------------------------ autotune_v1
HOP = 512


def _clip(seed, n):
    t = np.arange(n)
    rng = np.random.default_rng(seed)
    return (0.5 * np.sin(2 * np.pi * t / (30.0 + seed)) + 0.1 * rng.standard_normal(n)).astype(np.float32)


def _at_batch(d, ragged, lengths, uniform_n, seed, name="x"):
    lengths = lengths if ragged else [uniform_n] * 5
    return Batch(d, [_clip(seed + i, k) for i, k in enumerate(lengths)], ragged, name), lengths


def _rows(b, unit):
    span = int(b.starts[-1] - b.starts[0] + b.lengths[-1])
    return span // unit + len(b.lengths) if b.ragged else len(b.lengths) * -(-int(b.lengths[0]) // unit)


@pytest.mark.parametrize("ragged", [False, True], ids=["uniform", "ragged"])
def test_emu_split_at_filters(emu_at, ragged):
    sos, zi = [], []
    for hz, btype in [(400.0, "high"), (5000.0, "low")]:
        s = butter(4, hz / 24000.0, btype=btype, output="sos")
        sos.append(s)
        zi.append(sosfilt_zi(s))
    with tempfile.TemporaryDirectory() as d:
        np.array(sos, np.float64).tofile(os.path.join(d, "sos"))
        np.array(zi, np.float64).tofile(os.path.join(d, "zi"))
        b, _ = _at_batch(d, ragged, [9000, 16, 0, 5000, 4097], 3000, 10)
        y, = _splits(emu_at, b, ["filt", b.path("sos"), b.path("zi"), b.x] + b.layout + ["@y"], ["y"])
        y = y.reshape(2, -1)
        assert np.all(y[:, b.gaps(y.shape[1])] == 0.0)


@pytest.mark.parametrize("ragged", [False, True], ids=["uniform", "ragged"])
def test_emu_split_at_yin_walk(emu_at, ragged):
    with tempfile.TemporaryDirectory() as d:
        b, _ = _at_batch(d, ragged, [1500, 0, 63, 700, 65], 700, 0)
        diff, = _splits(emu_at, b, ["yin", "512", "64", "100", "3", b.x] + b.layout + ["@diff"], ["diff"],
                        dtypes=[np.float64])
        assert len(diff) == _rows(b, 64) * 102


@pytest.mark.parametrize("ragged", [False, True], ids=["uniform", "ragged"])
def test_emu_split_at_shifter(emu_at, ragged):
    with tempfile.TemporaryDirectory() as d:
        b, lengths = _at_batch(d, ragged, [9000, 0, 1, 513, 4097], 2049, 40, "body")
        np.exp(np.random.default_rng(5).uniform(np.log(0.5), np.log(2.0), _rows(b, HOP))).tofile(b.path("ratio"))
        cmd = ["shift", str(HOP), "2048", "1024", "4096", b.x] + b.layout + [b.path("ratio"), "@out", "@track", "@flag"]
        out, track, _ = _splits(emu_at, b, cmd, ["out", "track", "flag"], dtypes=[np.float32, np.float32, np.int32])
        for v in (out, track):
            assert np.all(v[b.gaps(len(v))] == AT_FILL)


# a fast envelope (halo 4608 samples) so that the segment follower (clips of at least seg_min = 4 tiles) runs on clips
# the emulator renders quickly
ENV = [repr(float(np.float32(0.99))), repr(float(np.float32(0.995))), "1024", "4608", "4096"]


@pytest.mark.parametrize("ragged", [False, True], ids=["uniform", "ragged"])
def test_emu_split_at_envelope(emu_at, ragged):
    with tempfile.TemporaryDirectory() as d:
        b, _ = _at_batch(d, ragged, [9000, 0, 1, 4096, 5000], 6000, 60)
        env, emax = _splits(emu_at, b, ["env", *ENV, b.x] + b.layout + ["@env", "@emax"], ["env", "emax"])
        assert np.all(env[b.gaps(len(env))] == AT_FILL)
        assert np.all(emax >= 0.0)


@pytest.mark.parametrize("ragged", [False, True], ids=["uniform", "ragged"])
def test_emu_split_at_mix(emu_at, ragged):
    with tempfile.TemporaryDirectory() as d:
        b, lengths = _at_batch(d, ragged, [9000, 0, 1, 4096, 5000], 6000, 80)
        rng = np.random.default_rng(9)
        for name in ("sub", "air", "corr"):
            Batch(d, [(rng.standard_normal(k) * 0.3).astype(np.float32) for k in lengths], ragged, name)
        mix = ["1", "1", *ENV[:2], *ENV[2:], repr(float(np.float32(0.35))), repr(float(np.float32(0.15))), "1.0",
               repr(float(np.float32(2 * np.pi * 73.41619197935188))), "48000.0"]
        cmd = ["mix", *mix, b.x, b.path("sub"), b.path("air"), b.path("corr")] + b.layout + ["@y", "@layer"]
        for out in _splits(emu_at, b, cmd, ["y", "layer"]):
            assert np.all(out[b.gaps(len(out))] == AT_FILL)
