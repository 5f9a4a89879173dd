"""CPU: the kernels of a ragged batch (per-clip starts / lengths, packed with gaps), single-stepped through
tests/emu/cuda_emu.h.  Every clip of the packed batch must come out bit-identical to the same clip run alone through
the uniform path.  cuda_emu.h implements barriers with pthread barriers, so a clip group that returned before a
CTA-wide barrier shows up as a hang: every emulator run has a timeout, which turns that into a failure."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

from oracle import qd_oracle as orc
from quantumdistortion_b200 import synth
from quantumdistortion_b200.pipeline import pack_layout

HERE = os.path.dirname(os.path.abspath(__file__))
EMU_DIR = os.path.join(HERE, "emu")
CSRC = os.path.join(os.path.dirname(HERE), "quantumdistortion_b200", "csrc")
TIMEOUT = 600


@pytest.fixture(scope="module")
def emu_ragged():
    exe = os.path.join(tempfile.gettempdir(), f"qd_emu_ragged_{os.getuid()}")
    srcs = [os.path.join(EMU_DIR, f) for f in ("emu_ragged.cpp", "cuda_emu.h")]
    srcs += [os.path.join(CSRC, f) for f in ("qd_spec.cuh", "qd_spec_team.cuh", "qd_common.cuh", "qd_host_tables.hpp",
                                             "qd_time.cuh", "qd_host_time.hpp")]
    if not os.path.exists(exe) or any(os.path.getmtime(s) > os.path.getmtime(exe) for s in srcs):
        tmp = f"{exe}.{os.getpid()}"
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-DQD_EMU", "-I", EMU_DIR, "-o", tmp,
                               os.path.join(EMU_DIR, "emu_ragged.cpp"), "-lpthread"], timeout=TIMEOUT)
        os.replace(tmp, exe)
    return exe


def _clips(lengths, seed=0):
    return [(0.5 * synth.bass_clip(seed + i, n) if n else np.zeros(0, np.float32)).astype(np.float32)
            for i, n in enumerate(lengths)]


def _run(cmd):
    subprocess.run(cmd, check=True, timeout=TIMEOUT, stdout=subprocess.DEVNULL)


def _packed(d, clips, gap_value=7.0):
    """Write the packed input (gaps filled with junk: a kernel must never read them) and the layout files."""
    lengths = np.array([len(c) for c in clips], dtype=np.int64)
    starts, span = pack_layout(lengths, 4)
    starts = starts + 3 * np.arange(len(clips), dtype=np.int64) * 4   # wider gaps than the packer's, still aligned
    span = int(starts[-1] + lengths[-1])
    x = np.full(span, gap_value, dtype=np.float32)
    for s, c in zip(starts, clips):
        x[s:s + len(c)] = c
    x.tofile(os.path.join(d, "x"))
    starts.astype(np.int64).tofile(os.path.join(d, "starts"))
    lengths.astype(np.int32).tofile(os.path.join(d, "lengths"))
    return starts, lengths


def _quant_tables(d, n_fft, sr=48000):
    freqs = np.fft.rfftfreq(n_fft, d=1.0 / sr)
    orc.target_bins_for_freqs(freqs, "D", "minor").astype(np.int32).tofile(os.path.join(d, "tb"))
    orc.quantize_band_mask(freqs, 110.0, 5000.0).astype(np.uint8).tofile(os.path.join(d, "mask"))


def _spec(exe, d, prec, n_fft, nw, tile, quant, x_path, layout):
    p = lambda f: os.path.join(d, f)  # noqa: E731
    out = p("y_%d" % np.random.randint(1 << 30))
    _run([exe, "spec", prec, str(n_fft), str(nw), str(tile), str(quant), x_path] + layout +
         [p("tb"), p("mask"), out])
    return np.fromfile(out, dtype=np.float32)


# (prec, n_fft, nw, tile, lengths).  nw = 16 is the NG = 2 kernel: CTA y-rows pair clips (0,1), (2,3), ...  With tile
# 3 the pair (9000, 700) has tiles where only the long clip works, the pair (0, 5003) has a group with no tile at all,
# and the last CTA has an empty second group.
SPEC_CASES = [
    ("f32", 2048, 16, 3, [9000, 700, 0, 5003, 1]),
    ("f32", 2048, 16, 64, [700, 6001, 511, 3]),
    ("f32", 1024, 4, 5, [3000, 1, 0, 1500, 257]),
    ("f32", 1024, 801, 4, [2500, 0, 333, 4100]),     # team kernel, one warp per frame
    ("f32", 4096, 202, 2, [9000, 1025, 0, 6000]),    # team kernel, two warps per frame
    ("f64", 1024, 4, 64, [1999, 0, 260]),
]


@pytest.mark.parametrize("prec,n_fft,nw,tile,lengths", SPEC_CASES)
def test_emu_ragged_spec(emu_ragged, prec, n_fft, nw, tile, lengths):
    clips = _clips(lengths)
    with tempfile.TemporaryDirectory() as d:
        p = lambda f: os.path.join(d, f)  # noqa: E731
        _quant_tables(d, n_fft)
        starts, lens = _packed(d, clips)
        y = _spec(emu_ragged, d, prec, n_fft, nw, tile, 1, p("x"), [p("starts"), p("lengths")])
        for i, c in enumerate(clips):
            got = y[starts[i]:starts[i] + lens[i]]
            if len(c) == 0:
                continue
            c.tofile(p("xc"))
            alone = _spec(emu_ragged, d, prec, n_fft, nw, tile, 1, p("xc"), ["-", "-"])
            assert np.array_equal(got, alone), (i, lens[i], float(np.max(np.abs(got - alone))))
        # the gaps between clips are not written by the spectral pass
        covered = np.zeros(len(y), bool)
        for s, n in zip(starts, lens):
            covered[s:s + n] = True
        assert np.all(y[~covered] == -777.0)


def test_emu_ragged_limiter(emu_ragged):
    ceiling, L, c = orc.limiter_constants(48000, -1.0, 5.0, 30.0)
    clips = [(2.0 * synth.noise_clip(i + 1, n)).astype(np.float32) if n else np.zeros(0, np.float32)
             for i, n in enumerate([6000, 0, 2049, 13, 5000])]
    with tempfile.TemporaryDirectory() as d:
        p = lambda f: os.path.join(d, f)  # noqa: E731
        starts, lens = _packed(d, clips)
        _run([emu_ragged, "limiter", str(L), p("x"), p("starts"), p("lengths"), p("y")])
        y = np.fromfile(p("y"), dtype=np.float32)
        for i, cl in enumerate(clips):
            if len(cl) == 0:
                continue
            cl.tofile(p("xc"))
            _run([emu_ragged, "limiter", str(L), p("xc"), "-", "-", p("yc")])
            alone = np.fromfile(p("yc"), dtype=np.float32)
            assert np.max(np.abs(alone - cl)) > 1e-3 or len(cl) < 100, "limiter must engage"
            assert np.array_equal(y[starts[i]:starts[i] + lens[i]], alone), i


@pytest.mark.parametrize("delay,tiling", [(1024, (256, 1632)), (0, (32, 1632)), (300, (512, 2048))])
def test_emu_ragged_crossover(emu_ragged, delay, tiling):
    clips = [synth.loud_clip(i + 3, n) if n else np.zeros(0, np.float32) for i, n in enumerate([6000, 100, 0, 5003, 1500])]
    clips = [c.astype(np.float32) for c in clips]
    sl, sh = orc.linkwitz_riley_sos(48000, 300.0)
    with tempfile.TemporaryDirectory() as d:
        p = lambda f: os.path.join(d, f)  # noqa: E731
        sl.astype(np.float64).tofile(p("lp"))
        sh.astype(np.float64).tofile(p("hp"))
        starts, lens = _packed(d, clips)
        head = [emu_ragged, "crossover", str(delay), p("lp"), p("hp"), str(tiling[0]), str(tiling[1])]
        _run(head + [p("x"), p("starts"), p("lengths"), p("lo"), p("hi")])
        lo, hi = np.fromfile(p("lo"), dtype=np.float32), np.fromfile(p("hi"), dtype=np.float32)
        for i, cl in enumerate(clips):
            if len(cl) == 0:
                continue
            cl.tofile(p("xc"))
            _run(head + [p("xc"), "-", "-", p("loc"), p("hic")])
            s, n = starts[i], lens[i]
            assert np.array_equal(lo[s:s + n], np.fromfile(p("loc"), dtype=np.float32)), i
            assert np.array_equal(hi[s:s + n], np.fromfile(p("hic"), dtype=np.float32)), i
