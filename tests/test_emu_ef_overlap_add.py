"""CPU: the overlap-add of the n_fft 2048 two-group kernel's EF instantiation (float32 epilogue: none, or a wavefold
exact in float32), single-stepped through tests/emu/cuda_emu.h.  Interior batches -- every output hop inside the tile
and covered by four frames of the clip -- take an unrolled hop body with one row of 1/sum(w^2) per column; every
other batch takes the general hop.  The EF kernel must match the general instantiation bit for bit on the same
input: output samples, the sign of zeros included, and per-clip peaks.  The clip lengths put the switch between
interior and edge batches at every offset within a batch."""
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
TIMEOUT = 900
N_FFT, HOP, NW, SR = 2048, 512, 8, 48000   # the kernel <float, 1024, 8, TS, noFX, NG = 2>: 8 frames per batch


@pytest.fixture(scope="module")
def emu_ef():
    exe = os.path.join(tempfile.gettempdir(), f"qd_emu_spec_ef_{os.getuid()}")
    srcs = [os.path.join(EMU_DIR, f) for f in ("emu_spec_ef.cpp", "cuda_emu.h")]
    srcs += [os.path.join(CSRC, f) for f in ("qd_spec.cuh", "qd_common.cuh", "qd_host_tables.hpp")]
    if not os.path.exists(exe) or any(os.path.getmtime(s) > os.path.getmtime(exe) for s in srcs):
        tmp = f"{exe}.{os.getpid()}"
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-DQD_EMU", "-I", EMU_DIR, "-o", tmp,
                               os.path.join(EMU_DIR, "emu_spec_ef.cpp"), "-lpthread"], timeout=TIMEOUT)
        os.replace(tmp, exe)
    return exe


def _run(exe, d, x, layout, tile, epilogue, fold, ef):
    p = lambda f: os.path.join(d, f)  # noqa: E731
    x.astype(np.float32).tofile(p("x"))
    freqs = np.fft.rfftfreq(N_FFT, d=1.0 / SR)
    orc.target_bins_for_freqs(freqs, "D", "minor").astype(np.int32).tofile(p("tb"))
    orc.quantize_band_mask(freqs, 110.0, 5000.0).astype(np.uint8).tofile(p("mask"))
    subprocess.run([exe, str(ef), str(epilogue), repr(float(fold)), str(tile), p("x")] + layout +
                   [p("tb"), p("mask"), p("y")], check=True, timeout=TIMEOUT, stdout=subprocess.DEVNULL)
    return np.fromfile(p("y"), dtype=np.float32), np.fromfile(p("y") + ".peak", dtype=np.float32)


def run_spec(exe, x, tile, epilogue, fold, ef):
    """One quantised pass of x [clips, n]; ef = 1: the EF kernel, 0: the general one (both without a tap).
    Returns y [clips, n] and the peaks (one per clip, then two rows no clip owns)."""
    with tempfile.TemporaryDirectory() as d:
        y, peak = _run(exe, d, x, ["u%d" % x.shape[0], "-"], tile, epilogue, fold, ef)
        return y.reshape(x.shape), peak


def run_ragged(exe, clips, tile, ef):
    """A packed batch of clips of any lengths (gaps filled with junk), wavefold 2.0.  Returns the clips' outputs, the
    whole output buffer and the peaks."""
    with tempfile.TemporaryDirectory() as d:
        lengths = np.array([len(c) for c in clips], dtype=np.int64)
        starts, _ = pack_layout(lengths, 4)
        starts = starts + 8 * np.arange(len(clips), dtype=np.int64)
        x = np.full(int(starts[-1] + lengths[-1]), 7.0, dtype=np.float32)
        for s, c in zip(starts, clips):
            x[s:s + len(c)] = c
        starts.tofile(os.path.join(d, "starts"))
        lengths.astype(np.int32).tofile(os.path.join(d, "lengths"))
        y, peak = _run(exe, d, x, [os.path.join(d, "starts"), os.path.join(d, "lengths")], tile, 1, 2.0, ef)
        return [y[s:s + len(c)] for s, c in zip(starts, clips)], y, peak


def interior_batches(n, tile):
    """Batches of one clip of n samples that take the unrolled hop body, per tile (the kernel's test, in Python)."""
    j_end = 2 + (n + HOP - 1) // HOP
    n_frames = 1 + n // HOP
    out = []
    for j0 in range(2, j_end, tile):
        j1 = min(j0 + tile, j_end)
        out.append([tb for tb in range(j0 - 3, j1, NW) if tb >= 3 and tb >= j0 and tb + NW <= j1 and tb + NW <= n_frames])
    return out


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _noise(seed, n, clips=1):
    return np.stack([synth.noise_clip(seed + i, n) for i in range(clips)]).astype(np.float32)


# (n, clips, tile, epilogue, fold).  n_frames = 1 + n // 512, so these put the last interior batch's end at every offset
# 0 .. 7 within the next batch; 12288 = 24 hops (the last hop ends exactly at the clip end), 12286 one sample pair short
# of it.  3 clips: the last CTA carries an empty group.  Tile 20 cuts the clip into tiles with one interior batch in the
# middle of each; tile 12 leaves no interior batch at all.
UNIFORM_CASES = [
    (12288, 3, 64, 1, 2.0), (12288, 1, 64, 0, 1.0), (12286, 2, 64, 1, 4.0), (12286, 1, 64, 0, 1.0),
    (12800, 1, 64, 1, 2.0), (13312, 1, 64, 0, 1.0), (13826, 1, 64, 1, 0.5), (14336, 1, 64, 1, 2.0),
    (14850, 1, 64, 0, 1.0), (15360, 1, 64, 1, 2.0), (15874, 1, 64, 1, 2.0),
    (21000, 2, 20, 1, 2.0), (21000, 1, 12, 0, 1.0),
]


@pytest.mark.parametrize("n,clips,tile,epilogue,fold", UNIFORM_CASES)
def test_ef_kernel_matches_general_kernel(emu_ef, n, clips, tile, epilogue, fold):
    x = _noise(40 + n % 97, n, clips)
    if epilogue == 1:
        x *= 2.0 / fold   # drive the wavefold into both folds and the clamp
    y_ef, pk_ef = run_spec(emu_ef, x, tile, epilogue, fold, 1)
    y_gen, pk_gen = run_spec(emu_ef, x, tile, epilogue, fold, 0)
    assert np.array_equal(bits(y_ef), bits(y_gen))
    assert np.array_equal(bits(pk_ef), bits(pk_gen))
    assert np.all(pk_ef[clips:] == 0.0)
    np.testing.assert_array_equal(pk_ef[:clips], np.max(np.abs(y_ef), axis=1))
    assert not np.any(y_ef == -777.0)
    ib = interior_batches(n, tile)
    if tile == 20:
        assert [len(t) for t in ib] == [1, 1, 0], ib   # one in each full tile, none in the short last one
    elif tile == 12:
        assert not any(ib), ib
    else:
        assert len(ib) == 1 and ib[0], ib


def test_ef_kernel_odd_length_takes_general_path(emu_ef):
    """An odd clip length has no 8-byte stores: the EF kernel runs the general hop on every batch."""
    x = _noise(71, 12287)
    y_ef, pk_ef = run_spec(emu_ef, x, 64, 1, 2.0, 1)
    y_gen, pk_gen = run_spec(emu_ef, x, 64, 1, 2.0, 0)
    assert np.array_equal(bits(y_ef), bits(y_gen)) and np.array_equal(bits(pk_ef), bits(pk_gen))


def test_ef_kernel_against_oracle(emu_ef):
    """The EF kernel with the reference-default epilogue (wavefold 2.0, no bias) against the oracle."""
    n = 14000
    x = _noise(77, n)[0]
    y, pk = run_spec(emu_ef, x[None], 64, 1, 2.0, 1)
    ref = orc.apply_distortion(oracle_pass(x), "wavefold", fold_amount=2.0, bias=0.0)
    assert float(np.max(np.abs(y[0] - ref))) < 1e-5
    assert abs(float(pk[0]) - float(np.max(np.abs(ref)))) < 1e-5


def oracle_pass(x):
    S, freqs = orc.stft(x, SR, N_FFT)
    S = orc.spectral_quantize_stft(S, freqs, "D", "minor", 1.0, 0.1, True, quantize_min_hz=110.0, quantize_max_hz=5000.0)
    return orc.istft(S, SR, N_FFT, length=len(x))


# packed clips of different lengths: CTA rows pair (0,1), (2,3), ... so each CTA runs two groups whose batches turn
# from interior to edge at different times; 12287 is odd (general path), the last CTA has an empty group
RAGGED_LENGTHS = [14336, 9730, 12288, 15874, 12287]


@pytest.mark.parametrize("tile", [64, 20])
def test_ef_kernel_ragged_groups_of_different_lengths(emu_ef, tile):
    clips = [0.5 * _noise(90 + i, n)[0] for i, n in enumerate(RAGGED_LENGTHS)]
    ys_ef, y_ef, pk_ef = run_ragged(emu_ef, clips, tile, True)
    _, y_gen, pk_gen = run_ragged(emu_ef, clips, tile, False)
    assert np.array_equal(bits(y_ef), bits(y_gen))   # the gaps included, which no kernel writes
    assert np.array_equal(bits(pk_ef), bits(pk_gen))
    for i, y in enumerate(ys_ef):
        assert float(pk_ef[i]) == float(np.max(np.abs(y)))
    assert all(any(interior_batches(n, tile)) for n in RAGGED_LENGTHS)
