"""CPU: peaks_kernel (csrc/qd_peaks.cuh, the device half of the scale-alignment metric) single-stepped through
tests/emu/cuda_emu.h with the library's FFT tables and launch geometry.

* Uniform clips against the oracle's chosen bins, at every n_fft and topn 1, 3 and 8.
* Ragged batches packed with NaN in the gaps: every clip's rows are bit-identical to the clip alone, and rows no clip
  owns keep their sentinel.
* Launch splits through qd::for_each_launch match one launch bit for bit.

cuda_emu.h implements warp barriers with pthread barriers, so a warp that leaves early shows up as a hang: every
emulator run has a timeout, which turns that into a failure."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

import qd_cases
from oracle import qd_oracle as orc
from quantumdistortion_b200 import synth
from quantumdistortion_b200.analyses import peak_rows
from quantumdistortion_b200.pipeline import pack_layout

HERE = os.path.dirname(os.path.abspath(__file__))
EMU_DIR = os.path.join(HERE, "emu")
CSRC = os.path.join(os.path.dirname(HERE), "quantumdistortion_b200", "csrc")
TIMEOUT = 600
SENTINEL = 0x5A5A
NFFTS = [512, 1024, 2048, 4096, 8192]
TOPNS = [1, 3, 8]


@pytest.fixture(scope="module")
def emu_peaks():
    exe = os.path.join(tempfile.gettempdir(), f"qd_emu_peaks_{os.getuid()}")
    srcs = [os.path.join(EMU_DIR, f) for f in ("emu_peaks.cpp", "cuda_emu.h")]
    srcs += [os.path.join(CSRC, f) for f in ("qd_peaks.cuh", "qd_spec.cuh", "qd_common.cuh", "qd_host_tables.hpp")]
    if not os.path.exists(exe) or any(os.path.getmtime(s) > os.path.getmtime(exe) for s in srcs):
        tmp = f"{exe}.{os.getpid()}"
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-DQD_EMU", "-I", EMU_DIR, "-o", tmp,
                               os.path.join(EMU_DIR, "emu_peaks.cpp"), "-lpthread"], timeout=TIMEOUT)
        os.replace(tmp, exe)
    return exe


def _min_mag(min_db):
    return repr(float(10.0 ** (min_db / 20.0)))


def _run(exe, d, prec, n_fft, topn, min_db, x, layout=("-", "-"), per_launch=None):
    """bins of x (one clip, "u<B>" uniform clips or a packed batch with layout (starts file, lengths file))"""
    xp, out = os.path.join(d, "x_in"), os.path.join(d, "bins_out")
    np.asarray(x, dtype=np.float32).tofile(xp)
    cmd = [exe] + (["-p", str(per_launch)] if per_launch else [])
    cmd += [prec, str(n_fft), str(topn), _min_mag(min_db), xp, layout[0], layout[1], out]
    subprocess.run(cmd, check=True, timeout=TIMEOUT, stdout=subprocess.DEVNULL)
    return np.fromfile(out, dtype=np.int16).reshape(-1, topn)


# ---------------------------------------------------------------- uniform clips vs the oracle

def _inputs():
    out = {}
    for name, (kind, seed, n, sr, key, scale, kw) in qd_cases.ANALYSIS_CASES.items():
        out[name] = (qd_cases.make_signal(kind, seed, n, sr), sr, key, scale, kw.get("min_db", -60.0))
    out["bass"] = (synth.bass_clip(90, 24000, 48000), 48000, "D", "minor", -60.0)
    out["noise"] = (synth.noise_clip(91, 24000), 48000, "A", "pentatonic", -30.0)
    return out


INPUTS = _inputs()
_near_ties = {"count": 0}


@pytest.mark.parametrize("n_fft", NFFTS)
@pytest.mark.parametrize("name", list(INPUTS))
def test_emu_peaks_uniform_vs_oracle(emu_peaks, name, n_fft):
    x, sr, key, scale, min_db = INPUTS[name]
    x = np.asarray(x, dtype=np.float32)
    _, _, ref8 = orc.avg_cents_offset_from_scale(x.astype(np.float64), sr, key, scale, frame_length=n_fft,
                                                 topn_peaks=max(TOPNS), min_db=min_db, return_bins=True)
    mag = np.abs(orc.stft(x.astype(np.float64), sr, n_fft=n_fft)[0]).T     # [frames, bins]
    assert (ref8 >= 0).any() or name == "an_quiet", "the input must have peaks above min_db"   # an_quiet has none
    near = 0
    with tempfile.TemporaryDirectory() as d:
        for topn in TOPNS:
            ref = ref8[:, :topn]   # the oracle stops after topn bins, so its first columns are the smaller topn
            b64 = _run(emu_peaks, d, "f64", n_fft, topn, min_db, x)
            assert b64.shape == ref.shape
            for t in np.nonzero((b64 != ref).any(axis=1))[0]:
                # the only admitted difference: two bins whose oracle magnitudes agree to 1e-12 relative, in either order
                for j in np.nonzero(b64[t] != ref[t])[0]:
                    a, b = int(b64[t, j]), int(ref[t, j])
                    assert a >= 0 and b >= 0, (topn, t, b64[t], ref[t])
                    assert abs(mag[t, a] - mag[t, b]) <= 1e-12 * max(mag[t, a], mag[t, b]), (topn, t, b64[t], ref[t])
                near += 1
            b32 = _run(emu_peaks, d, "f32", n_fft, topn, min_db, x)
            assert np.mean(b32 == ref) >= 0.98, (topn, float(np.mean(b32 == ref)))
    _near_ties["count"] += near
    print(f"{name} n_fft {n_fft}: {near} frames with near-tied bins in another order (total {_near_ties['count']})")


# ---------------------------------------------------------------- ragged batches

def _pack(d, clips, offset=0, gap=np.nan):
    """Packed input with NaN gaps (a kernel that reads one poisons a frame) and wider gaps than the packer's;
    `offset` shifts every start, as a sub-range of a larger batch does."""
    lengths = np.array([len(c) for c in clips], dtype=np.int64)
    starts, _ = pack_layout(lengths, 4)
    starts = starts + 5 * np.arange(len(clips), dtype=np.int64) + offset
    x = np.full(int(starts[-1] + lengths[-1] - starts[0]), gap, dtype=np.float32)
    for s, c in zip(starts - starts[0], clips):
        x[s:s + len(c)] = c
    starts.astype(np.int64).tofile(os.path.join(d, "starts"))
    lengths.astype(np.int32).tofile(os.path.join(d, "lengths"))
    return x, starts, lengths, (os.path.join(d, "starts"), os.path.join(d, "lengths"))


def _ragged_lengths(n_fft, seconds=2.5, sr=48000):
    hop = n_fft // 4
    return [int(seconds * sr), 0, 1, hop - 1, hop, hop + 1, n_fft, 3 * hop + 2, 0, 5 * hop - 1]


def _clips(lengths, seed=0):
    out = []
    for i, n in enumerate(lengths):
        c = synth.bass_clip(seed + i, n, 48000) if n >= 2 else 0.7 * np.ones(n)
        out.append(np.asarray(c, dtype=np.float32))
    return out


@pytest.mark.parametrize("prec", ["f32", "f64"])
@pytest.mark.parametrize("n_fft,topn,min_db,offset", [(512, 3, -60.0, 0), (1024, 8, -40.0, 77), (2048, 3, -60.0, 3),
                                                      (4096, 1, -60.0, 0), (8192, 8, -60.0, 1000)])
def test_emu_peaks_ragged_matches_clips_alone(emu_peaks, prec, n_fft, topn, min_db, offset):
    hop = n_fft // 4
    clips = _clips(_ragged_lengths(n_fft))
    with tempfile.TemporaryDirectory() as d:
        x, starts, lengths, layout = _pack(d, clips, offset)
        got = _run(emu_peaks, d, prec, n_fft, topn, min_db, x, layout)
        row0, frames, n_rows = peak_rows(starts, lengths, hop)
        assert got.shape[0] == n_rows == int((starts[-1] - starts[0] + lengths[-1]) // hop + len(clips))
        owned = np.zeros(n_rows, bool)
        for i, c in enumerate(clips):
            alone = _run(emu_peaks, d, prec, n_fft, topn, min_db, c)
            assert alone.shape[0] == frames[i] == 1 + len(c) // hop
            mine = got[row0[i]:row0[i] + frames[i]]
            assert np.array_equal(mine, alone), (i, len(c))
            assert not owned[row0[i]:row0[i] + frames[i]].any(), "rows of two clips overlap"
            owned[row0[i]:row0[i] + frames[i]] = True
            if len(c) == 0:
                assert np.all(mine == -1)
        assert (got[row0[0]:row0[0] + frames[0]] >= 0).any(), "the long clip must have peaks"
        assert (~owned).any() and np.all(got[~owned] == SENTINEL), "a row no clip owns was written"


# ---------------------------------------------------------------- launch splits

@pytest.mark.parametrize("prec", ["f32", "f64"])
def test_emu_peaks_launch_split(emu_peaks, prec):
    n_fft, topn = 1024, 3
    clips = _clips([3000, 0, 700, 1, 2100, 256, 4097], seed=5)
    uni = np.concatenate(_clips([1500] * 5, seed=9))
    with tempfile.TemporaryDirectory() as d:
        x, _, _, layout = _pack(d, clips, 13)
        whole = _run(emu_peaks, d, prec, n_fft, topn, -60.0, x, layout)
        whole_u = _run(emu_peaks, d, prec, n_fft, topn, -60.0, uni, ("u5", "-"))
        assert (whole >= 0).any() and (whole == SENTINEL).any() and (whole_u >= 0).any()
        for p in (1, 2, 3):
            assert np.array_equal(_run(emu_peaks, d, prec, n_fft, topn, -60.0, x, layout, per_launch=p), whole), p
            assert np.array_equal(_run(emu_peaks, d, prec, n_fft, topn, -60.0, uni, ("u5", "-"), per_launch=p),
                                  whole_u), p
