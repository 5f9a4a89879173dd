"""CPU: host side of the scale-alignment metric on ragged batches -- the C declaration and binding of
qd_spectral_peaks_device_varlen, its argument checks (which run before the device is touched), the row layout of the
bins, and the validation of a list of clips."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from quantumdistortion_b200 import _lib, analyses
from quantumdistortion_b200.pipeline import pack_layout

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
QD_ERR_INVALID_ARG = -1


def test_varlen_peaks_symbol_declared_and_bound():
    header = open(os.path.join(ROOT, "include", "qd_b200.h")).read()
    assert re.search(r"#define QD_ABI_VERSION 6\b", header)
    assert "int qd_spectral_peaks_device_varlen(" in header
    src = open(os.path.join(ROOT, "quantumdistortion_b200", "_lib.py")).read()
    assert "lib.qd_spectral_peaks_device_varlen.argtypes" in src
    assert hasattr(_lib.load(), "qd_spectral_peaks_device_varlen")


def _ptr(a):
    return C.c_void_p(a.ctypes.data)


def test_varlen_peaks_rejects_invalid_arguments_without_a_device():
    lib = _lib.load()
    x = np.zeros(64, np.float32)             # host memory: never read, the argument checks come first
    st = np.zeros(4, np.int64)
    ln = np.zeros(4, np.int32)
    bins = np.zeros(64, np.int16)
    ok = dict(x=_ptr(x), starts=_ptr(st), lengths=_ptr(ln), batch=4, max_samples=16, n_fft=2048, topn=3, min_mag=1e-3,
              precision=1, bins=_ptr(bins))

    def call(**kw):
        a = dict(ok, **kw)
        return lib.qd_spectral_peaks_device_varlen(a["x"], a["starts"], a["lengths"], a["batch"], a["max_samples"],
                                                   a["n_fft"], a["topn"], a["min_mag"], a["precision"], a["bins"], None)

    bad = [dict(x=None), dict(starts=None), dict(lengths=None), dict(bins=None), dict(batch=-1), dict(batch=2 ** 31),
           dict(topn=0), dict(topn=9), dict(precision=2), dict(precision=-1), dict(max_samples=-1)]
    for kw in bad:
        assert call(**kw) == QD_ERR_INVALID_ARG, kw
    assert call(batch=2 ** 31) == QD_ERR_INVALID_ARG and b"2^31" in lib.qd_last_error()
    assert call(batch=0) == 0                 # an empty batch is fine and touches nothing


@pytest.mark.parametrize("seed", range(6))
@pytest.mark.parametrize("n_fft", [512, 2048, 8192])
def test_peak_rows_are_disjoint_within_the_bound(seed, n_fft):
    rng = np.random.default_rng(seed)
    hop = n_fft // 4
    b = int(rng.integers(1, 60))
    lengths = rng.integers(0, 5 * n_fft, b)
    lengths[rng.random(b) < 0.2] = 0
    lengths[rng.random(b) < 0.2] = hop * rng.integers(0, 4, 1) + rng.integers(-1, 2, 1)
    lengths = np.maximum(lengths, 0)
    starts, _ = pack_layout(lengths, 4)
    starts = starts + np.cumsum(rng.integers(0, 3 * hop, b)) + int(rng.integers(0, 10 ** 6))  # gaps; a sub-range
    for lo in (0, b // 3):                  # the whole batch and a sub-range that does not start at clip 0
        st, ln = starts[lo:], lengths[lo:]
        if st.size == 0:
            continue
        row0, frames, n_rows = analyses.peak_rows(st, ln, hop)
        assert n_rows == (st[-1] - st[0] + ln[-1]) // hop + st.size
        assert np.array_equal(frames, 1 + ln // hop)
        used = np.zeros(n_rows, np.int64)
        for r, f in zip(row0, frames):
            assert 0 <= r and r + f <= n_rows
            used[r:r + f] += 1
        assert used.max() == 1, "rows of two clips overlap"


def test_peak_rows_empty():
    row0, frames, n_rows = analyses.peak_rows([], [], 512)
    assert row0.size == 0 and frames.size == 0 and n_rows == 0


@pytest.mark.parametrize("fn", ["spectral_peak_bins", "avg_cents_offset_batch"])
def test_list_validation_needs_no_device(fn):
    import torch
    call = (lambda x: analyses.spectral_peak_bins(x)) if fn == "spectral_peak_bins" else \
        (lambda x: analyses.avg_cents_offset_batch(x, 48000, "D", "minor"))
    with pytest.raises(ValueError, match="all NumPy arrays or all tensors"):
        call([np.zeros(100, np.float32), torch.zeros(100)])
    with pytest.raises(ValueError, match="all NumPy arrays or all tensors"):
        call([np.zeros(100, np.float32), [0.0] * 100])
    with pytest.raises(ValueError, match="1-D"):
        call([np.zeros(100, np.float32), np.zeros((2, 100), np.float32)])
    with pytest.raises(ValueError, match="1-D"):
        call((torch.zeros(3), torch.zeros(()),))
    out = call([])
    if fn == "spectral_peak_bins":
        assert out == []
    else:
        assert out[0].shape == (0,) and out[1] == []
