"""Scale-alignment metric ``avg_cents_offset_from_scale`` (quantum_distortion/dsp/analyses.py:53-142).

The reference walks every STFT frame, takes the ``topn_peaks`` strongest bins above ``min_db`` and averages
their distance in cents to the nearest note of the key/scale.  That distance depends only on the bin's
frequency, so the split here is:

* host (this file, NumPy float64): ``scale_cents_table`` -- |cents| per bin with the reference's own formulas
  (``freq_to_midi``, ``build_scale_notes`` over ``[f/4, 4f]``, first-index ``argmin``), bit-exact;
* device (csrc/qd_peaks.cuh through ``qd_spectral_peaks_device``): the STFT of every clip and the strongest
  bins per frame, for a whole batch of clips at once.

There is no CPU fallback: without a B200 and the built library every call raises.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Tuple, Union

import numpy as np

from . import _lib, tables


def _note_midis(key: str, scale: str, min_freq: float, max_freq: float) -> np.ndarray:
    """MIDI numbers of build_scale_notes(key, scale, min_freq, max_freq) (dsp/quantizer.py:98-124)."""
    root_pc = tables.note_name_to_pitch_class(key)
    intervals = tables.SCALE_INTERVALS[scale]
    lo = int(np.floor(69.0 + 12.0 * np.log2(max(min_freq, 20.0) / 440.0))) - 12
    hi = int(np.ceil(69.0 + 12.0 * np.log2(min(max_freq, 22050.0) / 440.0))) + 12
    out = []
    for midi in range(lo, hi + 1):
        if ((midi % 12) - root_pc) % 12 in intervals:
            f = 440.0 * (2.0 ** ((float(midi) - 69.0) / 12.0))
            if f < min_freq * 0.5 or f > max_freq * 2.0:
                continue
            out.append(midi)
    return np.asarray(out, dtype=float)


def scale_cents_table(freqs: np.ndarray, key: str, scale: str) -> np.ndarray:
    """|100 * (midi(f) - nearest scale midi)| per bin (dsp/analyses.py:18-50, 120-130); NaN where the
    reference would skip the bin (f <= 0 or no scale note in range)."""
    out = np.full(len(freqs), np.nan)
    for i, f in enumerate(np.asarray(freqs, dtype=float)):
        f = float(f)
        if f <= 0.0:
            continue
        midi_est = 69.0 + 12.0 * np.log2(f / 440.0)          # freq_to_midi, dsp/quantizer.py:76-79
        if not np.isfinite(midi_est):
            continue
        freq = 440.0 * (2.0 ** ((midi_est - 69.0) / 12.0))   # midi_to_freq of the estimate (:35)
        notes = _note_midis(key, scale, float(max(20.0, freq / 4.0)), float(min(20000.0, freq * 4.0)))
        if notes.size == 0:
            continue
        scale_midi = float(notes[int(np.argmin(np.abs(notes - midi_est)))])
        out[i] = abs(float(100.0 * (midi_est - scale_midi)))
    return out


def peak_rows(starts, lengths, hop: int) -> Tuple[np.ndarray, np.ndarray, int]:
    """Rows of a ragged batch in the bins of qd_spectral_peaks_device_varlen (include/qd_b200.h): clip c's
    T_c = 1 + n_c // hop frames start at row (starts[c] - starts[0]) // hop + c.  Returns (row0, frames, n_rows) with
    n_rows = span // hop + batch, which holds every clip's rows without overlap."""
    st = np.asarray(starts, dtype=np.int64).reshape(-1)
    ln = np.asarray(lengths, dtype=np.int64).reshape(-1)
    if st.size == 0:
        return st, ln, 0
    rel = st - st[0]
    return rel // hop + np.arange(st.size, dtype=np.int64), 1 + ln // hop, int((rel[-1] + ln[-1]) // hop + st.size)


def _ragged_peak_rows(clips, n_fft: int, topn: int, min_db: float, precision: str):
    """The bins of a list of 1-D clips in one device call: (bins [n_rows, topn] int16 on the device, row0, frames,
    is_np, cuda), rows as in ``peak_rows``."""
    from .pipeline import clip_list_kind, pack_clips
    is_np, cuda = clip_list_kind(clips)   # ValueError before any device check
    prec = {"float32": 0, "float64": 1}[precision]
    import torch
    if not clips:
        return torch.zeros((0, topn), dtype=torch.int16), np.zeros(0, np.int64), np.zeros(0, np.int64), is_np, cuda
    if not torch.cuda.is_available():
        raise _lib.QdError("no CUDA device visible: quantumdistortion_b200 has no CPU fallback")
    lib = _lib.load()
    xf, starts, span = pack_clips(clips, cuda)
    lengths = np.array([int(c.shape[0]) for c in clips], dtype=np.int64)
    row0, frames, n_rows = peak_rows(starts, lengths, int(n_fft) // 4)
    xd = xf.cuda(non_blocking=True) if span else torch.zeros(1, device="cuda")   # all clips empty: x is never read
    d_starts = torch.from_numpy(starts).cuda(non_blocking=True)
    d_lengths = torch.from_numpy(lengths.astype(np.int32)).cuda(non_blocking=True)
    bins = torch.empty((n_rows, topn), dtype=torch.int16, device="cuda")
    _lib.check(lib.qd_spectral_peaks_device_varlen(xd.data_ptr(), d_starts.data_ptr(), d_lengths.data_ptr(), len(clips),
                                                   int(lengths.max()), int(n_fft), int(topn),
                                                   float(10.0 ** (min_db / 20.0)), prec, bins.data_ptr(),
                                                   torch.cuda.current_stream().cuda_stream))
    return bins, row0, frames, is_np, cuda


def spectral_peak_bins(x, n_fft: int = 2048, topn: int = 3, min_db: float = -60.0, precision: str = "float64"):
    """Strongest ``topn`` bins per STFT frame of every clip: x [B, n] (CUDA tensor, CPU tensor or NumPy) ->
    int16 [B, 1 + n // (n_fft/4), topn] on the same kind of container, -1 where fewer bins reach ``min_db``.

    ``x`` may also be a list or tuple of 1-D clips of any lengths: all NumPy arrays, all CPU tensors or all CUDA tensors,
    each cast to float32.  They are packed into one buffer and run in one call (qd_spectral_peaks_device_varlen); the
    result is a list of the same kind, clip c's int16 [1 + n_c // (n_fft/4), topn], equal to the clip run alone."""
    import torch
    if isinstance(x, (list, tuple)):
        bins, row0, frames, is_np, cuda = _ragged_peak_rows(list(x), n_fft, topn, min_db, precision)
        if not cuda:
            bins = bins.cpu().numpy() if is_np else bins.cpu()
        return [bins[r:r + f] for r, f in zip(row0.tolist(), frames.tolist())]
    if not torch.cuda.is_available():
        raise _lib.QdError("no CUDA device visible: quantumdistortion_b200 has no CPU fallback")
    lib = _lib.load()
    is_np = isinstance(x, np.ndarray)
    xt = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)) if is_np else x
    if xt.dim() != 2:
        raise ValueError("spectral_peak_bins expects [batch, samples]")
    on_cuda = xt.is_cuda
    xd = xt.float().contiguous().cuda()
    b, n = int(xd.shape[0]), int(xd.shape[1])
    frames = 1 + n // (n_fft // 4)
    bins = torch.empty((b, frames, topn), dtype=torch.int16, device="cuda")
    prec = {"float32": 0, "float64": 1}[precision]
    if b:
        _lib.check(lib.qd_spectral_peaks_device(xd.data_ptr(), b, n, int(n_fft), int(topn),
                                                float(10.0 ** (min_db / 20.0)), prec, bins.data_ptr(),
                                                torch.cuda.current_stream().cuda_stream))
    if on_cuda:
        return bins
    return bins.cpu().numpy() if is_np else bins.cpu()


def _cents_per_clip(bins: np.ndarray, row0: np.ndarray, frames: np.ndarray, table: np.ndarray):
    """(avgs, per-clip |cents| arrays) from bins [rows, topn], clip c owning rows row0[c] .. + frames[c]: one table
    lookup over every owned row, then a split by clip."""
    b = len(row0)
    owned = np.repeat(row0 - np.cumsum(frames) + frames, frames) + np.arange(int(frames.sum()), dtype=np.int64)
    flat = bins[owned].reshape(-1)
    owner = np.repeat(np.arange(b), frames * bins.shape[1])
    keep = flat >= 0
    cents = table[flat[keep].astype(np.int64)]
    owner = owner[keep]
    fin = np.isfinite(cents)
    cents, owner = cents[fin].astype(float), owner[fin]
    per_clip = np.split(cents, np.cumsum(np.bincount(owner, minlength=b))[:-1]) if b else []
    avgs = np.array([float(np.mean(c)) if c.size else np.nan for c in per_clip], dtype=float)
    return avgs, per_clip


def avg_cents_offset_batch(x, sr: int, key: str, scale: str, frame_length: int = 2048, topn_peaks: int = 3,
                           min_db: float = -60.0, precision: str = "float64") -> Tuple[np.ndarray, List[np.ndarray]]:
    """The metric for every clip of a batch: (avg_abs_cents [B] (NaN for a silent clip), per-clip arrays of
    per-peak |cents| in the reference's order: frame by frame, strongest bin first).  ``x`` is [B, n] or a list of
    1-D clips of any lengths (see ``spectral_peak_bins``); each clip gets the values it gets alone."""
    table = scale_cents_table(np.fft.rfftfreq(frame_length, d=1.0 / sr), key, scale)
    if isinstance(x, (list, tuple)):
        bins, row0, frames, _, _ = _ragged_peak_rows(list(x), frame_length, topn_peaks, min_db, precision)
        return _cents_per_clip(bins.cpu().numpy(), row0, frames, table)
    bins = spectral_peak_bins(x, n_fft=frame_length, topn=topn_peaks, min_db=min_db, precision=precision)
    bins = bins.cpu().numpy() if hasattr(bins, "cpu") else np.asarray(bins)
    b, t = bins.shape[0], bins.shape[1]
    return _cents_per_clip(bins.reshape(b * t, bins.shape[2]), np.arange(b, dtype=np.int64) * t, np.full(b, t, np.int64), table)


def avg_cents_offset_from_scale(audio: np.ndarray, sr: int, key: str, scale: str, frame_length: int = 2048,
                                hop_length: Union[int, None] = None, topn_peaks: int = 3, min_db: float = -60.0,
                                precision: str = "float64") -> Tuple[float, np.ndarray]:
    """Drop-in for dsp/analyses.py:53-142 (one clip).  ``hop_length`` is accepted and, like in the reference,
    unused: stft_mono always hops by frame_length // 4 (:87-96)."""
    x = np.asarray(audio, dtype=float)
    if x.ndim != 1:
        raise ValueError("avg_cents_offset_from_scale expects mono (1D) audio")
    avgs, per = avg_cents_offset_batch(x[None, :].astype(np.float32), sr, key, scale, frame_length, topn_peaks,
                                       min_db, precision)
    if per[0].size == 0:
        return float("nan"), np.array([], dtype=float)
    return float(avgs[0]), per[0]
