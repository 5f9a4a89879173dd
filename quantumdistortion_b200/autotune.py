"""Host side of ``quantize_mode="autotune_v1"`` -- the reference's default mode (quantum_distortion/dsp/autotune.py
behind dsp/pipeline.py:537-601).

Everything the reference derives on the CPU is resolved here in float64 with the reference's own library calls
(``scipy.signal.butter`` / ``sosfilt_zi``, Python ``int()`` truncation for the YIN lag range, key / scale tables) and
handed to ``qd_autotune_render_device`` as plain numbers (``include/qd_b200.h``: ``qd_autotune_params``).  The CUDA
kernels are in ``csrc/qd_autotune.cuh``.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from typing import Any, Dict, Optional

import numpy as np
from scipy.signal import butter, sosfilt_zi

from . import _lib, tables

# AutotuneV1Config defaults the pipeline never overrides (dsp/autotune.py:18-45)
SUB_PRESERVE_MIX = 0.15
DETECTOR_LOW_HZ, DETECTOR_HIGH_HZ = 110.0, 3000.0
FRAME_SIZE, HOP_SIZE = 4096, 512
MIN_CONFIDENCE, RMS_THRESHOLD, FLATNESS_THRESHOLD = 0.72, 0.01, 0.55
NOTE_CHANGE_CENTS, NOTE_CONFIRM_FRAMES, NOTE_RELEASE_FRAMES = 40.0, 3, 2
GRAIN_SIZE, BUFFER_SIZE = 1024, 4096
YIN_THRESHOLD = 0.15


class QdAutotuneParams(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("sample_rate", C.c_int32), ("n_samples", C.c_int32), ("apply", C.c_int32),
        ("filt_on", C.c_int32 * 4), ("sos", ((C.c_double * 6) * 2) * 4), ("zi", ((C.c_double * 2) * 2) * 4),
        ("frame_size", C.c_int32), ("hop", C.c_int32), ("min_tau", C.c_int32), ("max_tau", C.c_int32),
        ("min_freq", C.c_double), ("max_freq", C.c_double), ("yin_threshold", C.c_double),
        ("rms_thr", C.c_double), ("flat_thr", C.c_double), ("conf_thr", C.c_double),
        ("root_pc", C.c_int32), ("n_intervals", C.c_int32), ("intervals", C.c_int32 * 8),
        ("strength", C.c_double), ("change_cents", C.c_double),
        ("confirm_frames", C.c_int32), ("release_frames", C.c_int32),
        ("max_delay", C.c_int32), ("buffer_size", C.c_int32),
        ("sub_enabled", C.c_int32), ("layer_on", C.c_int32),
        ("env_attack", C.c_float), ("env_release", C.c_float),
        ("sub_level", C.c_float), ("sub_preserve", C.c_float), ("air_mix", C.c_float), ("phase_k", C.c_float),
        ("distortion_mode", C.c_int32), ("tube_gain", C.c_float), ("tube_norm", C.c_float),
        ("limiter_on", C.c_int32), ("lookahead", C.c_int32), ("fold_amount", C.c_double), ("bias", C.c_double),
        ("ceiling_lin", C.c_double), ("release_coeff", C.c_double),
        ("wet", C.c_float), ("dry", C.c_float), ("trim_gain", C.c_float), ("apply_trim", C.c_int32),
        ("delta_listen", C.c_int32),
    ]


class QdAutotuneDebug(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("sub", "body", "air", "det", "ratio_track", "corrected", "sub_layer", "features")]


def _filter(p: QdAutotuneParams, which: int, sr: int, cutoff_hz: float, btype: str) -> None:
    """dsp/autotune.py:88-100: 4th-order Butterworth as two sections, plus scipy's steady-state initial conditions."""
    if cutoff_hz <= 0.0:
        p.filt_on[which] = 0
        return
    wn = float(np.clip(cutoff_hz / (sr / 2.0), 1e-5, 0.999))
    sos = butter(4, wn, btype=btype, output="sos")
    zi = sosfilt_zi(sos)
    p.filt_on[which] = 1
    for s in range(2):
        for c in range(6):
            p.sos[which][s][c] = float(sos[s, c])
        for c in range(2):
            p.zi[which][s][c] = float(zi[s, c])


def sub_frequency(key: str, scale: str, sub_source: str, sub_note: str, sub_scale_degree: int, sub_octave: int) -> float:
    """dsp/autotune.py:380-396."""
    if sub_source == "manual":
        pc = tables.note_name_to_pitch_class(sub_note)
    elif sub_source == "scale_degree":
        iv = tables.SCALE_INTERVALS[scale]
        pc = (tables.note_name_to_pitch_class(key) + iv[int(np.clip(sub_scale_degree, 0, len(iv) - 1))]) % 12
    else:
        pc = tables.note_name_to_pitch_class(key)
    midi = 12 * (int(np.clip(sub_octave, 0, 6)) + 1) + pc
    return float(440.0 * (2.0 ** ((float(midi) - 69.0) / 12.0)))


def resolve(*, sr: int, n_samples: int, key: str, scale: str, snap_strength: float, pre_quant: bool,
            distortion_mode: Optional[str], distortion_params: Optional[Dict[str, Any]], limiter_on: bool,
            limiter_ceiling_db: float, dry_wet: float, output_trim_db: float, delta_listen: bool,
            sub_enabled: bool = True, sub_source: str = "root", sub_note: str = "C", sub_scale_degree: int = 0,
            sub_octave: int = 2, sub_level: float = 0.35, sub_cut_hz: float = 110.0, air_cut_hz: float = 5000.0,
            air_mix: float = 1.0) -> QdAutotuneParams:
    """process_audio keyword arguments -> qd_autotune_params; raises the reference's exceptions before any launch."""
    p = QdAutotuneParams()
    p.struct_size = C.sizeof(QdAutotuneParams)
    p.sample_rate, p.n_samples = int(sr), int(n_samples)
    p.apply = int(bool(pre_quant and snap_strength > 0.0))                       # dsp/pipeline.py:538
    root_pc = tables.note_name_to_pitch_class(key)                               # ValueError for a bad key
    intervals = tables.SCALE_INTERVALS[scale]                                    # KeyError for a bad scale
    _filter(p, 0, sr, float(sub_cut_hz), "low")                                  # dsp/autotune.py:110
    _filter(p, 1, sr, float(air_cut_hz), "high")                                 # :111
    _filter(p, 2, sr, DETECTOR_LOW_HZ, "high")                                   # :123-124
    _filter(p, 3, sr, DETECTOR_HIGH_HZ, "low")                                   # :125-126
    p.frame_size, p.hop = int(max(1024, FRAME_SIZE)), int(max(128, HOP_SIZE))    # :206-207
    min_freq, max_freq = max(60.0, DETECTOR_LOW_HZ * 0.65), max(DETECTOR_HIGH_HZ, 400.0)   # :229-230
    p.min_freq, p.max_freq, p.yin_threshold = min_freq, max_freq, YIN_THRESHOLD
    p.max_tau = min(int(sr / max(min_freq, 1e-6)), max(2, p.frame_size // 2 - 1))  # :153
    p.min_tau = max(2, int(sr / max(max_freq, 1e-6)))                              # :154
    p.rms_thr, p.flat_thr, p.conf_thr = RMS_THRESHOLD, FLATNESS_THRESHOLD, MIN_CONFIDENCE
    p.root_pc, p.n_intervals = root_pc, len(intervals)
    for i, iv in enumerate(intervals):
        p.intervals[i] = iv
    p.strength = float(np.clip(snap_strength, 0.0, 1.0))                         # dsp/pipeline.py:547
    p.change_cents, p.confirm_frames, p.release_frames = NOTE_CHANGE_CENTS, NOTE_CONFIRM_FRAMES, NOTE_RELEASE_FRAMES
    max_delay = int(max(256, GRAIN_SIZE))                                        # dsp/autotune.py:312-319
    size = int(max(max_delay * 2, BUFFER_SIZE))
    if size & (size - 1):
        size = 1 << int(np.ceil(np.log2(size)))
    p.max_delay, p.buffer_size = max_delay, size
    f_sub = sub_frequency(key, scale, sub_source, sub_note, sub_scale_degree, sub_octave)
    p.sub_enabled = int(bool(sub_enabled))
    p.layer_on = int(bool(sub_enabled) and sub_level > 0.0 and f_sub > 0.0)       # :404-409
    p.env_attack = float(np.float32(np.exp(-1.0 / max(1.0, 8.0 * 0.001 * sr))))  # :369-370 (float32 in the loop, NEP 50)
    p.env_release = float(np.float32(np.exp(-1.0 / max(1.0, 90.0 * 0.001 * sr))))
    p.sub_level, p.sub_preserve, p.air_mix = float(sub_level), SUB_PRESERVE_MIX, float(air_mix)
    p.phase_k = float(np.float32(2.0 * np.pi * f_sub))                            # :417
    # shared tail (dsp/pipeline.py:577-601, 180-223), same rules as tables.resolve
    mode = distortion_mode or "wavefold"
    dp = distortion_params or {}
    if mode == "wavefold":
        p.distortion_mode = 0
    elif mode == "tube":
        p.distortion_mode = 1
    else:
        raise ValueError(f"Unsupported distortion mode: {mode}")
    p.fold_amount, p.bias = float(dp.get("fold_amount", 1.0)), float(dp.get("bias", 0.0))
    a = 1.0 + 4.0 * float(np.clip(float(dp.get("warmth", 0.5)), 0.0, 1.0))
    p.tube_gain = a * max(float(dp.get("drive", 1.0)), 0.0)
    p.tube_norm = 1.0 / float(np.tanh(a))
    ceiling, lookahead, coeff = tables.limiter_constants(sr, limiter_ceiling_db)
    p.limiter_on, p.lookahead, p.ceiling_lin, p.release_coeff = int(bool(limiter_on)), lookahead, ceiling, coeff
    dw = float(np.clip(dry_wet, 0.0, 1.0))
    p.wet, p.dry = float(np.float32(dw)), float(np.float32(1.0 - dw))
    p.apply_trim = int(output_trim_db != 0.0)
    p.trim_gain = float(np.float32(10.0 ** (output_trim_db / 20.0)))
    p.delta_listen = int(bool(delta_listen))
    check_lengths(p, [n_samples])
    return p


def check_lengths(p: QdAutotuneParams, lengths) -> None:
    """The reference's error for a clip the zero-phase filters cannot pad (scipy sosfiltfilt), per clip: with the pitch
    stage on, a clip of 1..15 samples raises ValueError; a zero-length clip is not rendered."""
    n = np.asarray(lengths, dtype=np.int64)
    if p.apply and ((n > 0) & (n <= 15)).any():
        raise ValueError("The length of the input vector x must be greater than padlen, which is 15.")


def render_device(p: QdAutotuneParams, x, want_taps: bool = False, debug: bool = False, chunk_clips: int = 2048,
                  workspace=None):
    """x: CUDA float32 [B, n] -> (y, taps or None, debug dict or None, workspace tensor to hand back in next time).  Clips are rendered ``chunk_clips`` at a time:
    the mode keeps its bands in HBM (40 bytes of workspace per sample plus the YIN difference functions, about 24 MB
    per 10 s clip), and the sequential sweeps cost the same for 1 clip as for a few thousand."""
    import torch
    lib = _lib.load()
    if x.dtype != torch.float32 or x.dim() != 2 or x.shape[1] != p.n_samples or not x.is_cuda:
        raise ValueError(f"expected a CUDA float32 tensor of shape [B, {p.n_samples}]")
    x = x.contiguous()
    b, n = int(x.shape[0]), int(x.shape[1])
    y = torch.empty_like(x)
    taps = {"pre_quant": torch.empty_like(x), "post_dist": torch.empty_like(x)} if want_taps else None
    dbg = None
    if debug:
        frames = (n + p.hop - 1) // p.hop
        dbg = {k: torch.zeros_like(x) for k in ("sub", "body", "air", "det", "ratio_track", "corrected", "sub_layer")}
        dbg["features"] = torch.zeros((b, frames, 4), dtype=torch.float64, device=x.device)
    if b == 0 or n == 0:
        return y, taps, dbg, workspace
    chunk = max(1, min(int(chunk_clips), b))
    need = int(lib.qd_autotune_workspace_bytes(C.byref(p), chunk))
    ws = workspace if workspace is not None and workspace.numel() >= need and workspace.device == x.device else \
        torch.empty(need, dtype=torch.uint8, device=x.device)
    stream = torch.cuda.current_stream().cuda_stream
    for b0 in range(0, b, chunk):
        nb = min(chunk, b - b0)
        ct = _lib.QdTaps(taps["pre_quant"][b0:].data_ptr(), taps["post_dist"][b0:].data_ptr()) if taps else None
        cd = None
        if dbg:
            cd = QdAutotuneDebug(*[dbg[k][b0:].data_ptr() for k in ("sub", "body", "air", "det", "ratio_track",
                                                                     "corrected", "sub_layer", "features")])
        _lib.check(lib.qd_autotune_render_device(C.byref(p), x[b0:].data_ptr(), y[b0:].data_ptr(), nb,
                                                 C.byref(ct) if ct is not None else None,
                                                 C.byref(cd) if cd is not None else None,
                                                 ws.data_ptr(), ws.numel(), stream))
    return y, taps, dbg, ws


def render_device_varlen(p: QdAutotuneParams, x, starts, lengths, span: int, max_samples: int, want_taps: bool = False,
                         workspace=None):
    """Ragged batch on the device: x is a flat CUDA float32 tensor holding clip c at x[starts[c] - starts[0] : ... +
    lengths[c]]; starts (int64) and lengths (int32) are CUDA tensors, already validated (pipeline.check_layout and
    check_lengths) -- the library does not read them on the host.  Returns (y, taps or None, workspace) with y and
    the taps packed like x (gap samples unspecified).  One call: the workspace holds about 40 bytes per packed sample
    plus the YIN difference functions (qd_autotune_workspace_bytes_varlen)."""
    import torch
    lib = _lib.load()
    if x.dtype != torch.float32 or x.dim() != 1 or not x.is_cuda or not x.is_contiguous():
        raise ValueError("expected a contiguous flat CUDA float32 tensor")
    if (starts.dtype != torch.int64 or lengths.dtype != torch.int32 or not starts.is_cuda or not lengths.is_cuda
            or starts.shape != lengths.shape or starts.dim() != 1):
        raise ValueError("starts / lengths: CUDA int64 / int32 tensors of one length")
    if max_samples > p.n_samples:
        raise ValueError(f"a clip of {max_samples} samples is longer than this renderer's {p.n_samples}")
    batch = int(starts.shape[0])
    y = torch.empty_like(x)
    taps = {"pre_quant": torch.empty_like(x), "post_dist": torch.empty_like(x)} if want_taps else None
    if batch and span and max_samples:
        need = int(lib.qd_autotune_workspace_bytes_varlen(C.byref(p), batch, int(span)))
        ws = workspace if workspace is not None and workspace.numel() >= need and workspace.device == x.device else \
            torch.empty(need, dtype=torch.uint8, device=x.device)
        ct = _lib.QdTaps(taps["pre_quant"].data_ptr(), taps["post_dist"].data_ptr()) if taps else None
        _lib.check(lib.qd_autotune_render_device_varlen(
            C.byref(p), x.data_ptr(), y.data_ptr(), starts.data_ptr(), lengths.data_ptr(), batch, int(span),
            int(max_samples), C.byref(ct) if ct is not None else None, ws.data_ptr(), ws.numel(),
            torch.cuda.current_stream().cuda_stream))
        workspace = ws
    return y, taps, workspace
