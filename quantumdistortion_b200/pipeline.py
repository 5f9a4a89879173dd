"""Batched STFT-path renderer behind the reference's ``process_audio`` parameter API.

``process_audio(audio, sr, **kwargs)`` keeps the reference's signature and return value
(quantum_distortion/dsp/pipeline.py:1113-1155: ``(float32[n], taps)``) for one clip;
``process_batch`` renders ``[B, n]`` clips in one go, which is what the hardware wants.
The arithmetic runs in the hand-written sm_100a kernels of ``csrc/`` through the C ABI of
``include/qd_b200.h``; PyTorch only provides device memory and streams.  There is no CPU
fallback: without a B200 and the built library every call raises.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import Any, Dict, List, Optional, Sequence, Tuple, Union

import numpy as np

from . import _lib, autotune, tables
from .config import (DEFAULT_AIR_CUT_HZ, DEFAULT_BIN_SMOOTHING, DEFAULT_DISTORTION_MODE, DEFAULT_DRY_WET,
                     DEFAULT_KEY, DEFAULT_LIMITER_CEILING_DB, DEFAULT_LIMITER_ON, DEFAULT_QUANTIZE_MODE,
                     DEFAULT_SAMPLE_RATE, DEFAULT_SCALE, DEFAULT_SMEAR, DEFAULT_SNAP_STRENGTH, DEFAULT_SUB_CUT_HZ,
                     N_FFT_DEFAULT, PREVIEW_ENABLED_DEFAULT, PREVIEW_MAX_SECONDS, PipelineConfig,
                     ensure_mono_float32)

_PC_FIELDS = ("key", "scale", "quantize_mode", "snap_strength", "smear", "bin_smoothing", "pre_quant", "post_quant",
              "sub_cut_hz", "air_cut_hz", "distortion_mode", "distortion_params", "limiter_on",
              "limiter_ceiling_db", "dry_wet", "preview_enabled", "use_multiband", "crossover_hz", "lowband_drive",
              "passthrough_test", "spectral_fx_mode", "spectral_fx_strength", "spectral_fx_params",
              "spectral_freeze", "formant_shift", "harmonic_lock_hz", "delta_listen", "mono_strength",
              "output_trim_db", "sub_enabled", "sub_source", "sub_note", "sub_scale_degree", "sub_octave", "sub_level",
              "air_mix")


@dataclass
class RenderTiming:
    """Device-side timing of a render, per kernel class (cf. RenderTiming, dsp/pipeline.py:153-161, whose stft / proc /
    istft stages are one fused kernel here).  Filled by ``Renderer.timing()`` from CUDA events recorded on the launch
    stream (qd_plan_enable_timing); milliseconds since the previous call."""
    spectral_ms: float = 0.0     # STFT -> FX -> quantizer -> iSTFT -> overlap-add -> distortion (both passes)
    limiter_ms: float = 0.0      # lookahead limiter + dry/wet + trim + recombine + delta
    crossover_ms: float = 0.0    # LR4 split + low-band delay / saturation
    other_ms: float = 0.0
    total_ms: float = 0.0
    launches: int = 0

    def line(self, mode: str = "spectral_bins") -> str:
        """The reference's one-line report (dsp/pipeline.py:1382-1390), with this implementation's stages."""
        return (f"[RENDER_TIMING] mode={mode} spectral={self.spectral_ms:.3f}ms limiter={self.limiter_ms:.3f}ms "
                f"crossover={self.crossover_ms:.3f}ms total={self.total_ms:.3f}ms launches={self.launches}")


def _torch():
    import torch
    if not torch.cuda.is_available():
        raise _lib.QdError("no CUDA device visible: quantumdistortion_b200 renders only on a B200 "
                           "(there is no CPU fallback; the CPU oracle lives in oracle/ for tests)")
    return torch


def fx_tables(r: "tables.Resolved", batch: int, seeds=None, shard=None, frames: Optional[Sequence[int]] = None):
    """np.random replay tables (tables.replay_fx_table) of the random spectral FX for `batch` clips.

    ``frames`` (a ragged batch): the frame count 1 + n_c // hop of every clip.  Each clip's table is then replayed
    with its own count -- the draws a reference call on that clip makes -- and padded to the plan's r.n_frames; the
    tables are always per clip, also for an int seed (reseeded before every clip).

    seeds=None : draw from the current global np.random state, clip after clip -- what a loop of reference
                 ``process_audio`` calls would consume;
    seeds=int  : ``np.random.seed(s)`` before EVERY clip -> one table shared by the whole batch;
    seeds=[..] : one seed per clip.
    ``shard=(lo, hi, total)`` says the batch is clips lo..hi of a larger batch of `total` clips rendered elsewhere
    (multi-GPU sharding): a seed list may then cover the whole batch (it is sliced), and with seeds=None the draws of
    the clips before the shard are consumed first and those of the clips after it afterwards, so every clip gets
    the draws it would get in an unsharded render and the global state ends where that render would leave it."""
    if frames is not None:
        if shard is not None:
            raise ValueError("a ragged batch cannot be sharded")
        frames = [int(t) for t in frames]
        if len(frames) != batch or any(t < 1 or t > r.n_frames for t in frames):
            raise ValueError("need one frame count in 1..n_frames per clip")
        if isinstance(seeds, (int, np.integer)):
            seeds = [int(seeds)] * batch
        elif seeds is not None:
            seeds = list(seeds)
            if len(seeds) != batch:
                raise ValueError("need one seed per clip")
        tabs = []
        for c, t in enumerate(frames):
            if seeds is not None:
                np.random.seed(int(seeds[c]))
            tab = tables.replay_fx_table(r.fx_rng, r.fx_passes, t, r.n_bins)
            full = tables.replay_fx_table(r.fx_rng, 0, r.n_frames, r.n_bins)   # identity / zero: frames past T_c
            full[:, :t] = tab
            tabs.append(full)
        return tabs
    one = lambda: tables.replay_fx_table(r.fx_rng, r.fx_passes, r.n_frames, r.n_bins)  # noqa: E731
    lo, total = (int(shard[0]), int(shard[2])) if shard is not None else (0, batch)
    if seeds is None:
        for _ in range(lo):
            one()
        tabs = [one() for _ in range(batch)]
        for _ in range(total - lo - batch):
            one()
        return tabs
    if isinstance(seeds, (int, np.integer)):
        np.random.seed(int(seeds))
        return [one()]
    seeds = list(seeds)
    if shard is not None and len(seeds) == total:
        seeds = seeds[lo:lo + batch]
    if len(seeds) != batch:
        raise ValueError("need one seed per clip")
    tabs = []
    for sd in seeds:
        np.random.seed(int(sd))
        tabs.append(one())
    return tabs


def pack_layout(lengths: Sequence[int], itemsize: int = 4) -> Tuple[np.ndarray, int]:
    """Packed layout of a ragged batch: clip c starts at starts[c] (int64, samples), every start aligned to 16 bytes
    of ``itemsize``-byte samples; returns (starts, span) with span = starts[-1] + lengths[-1] (0 for no clips)."""
    n = np.asarray(lengths, dtype=np.int64).reshape(-1)
    if n.size == 0:
        return np.zeros(0, dtype=np.int64), 0
    if (n < 0).any():
        raise ValueError("clip lengths must be >= 0")
    align = max(1, 16 // int(itemsize))
    padded = (n + align - 1) // align * align
    starts = np.zeros(n.size, dtype=np.int64)
    np.cumsum(padded[:-1], out=starts[1:])
    return starts, int(starts[-1] + n[-1])


def clip_list_kind(clips: Sequence[Any]) -> Tuple[bool, bool]:
    """(is_numpy, on_cuda) of a list of 1-D clips: all NumPy arrays, all CPU tensors or all CUDA tensors; anything else
    raises ValueError.  Needs no device."""
    import torch
    if all(isinstance(c, np.ndarray) for c in clips):
        is_np, cuda = True, False
    elif all(isinstance(c, torch.Tensor) for c in clips):
        is_np, cuda = False, bool(clips and clips[0].is_cuda)
        if any(bool(c.is_cuda) != cuda for c in clips):
            raise ValueError("a list of clips must be all CUDA or all CPU tensors")
    else:
        raise ValueError("a list of clips must be all NumPy arrays or all tensors")
    if any(c.ndim != 1 for c in clips):
        raise ValueError("a list of clips holds 1-D (mono) clips")
    return is_np, cuda


def pack_clips(clips: Sequence[Any], cuda: bool, pcm: bool = False):
    """One buffer holding the clips in the ``pack_layout`` layout, zero in the gaps: CUDA clips with one concatenation on
    the device (cast to float32), host clips copied once into page-locked memory (float32, or int16 for PCM16), which
    is the H2D staging.  Returns (buffer, starts, span); at least one clip."""
    torch = _torch()
    lengths = np.array([int(c.shape[0]) for c in clips], dtype=np.int64)
    starts, span = pack_layout(lengths, 2 if pcm else 4)
    ends = starts + lengths
    if cuda:   # one concatenation on the device: clips and the zero gaps that align the next start
        zero = torch.zeros(4, dtype=torch.float32, device="cuda")
        pieces = []
        for k, c in enumerate(clips):
            pieces.append(c.float())
            if k + 1 < len(clips) and starts[k + 1] > ends[k]:
                pieces.append(zero[:int(starts[k + 1] - ends[k])])
        return torch.cat(pieces), starts, span
    xf = torch.empty(span, dtype=torch.int16 if pcm else torch.float32, pin_memory=True)
    xn = xf.numpy()
    for k, c in enumerate(clips):
        xn[starts[k]:ends[k]] = c if isinstance(c, np.ndarray) else c.numpy()
        if k + 1 < len(clips):
            xn[ends[k]:starts[k + 1]] = 0
    return xf, starts, span


def check_layout(starts, lengths, max_samples: int) -> None:
    """The rules of qd_render_*_varlen (include/qd_b200.h) on host arrays: starts non-decreasing, clips not
    overlapping, 0 <= length <= max_samples.  Raises ValueError; the device entry point does not check them."""
    st = np.asarray(starts)
    ln = np.asarray(lengths)
    if st.ndim != 1 or st.shape != ln.shape:
        raise ValueError("starts and lengths must be 1-D and of one length")
    if (ln < 0).any():
        raise ValueError("clip lengths must be >= 0")
    if (ln > int(max_samples)).any():
        raise ValueError(f"a clip is longer than the renderer's {int(max_samples)} samples")
    if st.size > 1 and (st[1:].astype(np.int64) < st[:-1].astype(np.int64) + ln[:-1].astype(np.int64)).any():
        raise ValueError("clip starts must be non-decreasing and clips must not overlap")


class Renderer:
    """One resolved parameter set bound to a CUDA plan on the current device."""

    def __init__(self, resolved: tables.Resolved):
        self._lib = _lib.load()
        self.resolved = resolved
        self.n = int(resolved.params.n_samples)
        handle = C.c_void_p()
        _lib.check(self._lib.qd_plan_create(C.byref(resolved.params),
                                            C.byref(resolved.tables) if resolved.tables is not None else None,
                                            C.byref(handle)))
        self._plan = handle
        self._ws = None
        self.launches_per_render = int(self._lib.qd_plan_launches_per_render(self._plan))

    def close(self) -> None:
        if getattr(self, "_plan", None):
            self._lib.qd_plan_destroy(self._plan)
            self._plan = None

    def __del__(self):  # best effort
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def enable_timing(self, on: bool = True) -> None:
        """Bracket every kernel class with CUDA events on the launch stream (qd_plan_enable_timing)."""
        _lib.check(self._lib.qd_plan_enable_timing(self._plan, int(on)))

    def read_timing(self) -> Dict[str, Dict[str, float]]:
        """Milliseconds and launch counts per kernel class since the last read (waits for the events)."""
        ms, cnt = (C.c_double * 4)(), (C.c_int64 * 4)()
        _lib.check(self._lib.qd_plan_read_timing(self._plan, C.byref(ms), C.byref(cnt)))
        names = ("spectral", "limiter", "crossover", "other")
        return {n: {"ms": float(ms[i]), "launches": int(cnt[i])} for i, n in enumerate(names)}

    def timing(self) -> RenderTiming:
        """RenderTiming of the renders since the last call (needs enable_timing(True); waits for the events)."""
        t = self.read_timing()
        ms = {k: v["ms"] for k, v in t.items()}
        return RenderTiming(spectral_ms=ms["spectral"], limiter_ms=ms["limiter"], crossover_ms=ms["crossover"],
                            other_ms=ms["other"], total_ms=sum(ms.values()),
                            launches=sum(v["launches"] for v in t.values()))

    def _workspace(self, batch: int):
        torch = _torch()
        need = int(self._lib.qd_plan_workspace_bytes(self._plan, batch))
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device="cuda")
        return self._ws, need

    def set_fx_seeds(self, batch: int, seeds=None, shard=None, frames: Optional[Sequence[int]] = None) -> None:
        """Replay the reference's np.random draws for the spectral FX (fx_tables) and upload them.  ``frames``: per-clip
        frame counts of a ragged batch (per-clip tables; the renderer must come from make_renderer(..., ragged=True))."""
        r = self.resolved
        if not r.fx_rng:
            return
        torch = _torch()
        tabs = fx_tables(r, batch, seeds, shard, frames)
        shared = isinstance(seeds, (int, np.integer)) and frames is None
        if bool(r.params.fx_table_per_clip) == shared:
            raise ValueError("renderer built for %s FX tables; use make_renderer(..., seeds=...) with the same kind of seeds"
                             % ("per-clip" if r.params.fx_table_per_clip else "shared"))
        self._fx_table = torch.from_numpy(np.ascontiguousarray(np.stack(tabs))).cuda()
        _lib.check(self._lib.qd_plan_set_fx_table(self._plan, self._fx_table.data_ptr(), len(tabs)))

    def render_device(self, x, want_taps: bool = False):
        """x: CUDA float32 tensor [B, n] -> (y [B, n], taps or None).  Asynchronous on the current stream."""
        torch = _torch()
        if x.dtype != torch.float32 or x.dim() != 2 or x.shape[1] != self.n or not x.is_cuda:
            raise ValueError(f"expected a CUDA float32 tensor of shape [B, {self.n}]")
        x = x.contiguous()
        batch = int(x.shape[0])
        y = torch.empty_like(x)
        taps = None
        ctaps = None
        if want_taps:
            taps = {"pre_quant": torch.empty_like(x), "post_dist": torch.empty_like(x)}
            ctaps = _lib.QdTaps(taps["pre_quant"].data_ptr(), taps["post_dist"].data_ptr())
        if batch and self.n:
            ws, need = self._workspace(batch)
            stream = torch.cuda.current_stream().cuda_stream
            _lib.check(self._lib.qd_render_device(self._plan, x.data_ptr(), y.data_ptr(), batch,
                                                  C.byref(ctaps) if ctaps is not None else None,
                                                  ws.data_ptr(), need, stream))
        return y, taps

    def render_device_varlen(self, x, starts, lengths, span: int, max_samples: int, want_taps: bool = False):
        """Ragged batch on the device: x is a flat CUDA float32 tensor holding clip c at
        x[starts[c] - starts[0] : ... + lengths[c]]; starts (int64) and lengths (int32) are CUDA tensors, already
        validated (pack_clips) -- the library does not read them on the host.  Returns (y, taps) packed like x (gap
        samples unspecified).  Asynchronous on the current stream."""
        torch = _torch()
        if x.dtype != torch.float32 or x.dim() != 1 or not x.is_cuda or not x.is_contiguous():
            raise ValueError("expected a contiguous flat CUDA float32 tensor")
        if (starts.dtype != torch.int64 or lengths.dtype != torch.int32 or not starts.is_cuda or not lengths.is_cuda
                or starts.shape != lengths.shape or starts.dim() != 1):
            raise ValueError("starts / lengths: CUDA int64 / int32 tensors of one length")
        if max_samples > self.n:
            raise ValueError(f"a clip of {max_samples} samples is longer than this renderer's {self.n}")
        batch = int(starts.shape[0])
        y = torch.empty_like(x)
        taps = None
        ctaps = None
        if want_taps:
            taps = {"pre_quant": torch.empty_like(x), "post_dist": torch.empty_like(x)}
            ctaps = _lib.QdTaps(taps["pre_quant"].data_ptr(), taps["post_dist"].data_ptr())
        if batch and span and max_samples:
            need = int(self._lib.qd_plan_workspace_bytes_varlen(self._plan, batch, int(span)))
            if self._ws is None or self._ws.numel() < need:
                self._ws = torch.empty(need, dtype=torch.uint8, device="cuda")
            stream = torch.cuda.current_stream().cuda_stream
            _lib.check(self._lib.qd_render_device_varlen(
                self._plan, x.data_ptr(), y.data_ptr(), starts.data_ptr(), lengths.data_ptr(), batch, int(span),
                int(max_samples), C.byref(ctaps) if ctaps is not None else None, self._ws.data_ptr(), need, stream))
        return y, taps

    def render_host_varlen(self, x_host, y_host, starts: np.ndarray, lengths: np.ndarray, chunk_samples: int = 0) -> None:
        """Ragged batch in host memory: flat contiguous CPU tensors x_host / y_host (float32 or int16 PCM16, like
        render_host) with clip c at [starts[c] - starts[0], + lengths[c]); starts / lengths: NumPy int64 / int32.
        Chunks are clip ranges whose packed span fits ``chunk_samples`` (0: 128 clips of this renderer's length).
        The library validates starts / lengths.  Synchronous."""
        torch = _torch()
        fmt = {torch.float32: 0, torch.int16: 1}
        if x_host.dtype not in fmt or y_host.dtype not in fmt:
            raise ValueError("host buffers must be float32 or int16 (PCM16)")
        if (x_host.dim() != 1 or x_host.shape != y_host.shape or not x_host.is_contiguous()
                or not y_host.is_contiguous()):
            raise ValueError("x_host and y_host must be flat, contiguous and of the same length")
        starts = np.ascontiguousarray(starts, dtype=np.int64)
        lengths = np.ascontiguousarray(lengths, dtype=np.int32)
        if starts.shape != lengths.shape or starts.ndim != 1:
            raise ValueError("starts and lengths must be 1-D and of one length")
        if len(starts) and int(starts[-1] - starts[0]) + int(lengths[-1]) > int(x_host.shape[0]):
            raise ValueError("the clips reach past the end of the host buffers")
        _lib.check(self._lib.qd_render_host_varlen(self._plan, x_host.data_ptr(), y_host.data_ptr(),
                                                   starts.ctypes.data, lengths.ctypes.data, len(starts),
                                                   int(chunk_samples), fmt[x_host.dtype], fmt[y_host.dtype]))

    def render_host(self, x_host, y_host, chunk_clips: int = 128) -> None:
        """x_host / y_host: contiguous CPU tensors [B, n], float32 or int16 (16-bit PCM, converted on the device with
        the WAV layer's rules: half the PCIe bytes).  Pinned memory is copied directly; pageable memory is staged
        through the library's pinned ring by copy threads.  Synchronous; H2D, kernels and D2H of consecutive chunks
        overlap inside the library (qd_render_host_ex)."""
        torch = _torch()
        fmt = {torch.float32: 0, torch.int16: 1}
        if x_host.dtype not in fmt or y_host.dtype not in fmt:
            raise ValueError("host buffers must be float32 or int16 (PCM16)")
        if x_host.shape != y_host.shape or not x_host.is_contiguous() or not y_host.is_contiguous():
            raise ValueError("x_host and y_host must be contiguous and of the same [B, n] shape")
        batch = int(x_host.shape[0])
        _lib.check(self._lib.qd_render_host_ex(self._plan, x_host.data_ptr(), y_host.data_ptr(), batch, int(chunk_clips),
                                               fmt[x_host.dtype], fmt[y_host.dtype]))


class AutotuneRenderer:
    """``quantize_mode="autotune_v1"`` (the reference's default mode) with the Renderer interface."""

    launches_per_render = 16

    def __init__(self, params: "autotune.QdAutotuneParams"):
        _lib.load()
        self.params = params
        self.n = int(params.n_samples)
        self._ws = None   # device workspace, kept between renders

    def close(self) -> None:
        self._ws = None

    def set_fx_seeds(self, batch: int, seeds=None, shard=None, frames: Optional[Sequence[int]] = None) -> None:
        pass   # no random stage in this mode

    def render_device(self, x, want_taps: bool = False, debug: bool = False, chunk_clips: int = 2048):
        _torch()
        y, taps, dbg, self._ws = autotune.render_device(self.params, x, want_taps=want_taps, debug=debug,
                                                        chunk_clips=chunk_clips, workspace=self._ws)
        return (y, taps, dbg) if debug else (y, taps)

    def render_device_varlen(self, x, starts, lengths, span: int, max_samples: int, want_taps: bool = False):
        """Ragged batch on the device, as Renderer.render_device_varlen (autotune.render_device_varlen)."""
        _torch()
        y, taps, self._ws = autotune.render_device_varlen(self.params, x, starts, lengths, span, max_samples,
                                                          want_taps=want_taps, workspace=self._ws)
        return y, taps

    def render_host_varlen(self, x_host, y_host, starts: np.ndarray, lengths: np.ndarray, chunk_samples: int = 0) -> None:
        """Ragged batch in host memory, as Renderer.render_host_varlen: flat contiguous CPU tensors (float32 or int16
        PCM16) with clip c at [starts[c] - starts[0], + lengths[c]).  Chunks are clip ranges whose packed span fits
        ``chunk_samples`` (0: 128 clips of this renderer's length; a longer clip gets a chunk of its own), and the
        copies overlap the kernels as in render_host.  Validates starts / lengths.  Synchronous."""
        torch = _torch()
        fmt = (torch.float32, torch.int16)
        if x_host.dtype not in fmt or y_host.dtype not in fmt:
            raise ValueError("host buffers must be float32 or int16 (PCM16)")
        if (x_host.dim() != 1 or x_host.shape != y_host.shape or not x_host.is_contiguous()
                or not y_host.is_contiguous()):
            raise ValueError("x_host and y_host must be flat, contiguous and of the same length")
        starts = np.ascontiguousarray(starts, dtype=np.int64)
        lengths = np.ascontiguousarray(lengths, dtype=np.int32)
        check_layout(starts, lengths, self.n)
        autotune.check_lengths(self.params, lengths)
        if not len(starts):
            return
        off = starts - starts[0]
        ends = off + lengths
        if int(ends[-1]) > int(x_host.shape[0]):
            raise ValueError("the clips reach past the end of the host buffers")
        budget = int(chunk_samples) if chunk_samples > 0 else 128 * max(1, self.n)
        d_starts, d_lengths = torch.from_numpy(starts).cuda(), torch.from_numpy(lengths).cuda()
        run = torch.cuda.current_stream()
        if not hasattr(self, "_s_in"):
            self._s_in, self._s_out = torch.cuda.Stream(), torch.cuda.Stream()
        s_in, s_out = self._s_in, self._s_out
        s_in.wait_stream(run)
        c0 = 0
        while c0 < len(starts):
            c1 = c0 + 1
            while c1 < len(starts) and ends[c1] - off[c0] <= budget:
                c1 += 1
            lo, hi = int(off[c0]), int(ends[c1 - 1])
            with torch.cuda.stream(s_in):
                xs = x_host[lo:hi].to("cuda", non_blocking=True)
            run.wait_stream(s_in)
            xs.record_stream(run)
            if xs.dtype == torch.int16:
                xs = xs.to(torch.float32) * (1.0 / 32768.0)
            y, _ = self.render_device_varlen(xs.float(), d_starts[c0:c1], d_lengths[c0:c1], hi - lo,
                                             int(lengths[c0:c1].max()))
            if y_host.dtype == torch.int16:
                y = torch.clamp(torch.round(y.double() * 32767.0), -32768.0, 32767.0).to(torch.int16)
            s_out.wait_stream(run)
            with torch.cuda.stream(s_out):
                y_host[lo:hi].copy_(y, non_blocking=True)
            y.record_stream(s_out)
            c0 = c1
        s_out.synchronize()
        run.synchronize()

    def render_host(self, x_host, y_host, chunk_clips: int = 128) -> None:
        """Chunked H2D -> render -> D2H with the copies on their own streams, so that the transfers of chunk i+1 / i-1
        run under the kernels of chunk i (pinned host tensors).  float32 or int16 (PCM16, converted on the device:
        sample / 32768 in, rint(y * 32767) clipped out -- the rules of audio_io)."""
        torch = _torch()
        run = torch.cuda.current_stream()
        if not hasattr(self, "_s_in"):
            self._s_in, self._s_out = torch.cuda.Stream(), torch.cuda.Stream()
        s_in, s_out = self._s_in, self._s_out
        s_in.wait_stream(run)
        for b0 in range(0, int(x_host.shape[0]), int(chunk_clips)):
            with torch.cuda.stream(s_in):
                xs = x_host[b0:b0 + chunk_clips].to("cuda", non_blocking=True)
            run.wait_stream(s_in)
            xs.record_stream(run)
            if xs.dtype == torch.int16:
                xs = xs.to(torch.float32) * (1.0 / 32768.0)
            y, _ = self.render_device(xs.float(), chunk_clips=chunk_clips)
            if y_host.dtype == torch.int16:
                y = torch.clamp(torch.round(y.double() * 32767.0), -32768.0, 32767.0).to(torch.int16)
            s_out.wait_stream(run)
            with torch.cuda.stream(s_out):
                y_host[b0:b0 + chunk_clips].copy_(y, non_blocking=True)
            y.record_stream(s_out)
        s_out.synchronize()
        run.synchronize()


_RENDERERS: Dict[Any, Renderer] = {}


def _renderer_for(resolved: tables.Resolved) -> Renderer:
    torch = _torch()
    key = (torch.cuda.current_device(), bytes(resolved.params),
           None if resolved.tables is None else (resolved.target_bins.tobytes(), resolved.active_mask.tobytes(),
                                                 resolved.tables.snap, resolved.tables.smear))
    r = _RENDERERS.get(key)
    if r is None:
        if len(_RENDERERS) > 32:
            _RENDERERS.pop(next(iter(_RENDERERS))).close()
        r = _RENDERERS[key] = Renderer(resolved)
    return r


def _parse_ui_config(config: Dict[str, Any], kw: Dict[str, Any]) -> Dict[str, Any]:
    """dsp/pipeline.py:923-1008: the Streamlit V2 UI dict -> keyword overrides.  A UI dict always means a
    multiband render; in "high_band" the first non-zero of bin_scrambling / phase_dispersal / mag_decimation
    (defaults 0.2 / 0.3 / 0.5) selects the single active spectral FX."""
    out: Dict[str, Any] = {"use_multiband": True, "low_trim_db": 0.0}
    if "quantization" in config:
        q = config["quantization"]
        out["key"] = str(q.get("key", kw.get("key", DEFAULT_KEY)))
        out["scale"] = str(q.get("scale", kw.get("scale", DEFAULT_SCALE)))
        out["quantize_mode"] = str(q.get("mode", kw.get("quantize_mode", DEFAULT_QUANTIZE_MODE)))
        out["sub_enabled"] = bool(q.get("sub_enabled", kw.get("sub_enabled", True)))          # :966-974: the
        out["sub_source"] = str(q.get("sub_source", kw.get("sub_source", "root")))            # autotune_v1 sub layer
        out["sub_note"] = str(q.get("sub_note", kw.get("sub_note", "C")))
        out["sub_scale_degree"] = int(q.get("sub_scale_degree", kw.get("sub_scale_degree", 0)))
        out["sub_octave"] = int(q.get("sub_octave", kw.get("sub_octave", 2)))
        out["sub_level"] = float(q.get("sub_level", kw.get("sub_level", 0.35)))
        out["sub_cut_hz"] = float(q.get("sub_cut_hz", kw.get("sub_cut_hz", DEFAULT_SUB_CUT_HZ)))
        out["air_cut_hz"] = float(q.get("air_cut_hz", kw.get("air_cut_hz", DEFAULT_AIR_CUT_HZ)))
        out["air_mix"] = float(q.get("air_mix", kw.get("air_mix", 1.0)))
    if "crossover_freq" in config:
        out["crossover_hz"] = float(config["crossover_freq"])
    if "low_band" in config:
        lb = config["low_band"]
        out["lowband_drive"] = 1.0 + (lb.get("saturation_amount", 0.3) * 4.0)
        out["mono_strength"] = float(lb.get("mono_strength", kw.get("mono_strength", 1.0)))
        out["low_trim_db"] = float(lb.get("output_trim_db", 0.0))
    if "high_band" in config:
        hb = config["high_band"]
        scr, dis, dec = hb.get("bin_scrambling", 0.2), hb.get("phase_dispersal", 0.3), hb.get("mag_decimation", 0.5)
        if scr > 0.0:
            out["spectral_fx_mode"], out["spectral_fx_strength"] = "bin_scramble", scr
        elif dis > 0.0:
            out["spectral_fx_mode"], out["spectral_fx_strength"] = "phase_dispersal", dis
        elif dec > 0.0:
            out["spectral_fx_mode"], out["spectral_fx_strength"] = "bitcrush", dec
        out["output_trim_db"] = float(hb.get("output_trim_db", kw.get("output_trim_db", 0.0)))
    if "quantum_fx" in config:
        qf = config["quantum_fx"]
        out["spectral_freeze"] = bool(qf.get("spectral_freeze", kw.get("spectral_freeze", False)))
        out["formant_shift"] = float(qf.get("formant_shift", kw.get("formant_shift", 0.0)))
        out["harmonic_lock_hz"] = float(qf.get("fundamental_hz", kw.get("harmonic_lock_hz", 0.0)))
    if "delta_listen" in config:
        out["delta_listen"] = bool(config["delta_listen"])
    return out


def _resolve_kwargs(n_samples: int, sr: int, n_fft: int, kw: Dict[str, Any]) -> Tuple[tables.Resolved, Dict[str, Any]]:
    """Apply the reference's argument rules (dsp/pipeline.py:1201-1327) and build the C structs."""
    pc = kw.pop("pipeline_config", None)
    if pc is not None:  # overrides every individual keyword (:1201-1238)
        for f in _PC_FIELDS:
            kw[f] = getattr(pc, f)
    ui = kw.pop("config", None)
    if ui is not None:  # Streamlit V2 nested dict: overrides a subset of the keywords (:1264-1300)
        kw.update(_parse_ui_config(ui, kw))
    g = lambda k, d: kw.pop(k, d)  # noqa: E731
    key, scale = g("key", DEFAULT_KEY), g("scale", DEFAULT_SCALE)
    quantize_mode = g("quantize_mode", DEFAULT_QUANTIZE_MODE)
    snap, smear = g("snap_strength", DEFAULT_SNAP_STRENGTH), g("smear", DEFAULT_SMEAR)
    bin_smoothing = g("bin_smoothing", DEFAULT_BIN_SMOOTHING)
    pre_quant, post_quant = g("pre_quant", True), g("post_quant", True)
    distortion_mode = g("distortion_mode", DEFAULT_DISTORTION_MODE)
    distortion_params = g("distortion_params", None) or {}
    limiter_on, ceiling_db = g("limiter_on", DEFAULT_LIMITER_ON), g("limiter_ceiling_db", DEFAULT_LIMITER_CEILING_DB)
    dry_wet = g("dry_wet", DEFAULT_DRY_WET)
    use_multiband, crossover_hz = g("use_multiband", False), g("crossover_hz", 300.0)
    lowband_drive = g("lowband_drive", 1.0)
    passthrough = g("passthrough_test", False)
    fx_mode, fx_strength = g("spectral_fx_mode", None), g("spectral_fx_strength", 0.0)
    fx_params = g("spectral_fx_params", None) or {}
    freeze, formant, lock_hz = g("spectral_freeze", False), g("formant_shift", 0.0), g("harmonic_lock_hz", 0.0)
    delta_listen, mono_strength = g("delta_listen", False), g("mono_strength", 1.0)
    trim_db = g("output_trim_db", 0.0)
    sub_cut, air_cut = g("sub_cut_hz", DEFAULT_SUB_CUT_HZ), g("air_cut_hz", DEFAULT_AIR_CUT_HZ)
    low_trim_db = g("low_trim_db", 0.0)
    precision = g("precision", "auto")
    g("preview_enabled", None)
    sub_kw = {k: g(k, d) for k, d in (("sub_enabled", True), ("sub_source", "root"), ("sub_note", "C"),
                                      ("sub_scale_degree", 0), ("sub_octave", 2), ("sub_level", 0.35),
                                      ("air_mix", 1.0))}  # autotune-only fields (config.py:80-89)
    if kw:
        raise TypeError(f"process_audio() got unexpected keyword arguments: {sorted(kw)}")
    if quantize_mode == "autotune_v1" and (fx_mode is not None or freeze or formant != 0.0 or lock_hz > 0.0):
        quantize_mode = "spectral_bins"  # :1315-1324
    if quantize_mode == "autotune_v1" and snap > 0.0:
        use_multiband = False  # :1326-1327, ahead of every branch: also a passthrough_test render is single band then
    no_spectral = False
    if quantize_mode == "autotune_v1" and not passthrough and use_multiband and not snap > 0.0:
        # :1326-1327 only forces single band when snap > 0; with snap <= 0 the high band of the multiband render goes
        # through the autotune branch with its pitch stage gated off (:538, :570): band -> distortion -> limiter -> mix
        no_spectral = True
    elif quantize_mode == "autotune_v1" and not passthrough:   # dsp/pipeline.py:537-601 (after the passthrough branch :477)
        ap = autotune.resolve(sr=sr, n_samples=n_samples, key=key, scale=scale, snap_strength=snap,
                              pre_quant=pre_quant, distortion_mode=distortion_mode,
                              distortion_params=distortion_params, limiter_on=limiter_on,
                              limiter_ceiling_db=ceiling_db, dry_wet=dry_wet, output_trim_db=trim_db,
                              delta_listen=delta_listen, sub_cut_hz=sub_cut, air_cut_hz=air_cut, **sub_kw)
        return ap, {}
    if quantize_mode not in ("spectral_bins", "autotune_v1"):
        raise NotImplementedError(f"unknown quantize_mode {quantize_mode!r}: 'spectral_bins' and 'autotune_v1' are built")
    res = tables.resolve(sr=sr, n_samples=n_samples, n_fft=n_fft, key=key, scale=scale, snap_strength=snap,
                         smear=smear, bin_smoothing=bin_smoothing, pre_quant=pre_quant, post_quant=post_quant,
                         distortion_mode=distortion_mode, distortion_params=distortion_params,
                         limiter_on=limiter_on, limiter_ceiling_db=ceiling_db, dry_wet=dry_wet,
                         use_multiband=use_multiband, crossover_hz=crossover_hz, lowband_drive=lowband_drive,
                         passthrough_test=passthrough, harmonic_lock_hz=lock_hz, delta_listen=delta_listen,
                         mono_strength=mono_strength, output_trim_db=trim_db, low_trim_db=low_trim_db,
                         sub_cut_hz=sub_cut, air_cut_hz=air_cut, spectral_fx_mode=fx_mode,
                         spectral_fx_strength=fx_strength, spectral_fx_params=fx_params, precision=precision,
                         spectral_freeze=bool(freeze), formant_shift=float(formant), no_spectral=no_spectral)
    return res, {"fx_params": fx_params}


def make_renderer(n_samples: int, sr: int = DEFAULT_SAMPLE_RATE, n_fft: int = N_FFT_DEFAULT, seeds=None,
                  ragged: bool = False, **kwargs) -> Renderer:
    """Resolve the reference keyword arguments once and return the cached CUDA renderer.  ``seeds`` only
    matters for the random spectral FX (see Renderer.set_fx_seeds): an int selects one shared table, unless
    ``ragged`` (a renderer for clips of up to ``n_samples``, Renderer.render_*_varlen): per-clip tables always."""
    res, _ = _resolve_kwargs(int(n_samples), int(sr), int(n_fft), dict(kwargs))
    if isinstance(res, autotune.QdAutotuneParams):
        torch = _torch()
        key = ("autotune_v1", torch.cuda.current_device(), bytes(res))
        r = _RENDERERS.get(key)
        if r is None:
            if len(_RENDERERS) > 32:
                _RENDERERS.pop(next(iter(_RENDERERS))).close()
            r = _RENDERERS[key] = AutotuneRenderer(res)
        return r
    if res.fx_rng:
        res.params.fx_table_per_clip = 0 if isinstance(seeds, (int, np.integer)) and not ragged else 1
    return _renderer_for(res)


def _ragged_batch(clips: List[Any], sr: int, n_fft: int, return_taps: bool, chunk_clips: int, seeds, kwargs):
    """process_batch on a list of 1-D clips of any lengths (see there)."""
    torch = _torch()
    is_np, cuda = clip_list_kind(clips)
    pcm_of = (lambda c: c.dtype == np.int16) if is_np else (lambda c: c.dtype == torch.int16)  # noqa: E731
    pcm = bool(clips) and pcm_of(clips[0])
    if any(pcm_of(c) != pcm for c in clips):
        raise ValueError("a list of clips is all int16 (PCM16) or all floating point")
    if pcm and (cuda or return_taps):
        raise ValueError("int16 (PCM16) input is the host transport format: CPU arrays only, no taps")
    lengths = np.array([int(c.shape[0]) for c in clips], dtype=np.int64)
    if seeds is not None and not isinstance(seeds, (int, np.integer)):
        seeds = list(seeds)
        if len(seeds) != len(clips):
            raise ValueError("need one seed per clip")
    out_dtype = (np.int16 if pcm else np.float32) if is_np else (torch.int16 if pcm else torch.float32)

    def empty():
        if is_np:
            return np.zeros(0, dtype=out_dtype)
        return torch.zeros(0, dtype=out_dtype, device="cuda" if cuda else "cpu")

    r = make_renderer(int(lengths.max()) if len(clips) else 0, sr, n_fft, seeds=seeds, ragged=True, **kwargs)
    ys: List[Any] = [None] * len(clips)
    taps: Optional[Dict[str, List[Any]]] = {"pre_quant": [None] * len(clips), "post_dist": [None] * len(clips)} \
        if return_taps else None
    live = [i for i in range(len(clips)) if lengths[i] > 0]
    if isinstance(r, AutotuneRenderer):
        autotune.check_lengths(r.params, lengths)
    if live:
        n_live = lengths[live]
        hop = int(n_fft) // 4
        r.set_fx_seeds(len(live), [seeds[i] for i in live] if isinstance(seeds, list) else seeds,
                       frames=[1 + int(n) // hop for n in n_live])
        xf, starts, span = pack_clips([clips[i] for i in live], cuda, pcm)
        max_n = int(n_live.max())
        ends = starts + n_live
        if cuda or return_taps:
            d_starts = torch.from_numpy(starts).cuda()
            d_lengths = torch.from_numpy(n_live.astype(np.int32)).cuda()
            yf, tf = r.render_device_varlen(xf if cuda else xf.cuda().float(), d_starts, d_lengths, span, max_n,
                                            want_taps=return_taps)
            if not cuda:
                yf, tf = yf.cpu(), {k: v.cpu() for k, v in tf.items()}
        else:
            yf, tf = torch.empty_like(xf, pin_memory=True), None
            r.render_host_varlen(xf, yf, starts, n_live, chunk_samples=int(chunk_clips) * max(1, span // len(live)))
        if is_np:
            yf, tf = yf.numpy(), (None if tf is None else {k: v.numpy() for k, v in tf.items()})
        for k, i in enumerate(live):
            ys[i] = yf[starts[k]:ends[k]]
            if taps is not None:
                for name in taps:
                    taps[name][i] = tf[name][starts[k]:ends[k]]
    for i in range(len(clips)):
        if ys[i] is None:   # zero-length clip: not rendered, consumes no FX draws
            ys[i] = empty()
            if taps is not None:
                for name in taps:
                    taps[name][i] = empty()
    return ys, taps


def process_batch(x, sr: int = DEFAULT_SAMPLE_RATE, *, n_fft: int = N_FFT_DEFAULT, return_taps: bool = False,
                  chunk_clips: int = 128, out=None, seeds=None, shard=None, **kwargs):
    """Render a batch of mono clips ``x[B, n]`` with one parameter set.

    ``x`` may also be a list or tuple of 1-D clips of any lengths (a ragged batch): all NumPy arrays, all CPU tensors
    or all CUDA tensors, floating point or all int16 (PCM16, host only).  The result is a list of the same kind, and
    the taps (``return_taps``) a dict of lists; a zero-length clip comes back empty.  Each clip renders exactly as it
    would alone: the STFT path packs the clips into one flat buffer and renders them in one call
    (qd_render_*_varlen, and qd_autotune_render_device_varlen in ``quantize_mode="autotune_v1"``), sized for the
    longest clip, with ``chunk_clips`` clips of mean length per host chunk.  Random spectral FX always get one table
    per clip, replayed over that clip's own frames: seeds=None draws clip after clip in list order (a loop of
    process_audio calls), an int reseeds before every clip, a list gives one seed per clip.  ``shard`` and ``out``
    are not supported with a list.  In ``autotune_v1`` with the pitch stage on, a clip of 1..15 samples raises the
    ValueError it raises alone.

    ``seeds`` controls the np.random replay of the random spectral FX (None: consume the global state clip by
    clip like a loop of reference calls; int: reseed before every clip; list: one seed per clip); ``shard=(lo, hi,
    total)`` marks ``x`` as clips lo..hi of a larger batch rendered across several processes (see fx_tables).
    ``x`` may be a CUDA tensor (returns CUDA tensors, asynchronous), a CPU tensor or a NumPy array
    (returns the same kind; the copy/compute pipeline of ``qd_render_host_ex`` is used when no taps are
    requested: pinned tensors are copied directly, pageable ones -- every NumPy array -- go through the
    library's pinned staging ring).  An int16 array / tensor is 16-bit PCM: it crosses PCIe as int16 and the
    result comes back as int16, converted on the device with the WAV layer's rules (audio_io).  ``out`` (CPU
    tensor, ideally pinned like ``x``) receives the result of the host path without a fresh allocation.  Keyword arguments are the reference's ``process_audio`` arguments.
    """
    if isinstance(x, (list, tuple)):
        if shard is not None:
            raise ValueError("shard= is not supported for a list of clips")
        if out is not None:
            raise ValueError("out= is not supported for a list of clips")
        return _ragged_batch(list(x), sr, n_fft, return_taps, chunk_clips, seeds, kwargs)
    torch = _torch()
    is_np = isinstance(x, np.ndarray)
    if is_np:
        pcm = x.dtype == np.int16
        xt = torch.from_numpy(np.ascontiguousarray(x, dtype=np.int16 if pcm else np.float32))
    else:
        xt, pcm = x, x.dtype == torch.int16
    if xt.dim() != 2:
        raise ValueError("process_batch expects [batch, samples]")
    if pcm and (xt.is_cuda or return_taps):
        raise ValueError("int16 (PCM16) input is the host transport format: CPU arrays only, no taps")
    r = make_renderer(xt.shape[1], sr, n_fft, seeds=seeds, **kwargs)
    r.set_fx_seeds(int(xt.shape[0]), seeds, shard)  # no-op unless a random spectral FX is active
    if xt.is_cuda:
        return r.render_device(xt.float(), want_taps=return_taps)
    if return_taps:
        y, taps = r.render_device(xt.float().cuda(), want_taps=True)
        y, taps = y.cpu(), {k: v.cpu() for k, v in taps.items()}
    else:
        xin = (xt if pcm else xt.float()).contiguous()
        if out is not None:
            if out.shape != xin.shape or out.dtype not in (torch.float32, torch.int16) or out.is_cuda or not out.is_contiguous():
                raise ValueError("out must be a contiguous CPU float32 (or int16) tensor shaped like x")
            y = out
        else:
            # the result lands in page-locked memory straight from the device (torch's host allocator caches the
            # block, so repeated renders do not pay the page-locking again); a pageable INPUT goes through the
            # library's staging ring
            y = torch.empty_like(xin, pin_memory=True)
        r.render_host(xin, y, chunk_clips=chunk_clips)
        taps = None
    if is_np:
        return y.numpy(), (None if taps is None else {k: v.numpy() for k, v in taps.items()})
    return y, taps


def preview_truncate(audio: np.ndarray, sr: int, preview_enabled: Optional[bool] = None,
                     pipeline_config: Optional[PipelineConfig] = None) -> np.ndarray:
    """dsp/pipeline.py:1241-1249, :1303-1310: preview mode (argument, else PipelineConfig, else the DSP_PREVIEW_MODE
    environment variable) keeps the first PREVIEW_MAX_SECONDS of the clip."""
    if preview_enabled is None and pipeline_config is not None:
        preview_enabled = pipeline_config.preview_enabled
    if preview_enabled is None:
        env = os.getenv("DSP_PREVIEW_MODE", "").strip().lower()
        preview_enabled = True if env in ("1", "true", "yes", "on") else PREVIEW_ENABLED_DEFAULT
    if preview_enabled:
        max_samples = int(sr * PREVIEW_MAX_SECONDS)
        if audio.shape[0] > max_samples:
            audio = audio[:max_samples]
    return audio


def process_audio(audio: np.ndarray, sr: int = DEFAULT_SAMPLE_RATE, key: str = DEFAULT_KEY, scale: str = DEFAULT_SCALE,
                  quantize_mode: str = DEFAULT_QUANTIZE_MODE, snap_strength: float = DEFAULT_SNAP_STRENGTH,
                  smear: float = DEFAULT_SMEAR, bin_smoothing: bool = DEFAULT_BIN_SMOOTHING, pre_quant: bool = True,
                  post_quant: bool = True, distortion_mode: str = DEFAULT_DISTORTION_MODE,
                  distortion_params: Optional[Dict[str, Any]] = None, limiter_on: bool = DEFAULT_LIMITER_ON,
                  limiter_ceiling_db: float = DEFAULT_LIMITER_CEILING_DB, dry_wet: float = DEFAULT_DRY_WET,
                  preview_enabled: Optional[bool] = None, use_multiband: bool = False, crossover_hz: float = 300.0,
                  lowband_drive: float = 1.0, passthrough_test: bool = False,
                  spectral_fx_mode: Optional[str] = None, spectral_fx_strength: float = 0.0,
                  spectral_fx_params: Optional[Dict[str, Any]] = None, config: Optional[Dict[str, Any]] = None,
                  spectral_freeze: bool = False, formant_shift: float = 0.0, harmonic_lock_hz: float = 0.0,
                  delta_listen: bool = False, mono_strength: float = 1.0, output_trim_db: float = 0.0,
                  sub_enabled: bool = True, sub_source: str = "root", sub_note: str = "C",
                  sub_scale_degree: int = 0, sub_octave: int = 2, sub_level: float = 0.35,
                  sub_cut_hz: float = DEFAULT_SUB_CUT_HZ, air_cut_hz: float = DEFAULT_AIR_CUT_HZ,
                  air_mix: float = 1.0, *, pipeline_config: Optional[PipelineConfig] = None,
                  n_fft: int = N_FFT_DEFAULT, precision: str = "auto") -> Tuple[np.ndarray, Dict[str, np.ndarray]]:
    """Drop-in for the reference's ``process_audio`` (one clip).

    Same positional/keyword arguments and defaults as dsp/pipeline.py:1113-1155 -- ``quantize_mode`` defaults to
    "autotune_v1" like the reference (config.py:44), the STFT path is ``quantize_mode="spectral_bins"`` or any spectral
    FX / freeze / formant / harmonic-lock option (:1315-1324).  Two extra keyword-only arguments: ``n_fft`` exposes the
    reference's module global N_FFT_DEFAULT (:149); ``precision`` ("auto" | "float32" | "float64") selects the
    arithmetic of the spectral pass (tables.choose_precision).  Returns ``(float32[n], taps)`` with taps
    ``input / pre_quant / post_dist / output`` (:1368, :1104-1109).
    """
    audio = preview_truncate(np.asarray(audio), sr, preview_enabled, pipeline_config)
    x = ensure_mono_float32(audio)  # :1312
    if x.ndim != 1:
        raise ValueError("stft_mono expects mono (1D) audio")  # dsp/stft_utils.py:47
    kw = dict(key=key, scale=scale, quantize_mode=quantize_mode, snap_strength=snap_strength, smear=smear,
              bin_smoothing=bin_smoothing, pre_quant=pre_quant, post_quant=post_quant,
              distortion_mode=distortion_mode, distortion_params=distortion_params, limiter_on=limiter_on,
              limiter_ceiling_db=limiter_ceiling_db, dry_wet=dry_wet, use_multiband=use_multiband,
              crossover_hz=crossover_hz, lowband_drive=lowband_drive, passthrough_test=passthrough_test,
              spectral_fx_mode=spectral_fx_mode, spectral_fx_strength=spectral_fx_strength,
              spectral_fx_params=spectral_fx_params, config=config, spectral_freeze=spectral_freeze,
              formant_shift=formant_shift, harmonic_lock_hz=harmonic_lock_hz, delta_listen=delta_listen,
              mono_strength=mono_strength, output_trim_db=output_trim_db, sub_cut_hz=sub_cut_hz,
              air_cut_hz=air_cut_hz, pipeline_config=pipeline_config, precision=precision,
              sub_enabled=sub_enabled, sub_source=sub_source, sub_note=sub_note, sub_scale_degree=sub_scale_degree,
              sub_octave=sub_octave, sub_level=sub_level, air_mix=air_mix)
    tap_input = x.copy()
    if x.shape[0] == 0:
        _resolve_kwargs(0, int(sr), int(n_fft), dict(kw))  # argument validation only
        e = np.zeros(0, dtype=np.float32)
        return e, {"input": tap_input, "pre_quant": e.copy(), "post_dist": e.copy(), "output": e.copy()}
    y, taps = process_batch(x[None, :], sr, n_fft=n_fft, return_taps=True, **kw)
    out = y[0]
    return out, {"input": tap_input, "pre_quant": taps["pre_quant"][0], "post_dist": taps["post_dist"][0],
                 "output": out.copy()}
