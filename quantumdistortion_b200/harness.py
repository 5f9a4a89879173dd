"""File-to-file front end (reference: quantum_distortion/dsp/harness.py:24-63), plus a batched variant that
renders many files, of any lengths, in one GPU call."""
from __future__ import annotations

from dataclasses import asdict
from pathlib import Path
from typing import Any, Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np

from .audio_io import load_audio, load_pcm16, save_audio, save_pcm16
from .config import PipelineConfig, ensure_mono_float32


def _config(preset: Optional[str], extra_params: Optional[Dict[str, Any]]) -> PipelineConfig:
    cfg = PipelineConfig.from_preset(preset) if preset is not None else PipelineConfig()
    if extra_params is not None:  # dsp/harness.py:56-60: unknown keys are ignored
        known = asdict(cfg)
        for k, v in extra_params.items():
            if k in known:
                setattr(cfg, k, v)
    return cfg


def process_file_to_file(infile: Path, outfile: Path, preset: Optional[str] = None,
                         extra_params: Optional[Dict[str, Any]] = None) -> None:
    """dsp/harness.py:24-63 (PipelineConfig defaults to quantize_mode="autotune_v1" like the reference's)."""
    from .pipeline import process_audio
    infile, outfile = Path(infile), Path(outfile)
    if not infile.exists():
        raise FileNotFoundError(f"Input file not found: {infile}")
    audio, sr = load_audio(infile)
    x = ensure_mono_float32(audio)
    cfg = _config(preset, extra_params)
    processed, _taps = process_audio(x, sr=sr, pipeline_config=cfg)
    save_audio(outfile, processed, sr)


def process_files(pairs: Iterable[Tuple[Path, Path]], preset: Optional[str] = None,
                  extra_params: Optional[Dict[str, Any]] = None, seeds=None) -> int:
    """Render many (infile, outfile) pairs with one parameter set -- the same files ``process_file_to_file`` would
    write one by one.  Files sharing (sample rate, 16-bit PCM mono or not) are rendered as one ragged batch
    (`process_batch` on a list of clips), whatever their lengths.  ``seeds`` (random spectral FX): None, one int for every file, or one seed per file in the order of ``pairs``.
    Returns the number of files written."""
    from .pipeline import preview_truncate, process_batch
    cfg = _config(preset, extra_params)
    pairs = list(pairs)
    per_file = seeds is not None and not isinstance(seeds, (int, np.integer))
    if per_file and len(seeds) != len(pairs):
        raise ValueError("need one seed per file")
    # (sample rate, is 16-bit PCM mono) -> [(outfile, samples, seed)]
    groups: Dict[Tuple[int, bool], List[Tuple[Path, np.ndarray, Any]]] = {}
    for i, (infile, outfile) in enumerate(pairs):
        infile = Path(infile)
        if not infile.exists():
            raise FileNotFoundError(f"Input file not found: {infile}")
        pcm, sr = load_pcm16(infile)
        if pcm is not None and pcm.ndim == 1:
            # mono 16-bit PCM stays int16 until it is on the device: same samples as load_audio's int16 / 32768
            x = preview_truncate(pcm, sr, None, cfg)
        else:
            audio, sr = load_audio(infile)
            x = ensure_mono_float32(preview_truncate(audio, sr, None, cfg))   # process_audio truncates before the mono mix
        groups.setdefault((sr, x.dtype == np.int16), []).append((Path(outfile), x, seeds[i] if per_file else None))
    written = 0
    for (sr, is_pcm), items in groups.items():
        live = [it for it in items if it[1].shape[0] > 0]
        ys, _ = process_batch([x for _, x, _ in live], sr, pipeline_config=cfg,
                              seeds=[s for _, _, s in live] if per_file else seeds) if live else ([], None)
        rendered = {id(it): y for it, y in zip(live, ys)}
        for it in items:
            out, x, _ = it
            if x.shape[0] == 0:
                save_audio(out, x.astype(np.float32), sr)
            elif is_pcm:
                save_pcm16(out, rendered[id(it)], sr)    # the device already applied save_audio's float -> PCM16 rule
            else:
                save_audio(out, rendered[id(it)], sr)
            written += 1
    return written
