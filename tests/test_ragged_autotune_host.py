"""CPU: the host side of ragged batches in quantize_mode="autotune_v1" -- the C ABI additions and the per-clip
short-clip rule."""
import os

import numpy as np
import pytest

from quantumdistortion_b200 import autotune

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_autotune_varlen_symbols_declared_and_bound():
    header = open(os.path.join(ROOT, "include", "qd_b200.h")).read()
    src = open(os.path.join(ROOT, "quantumdistortion_b200", "_lib.py")).read()
    for name in ("qd_autotune_workspace_bytes_varlen", "qd_autotune_render_device_varlen"):
        assert name + "(" in header, name
        assert f"lib.{name}.argtypes" in src, name
    assert "lib.qd_autotune_workspace_bytes_varlen.restype = C.c_size_t" in src


def test_autotune_varlen_workspace_bytes():
    """The ragged layout of a batch packed without gaps is never smaller than the uniform one of the same clips."""
    import ctypes as C
    from quantumdistortion_b200 import _lib
    lib = _lib.load()
    p = _params(48000)
    for b in (1, 3, 1024):
        uni = int(lib.qd_autotune_workspace_bytes(C.byref(p), b))
        rag = int(lib.qd_autotune_workspace_bytes_varlen(C.byref(p), b, b * p.n_samples))
        assert rag >= uni > 0
    assert int(lib.qd_autotune_workspace_bytes_varlen(C.byref(p), 0, 100)) == 0
    assert int(lib.qd_autotune_workspace_bytes_varlen(C.byref(p), 4, -1)) == 0


def _params(n, **kw):
    args = dict(sr=48000, n_samples=n, key="C", scale="major", snap_strength=1.0, pre_quant=True,
                distortion_mode=None, distortion_params=None, limiter_on=True, limiter_ceiling_db=-1.0, dry_wet=1.0,
                output_trim_db=0.0, delta_listen=False)
    args.update(kw)
    return autotune.resolve(**args)


def test_check_lengths_is_per_clip():
    p = _params(20000)
    autotune.check_lengths(p, [0, 16, 20000])
    for bad in ([5], [16, 1, 300], [15]):
        with pytest.raises(ValueError, match="padlen"):
            autotune.check_lengths(p, bad)
    autotune.check_lengths(_params(20000, snap_strength=0.0), [1, 5, 15])   # no zero-phase filters without the pitch stage
    with pytest.raises(ValueError, match="padlen"):
        _params(15)
    autotune.check_lengths(p, np.zeros(0, np.int64))
