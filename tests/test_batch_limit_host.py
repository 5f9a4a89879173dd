"""CPU: the uniform device entry points index clips with int, like the ragged ones, and reject a batch of 2^31 clips or
more with QD_ERR_INVALID_ARG before they read a buffer or touch the device.  (qd_render_device needs a plan, which
needs the device: its check is covered on the B200, tests/test_gpu_launch_split.py.)"""
import ctypes as C

import numpy as np

from quantumdistortion_b200 import _lib, autotune

QD_ERR_INVALID_ARG = -1
BATCH = 2 ** 31


def _ptr(a):
    return C.c_void_p(a.ctypes.data)


def test_uniform_entry_points_reject_batches_past_int32():
    lib = _lib.load()
    buf = np.zeros(64, np.float32)    # host memory: never read, the argument check comes first
    bins = np.zeros(64, np.int16)
    sos = ((C.c_double * 6) * 2)()
    p = autotune.resolve(sr=48000, n_samples=4096, key="C", scale="major", snap_strength=1.0, pre_quant=True,
                         distortion_mode=None, distortion_params=None, limiter_on=True, limiter_ceiling_db=-1.0,
                         dry_wet=1.0, output_trim_db=0.0, delta_listen=False)
    calls = {
        "qd_autotune_render_device": lambda b: lib.qd_autotune_render_device(
            C.byref(p), _ptr(buf), _ptr(buf), b, None, None, _ptr(buf), buf.nbytes, None),
        "qd_limiter_device": lambda b: lib.qd_limiter_device(_ptr(buf), _ptr(buf), b, 16, 4, 0.9, 0.999, None),
        "qd_crossover_device": lambda b: lib.qd_crossover_device(_ptr(buf), _ptr(buf), _ptr(buf), b, 16,
                                                                 C.byref(sos), C.byref(sos), None),
        "qd_spectral_peaks_device": lambda b: lib.qd_spectral_peaks_device(_ptr(buf), b, 16, 2048, 4, 1e-4, 0,
                                                                           _ptr(bins), None),
    }
    for name, call in calls.items():
        assert call(BATCH) == QD_ERR_INVALID_ARG, name
        assert b"2^31" in lib.qd_last_error(), name
        assert call(0) == 0, name   # an empty batch is still fine
