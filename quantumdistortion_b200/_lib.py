"""ctypes binding of libqd_b200.so (include/qd_b200.h).  Fails loudly: there is no CPU path."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "csrc", "libqd_b200.so")

QD_ABI_VERSION = 6
QD_FX = {"none": 0, "bitcrush_log": 1, "bitcrush_uniform": 2, "phase_dispersal": 3,
         "scramble_pick": 4, "scramble_swap": 5}


class QdParams(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("sample_rate", C.c_int32), ("n_fft", C.c_int32), ("n_samples", C.c_int32),
        ("passthrough", C.c_int32), ("pre_quant", C.c_int32), ("post_quant", C.c_int32), ("bin_smoothing", C.c_int32),
        ("distortion_mode", C.c_int32), ("tube_gain", C.c_float), ("tube_norm", C.c_float),
        ("limiter_on", C.c_int32), ("lookahead", C.c_int32), ("fold_amount", C.c_double), ("bias", C.c_double),
        ("ceiling_lin", C.c_double), ("release_coeff", C.c_double),
        ("wet", C.c_float), ("dry", C.c_float), ("trim_gain", C.c_float), ("apply_trim", C.c_int32),
        ("delta_listen", C.c_int32),
        ("multiband", C.c_int32), ("low_delay", C.c_int32), ("sos_low", (C.c_double * 6) * 2),
        ("sos_high", (C.c_double * 6) * 2), ("low_gain", C.c_float), ("low_norm", C.c_double),
        ("low_trim_gain", C.c_float), ("apply_low_trim", C.c_int32), ("mono_a", C.c_float), ("mono_b", C.c_float),
        ("apply_mono_blend", C.c_int32),
        ("fx_mode", C.c_int32), ("fx_a", C.c_double), ("fx_b", C.c_double), ("fx_c", C.c_double),
        ("fx_table_frames", C.c_int32), ("fx_table_per_clip", C.c_int32),
        ("precision", C.c_int32), ("spectral_freeze", C.c_int32),
        ("formant_ratio", C.c_double), ("formant_order", C.c_int32), ("no_spectral", C.c_int32),
    ]


class QdTables(C.Structure):
    _fields_ = [
        ("n_bins", C.c_int32), ("target_bins", C.POINTER(C.c_int32)), ("active_mask", C.POINTER(C.c_uint8)),
        ("snap", C.c_double), ("smear", C.c_double), ("smear_radius", C.c_int32), ("smear_w", C.POINTER(C.c_double)),
    ]


class QdTaps(C.Structure):
    _fields_ = [("pre_quant", C.c_void_p), ("post_dist", C.c_void_p)]


_lib = None


class QdError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the CUDA library; build it first if nvcc is present and it is missing or stale."""
    global _lib
    if _lib is not None:
        return _lib
    from . import build as _build
    override = os.environ.get("QD_B200_LIB")   # A/B runs of two builds on one box (profiles/): no rebuild, no fallback
    if override:
        path = override
    elif _build.needs_build():
        try:
            _build.build()
        except Exception as exc:  # noqa: BLE001
            if not os.path.exists(LIB_PATH):
                raise QdError(f"libqd_b200.so is missing and could not be built ({exc}); "
                              "quantumdistortion_b200 has no CPU fallback") from exc
    if not override:
        path = LIB_PATH
    lib = C.CDLL(path)
    vp, i64, i32, dbl, flt = C.c_void_p, C.c_int64, C.c_int32, C.c_double, C.c_float
    lib.qd_abi_version.restype = C.c_int
    lib.qd_last_error.restype = C.c_char_p
    lib.qd_device_count.restype = C.c_int
    lib.qd_plan_create.argtypes = [C.POINTER(QdParams), C.POINTER(QdTables), C.POINTER(vp)]
    lib.qd_plan_destroy.argtypes = [vp]
    lib.qd_plan_destroy.restype = None
    lib.qd_plan_workspace_bytes.argtypes = [vp, i64]
    lib.qd_plan_workspace_bytes.restype = C.c_size_t
    lib.qd_plan_launches_per_render.argtypes = [vp]
    lib.qd_plan_enable_timing.argtypes = [vp, C.c_int]
    lib.qd_plan_read_timing.argtypes = [vp, C.POINTER(C.c_double * 4), C.POINTER(C.c_int64 * 4)]
    lib.qd_plan_set_fx_table.argtypes = [vp, vp, i64]
    lib.qd_render_device.argtypes = [vp, vp, vp, i64, C.POINTER(QdTaps), vp, C.c_size_t, vp]
    lib.qd_render_host.argtypes = [vp, vp, vp, i64, i64]
    lib.qd_render_host_pcm16.argtypes = [vp, vp, vp, i64, i64]
    lib.qd_render_host_ex.argtypes = [vp, vp, vp, i64, i64, i32, i32]
    lib.qd_plan_workspace_bytes_varlen.argtypes = [vp, i64, i64]
    lib.qd_plan_workspace_bytes_varlen.restype = C.c_size_t
    lib.qd_render_device_varlen.argtypes = [vp, vp, vp, vp, vp, i64, i64, i32, C.POINTER(QdTaps), vp, C.c_size_t, vp]
    lib.qd_render_host_varlen.argtypes = [vp, vp, vp, vp, vp, i64, i64, i32, i32]
    lib.qd_limiter_device.argtypes = [vp, vp, i64, i64, i32, dbl, dbl, vp]
    lib.qd_crossover_device.argtypes = [vp, vp, vp, i64, i64, C.POINTER((dbl * 6) * 2), C.POINTER((dbl * 6) * 2), vp]
    lib.qd_distort_device.argtypes = [vp, vp, i64, i32, dbl, dbl, flt, flt, vp]
    lib.qd_spectral_peaks_device.argtypes = [vp, i64, i32, i32, i32, dbl, i32, vp, vp]
    lib.qd_autotune_workspace_bytes.argtypes = [vp, i64]
    lib.qd_autotune_workspace_bytes.restype = C.c_size_t
    lib.qd_autotune_render_device.argtypes = [vp, vp, vp, i64, vp, vp, vp, C.c_size_t, vp]
    lib.qd_autotune_workspace_bytes_varlen.argtypes = [vp, i64, i64]
    lib.qd_autotune_workspace_bytes_varlen.restype = C.c_size_t
    lib.qd_autotune_render_device_varlen.argtypes = [vp, vp, vp, vp, vp, i64, i64, i32, C.POINTER(QdTaps), vp,
                                                     C.c_size_t, vp]
    lib.qd_measure_fp32_peak.argtypes = [C.POINTER(C.c_double), vp]
    lib.qd_host_alloc.argtypes = [C.c_size_t]
    lib.qd_host_alloc.restype = vp
    lib.qd_host_free.argtypes = [vp]
    lib.qd_host_free.restype = None
    if lib.qd_abi_version() != QD_ABI_VERSION:
        raise QdError("libqd_b200.so ABI version mismatch; rebuild with python -m quantumdistortion_b200.build --force")
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().qd_last_error()
        raise QdError(f"libqd_b200 error {rc}: {msg.decode() if msg else '?'}")
