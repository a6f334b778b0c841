"""ctypes binding of libtoastb200.so (include/toast_b200.h).

This is the thin Python view of the C ABI used by the host-side operator mirror
(``toast_b200.ops``), the tests and ``bench.py``.  There is no CPU fallback: if the library
is missing ``load()`` raises, and every compute entry point raises ``RuntimeError`` when no
CUDA device is usable.
"""

import ctypes as ct
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TB_LIB_PATH", os.path.join(HERE, "libtoastb200.so"))

TB_MEM_HOST, TB_MEM_DEVICE, TB_MEM_TABLE = 0, 1, 2
TB_ERR_NO_DEVICE, TB_ERR_ARG = 2, 3

interval_dtype = np.dtype(
    {
        "names": ["start", "stop", "first", "last"],
        "formats": ["d", "d", "q", "q"],
        "offsets": [0, 8, 16, 24],
    }
)

P = ct.c_void_p
I64 = ct.c_int64
I32 = ct.c_int32
U8 = ct.c_uint8
F64 = ct.c_double
INT = ct.c_int
SZ = ct.c_size_t
STR = ct.c_char_p


class tb_obs_desc(ct.Structure):
    _fields_ = [
        ("n_det", I64), ("n_samp", I64), ("n_view", I64),
        ("intervals", P), ("focalplane", P),
        ("epsilon", P), ("gamma", P), ("cal", P),
        ("det_scale", P), ("amp_offsets", P), ("n_amp_views", P),
        ("step_length", I64),
        ("nside", I64), ("n_pix_submap", I64), ("n_submap", I64),
        ("nest", INT), ("IAU", INT),
        ("global2local", P),
        ("boresight", P), ("shared_flags", P), ("shared_flag_mask", U8),
        ("solver_flags", P), ("solver_flag_mask", U8),
        ("pixels", P), ("weights", P), ("hwp", P),
    ]


class tb_wcs_desc(ct.Structure):
    _fields_ = [
        ("projection", INT), ("is_azimuth", INT),
        ("euler", F64 * 5), ("crpix", F64 * 2), ("cdelt", F64 * 2), ("cea_lambda", F64),
        ("n_col", I64), ("n_row", I64),
    ]


class tb_offset_prior_desc(ct.Structure):
    _fields_ = [
        ("n_amp", I64), ("n_seg", I64),
        ("seg_start", P), ("seg_len", P), ("filt_start", P), ("filt_len", P),
        ("filters", P), ("n_filter_values", I64),
        ("precond_mode", INT),
        ("prec_start", P), ("prec_width", P), ("precond", P), ("n_precond_values", I64),
    ]


TB_PRECOND_TOEPLITZ, TB_PRECOND_BANDED = 1, 2

# name -> (restype, argtypes); every symbol declared in include/toast_b200.h
PROTOTYPES = {
    "tb_last_error": (STR, []),
    "tb_version": (STR, []),
    "tb_accel_enabled": (INT, []),
    "tb_accel_assign_device": (INT, [INT, INT, F64, INT]),
    "tb_accel_get_device": (INT, []),
    "tb_device_synchronize": (INT, []),
    "tb_launch_count": (I64, []),
    "tb_accel_present": (INT, [P, SZ]),
    "tb_accel_create": (INT, [P, SZ, STR]),
    "tb_accel_update_device": (INT, [P, SZ, STR]),
    "tb_accel_update_host": (INT, [P, SZ, STR]),
    "tb_accel_reset": (INT, [P, SZ, STR]),
    "tb_accel_delete": (INT, [P, SZ, STR]),
    "tb_accel_device_ptr": (P, [P]),
    "tb_accel_dump": (None, []),
    "tb_accel_bytes_in_use": (SZ, []),
    "tb_pointing_detector": (INT, [P, P, P, P, I64, P, I64, P, U8, I64, I64, INT, P]),
    "tb_pixels_healpix": (INT, [P, P, I64, P, U8, P, P, I64, P, I64, P, I64, I64, I64, INT,
                                I64, I64, INT, P]),
    "tb_pixels_wcs": (INT, [ct.POINTER(tb_wcs_desc), P, P, I64, P, U8, P, P, I64, P, I64, P, I64,
                            I64, I64, I64, INT, P]),
    "tb_stokes_weights_IQU": (INT, [P, P, I64, P, P, I64, P, P, I64, P, P, P, INT, I64, I64,
                                    INT, P]),
    "tb_stokes_weights_I": (INT, [P, P, I64, P, I64, P, I64, I64, INT, P]),
    "tb_pointing_fused": (INT, [P, P, P, U8, P, P, I64, P, P, I64, P, P, I64, P, P, I64, P, I64,
                                I64, I64, INT, P, P, P, INT, I64, I64, INT, P]),
    "tb_pointing_fused_wcs": (INT, [P, P, P, U8, P, P, I64, P, P, I64, P, P, I64, P, P, I64, P,
                                    I64, I64, ct.POINTER(tb_wcs_desc), P, P, P, INT, I64, I64,
                                    INT, P]),
    "tb_noise_weight": (INT, [P, I64, P, P, I64, P, I64, I64, INT, P]),
    "tb_build_noise_weighted": (INT, [P, I64, P, I64, I64, I64, P, P, I64, P, P, I64, P, P, I64,
                                      P, P, I64, P, U8, P, I64, P, U8, I64, I64, INT, P]),
    "tb_scan_map": (INT, [P, I64, I64, P, INT, I64, I64, P, I64, P, P, I64, P, P, I64, P, P,
                          I64, F64, INT, INT, INT, I64, I64, INT, P]),
    "tb_template_offset_add_to_signal": (INT, [I64, I64, P, P, P, I64, I32, P, I64, P, I64, I64,
                                               INT, P]),
    "tb_template_offset_project_signal": (INT, [I32, P, I64, I32, P, I64, U8, I64, I64, P, P, P,
                                                I64, P, I64, I64, INT, P]),
    "tb_template_offset_apply_diag_precond": (INT, [P, P, P, P, I64, INT, P]),
    "tb_template_offset_add_to_signal_batch": (INT, [I64, P, P, P, P, I64, P, P, I64, P, I64,
                                                     I64, I64, INT, P]),
    "tb_template_offset_project_signal_batch": (INT, [P, P, I64, P, P, I64, U8, I64, P, P, P, P,
                                                      I64, P, I64, I64, I64, INT, P]),
    "tb_cov_apply_diag": (INT, [I64, I64, I64, P, P, INT, P]),
    "tb_cov_accum": (INT, [P, I64, I64, I64, I64, P, P, P, P, I64, P, P, I64, P, P, I64, P, U8,
                           P, I64, P, U8, I64, I64, INT, P]),
    "tb_cov_invert": (INT, [I64, I64, P, P, F64, INT, P]),
    "tb_obs_create": (P, [ct.POINTER(tb_obs_desc)]),
    "tb_obs_create_wcs": (P, [ct.POINTER(tb_obs_desc), ct.POINTER(tb_wcs_desc)]),
    "tb_obs_create_intensity": (P, [ct.POINTER(tb_obs_desc), ct.POINTER(tb_wcs_desc)]),
    "tb_obs_nnz": (INT, [P]),
    "tb_obs_destroy": (None, [P]),
    "tb_lhs_pass1": (INT, [P, P, P, P, INT, P]),
    "tb_lhs_pass2": (INT, [P, P, P, P, P, INT, P]),
    "tb_obs_sorted_passes": (INT, [P]),
    "tb_obs_set_pixel_chunks": (INT, [P, I64, P]),
    "tb_bx_block_pixels": (INT, []),
    "tb_obs_blocked": (INT, [P]),
    "tb_obs_blocked_stats": (INT, [P, P, P, P, P]),
    "tb_bx_pass1": (INT, [P, P, P, P, INT, I64, P]),
    "tb_bx_pass2": (INT, [P, P, P, I64, P]),
    "tb_bx_fused": (INT, [P, P, P, P, P, P, P]),
    "tb_bx_direction_prescale": (INT, [P, P, P, P, P, P, P, I64, P]),
    "tb_rhs_project": (INT, [P, P, P, P, P, INT, P]),
    "tb_bin_signal": (INT, [P, P, P, INT, P]),
    "tb_offset_prior_create": (P, [ct.POINTER(tb_offset_prior_desc)]),
    "tb_offset_prior_destroy": (None, [P]),
    "tb_offset_prior_add": (INT, [P, P, P, P, INT, P]),
    "tb_offset_prior_precond": (INT, [P, P, P, P, INT, P]),
    "tb_peer_create": (P, [INT, INT, SZ]),
    "tb_peer_get_handles": (INT, [P, P]),
    "tb_peer_open": (INT, [P, P]),
    "tb_peer_map_ptr": (P, [P]),
    "tb_map_reduce_cov": (INT, [P, I64, P, P]),
    "tb_map_reduce_cov_range": (INT, [P, I64, I64, P, P]),
    "tb_peer_destroy": (None, [P]),
    "tb_peer_attach": (P, [INT, INT, SZ, P, P, ct.c_uint64]),
    "tb_peer_has_multicast": (INT, [P]),
    "tb_peer_set_multimem": (INT, [INT]),
    "tb_amp_dot": (INT, [P, P, P, I64, P, P]),
    "tb_pcg_update": (INT, [P, P, P, P, P, P, P, P, P, I64, P, P]),
    "tb_pcg_direction": (INT, [P, P, P, P, I64, P]),
    "tb_obs_pack_pointing": (INT, [P, P]),
    "tb_obs_has_compact_pointing": (INT, [P]),
    "tb_obs_has_pair_weights": (INT, [P]),
    "tb_obs_crossing_stats": (INT, [P, P, P, P]),
    "tb_set_option": (INT, [STR, INT]),
    "tb_get_option": (INT, [STR]),
    "tb_set_pixel_guard_scale": (None, [F64]),
    "tb_pixel_exact_count": (I64, [INT]),
}

_lib = None


def load():
    """Load libtoastb200.so and attach prototypes.  Raises if the library is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m toast_b200.build` "
            "(there is no CPU fallback for the toast_b200 kernels)"
        )
    lib = ct.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    # TB_OPTIONS="blocked=0,crossings=0": kernel-variant switches for A/B measurements
    for item in os.environ.get("TB_OPTIONS", "").split(","):
        if "=" in item:
            k, v = item.split("=", 1)
            if lib.tb_set_option(k.strip().encode(), int(v)) != 0:
                raise RuntimeError(f"TB_OPTIONS: unknown option {k!r}")
    return lib


def check(rc):
    """Translate a C-ABI status into the RuntimeError the reference bindings raise."""
    if rc != 0:
        msg = load().tb_last_error()
        raise RuntimeError(msg.decode() if msg else f"toast_b200 error {rc}")


def last_error():
    msg = load().tb_last_error()
    return msg.decode() if msg else ""


def accel_enabled():
    return bool(load().tb_accel_enabled())


def _is_tensor(a):
    return hasattr(a, "data_ptr") and hasattr(a, "is_cuda")


def ptr(a):
    """Raw pointer of a numpy array / torch tensor / None."""
    if a is None:
        return None
    if _is_tensor(a):
        if not a.is_contiguous():
            raise RuntimeError("tensor must be contiguous")
        return a.data_ptr()
    if not a.flags["C_CONTIGUOUS"]:
        raise RuntimeError("array must be C-contiguous")
    return a.ctypes.data


def mem_of(a, use_accel):
    """Memory mode implied by a LARGE array argument."""
    if _is_tensor(a):
        if not a.is_cuda:
            raise RuntimeError("large tensor arguments must be CUDA tensors")
        return TB_MEM_DEVICE
    return TB_MEM_TABLE if use_accel else TB_MEM_HOST


def host(a, dtype):
    """Small per-detector arrays are always host numpy arrays of the exact dtype."""
    if a is None:
        return None
    if _is_tensor(a):
        a = a.detach().cpu().numpy()
    a = np.ascontiguousarray(a, dtype=dtype)
    return a
