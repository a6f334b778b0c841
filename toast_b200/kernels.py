"""Kernel functions with the names and positional signatures of the reference's
``toast._libtoast`` hot-path functions (SURVEY.md section 8b), dispatching to the CUDA library
through its C ABI.

Large arrays may be numpy arrays (``use_accel=False``: staged per call, host in / host out;
``use_accel=True``: looked up in the device table created with ``accel_create``) or torch CUDA
tensors (used in place).  Small per-detector arrays are host numpy arrays.  Optional arrays
follow the reference's shape convention (length != n_samp means "absent").

Every function raises ``RuntimeError`` on failure like the reference bindings
(``common.hpp:50-122``).  There is no CPU implementation behind these names.
"""

import numpy as np

from . import lib as L

interval_dtype = L.interval_dtype


def _shape(a):
    return tuple(a.shape)


def _dtype_name(a):
    if L._is_tensor(a):
        return str(a.dtype).replace("torch.", "")
    return a.dtype.name


def _require(a, name, dtype, ndim):
    """extract_buffer<T> equivalent (common.hpp:33-125): dtype, ndim, contiguity."""
    if a is None:
        raise RuntimeError(f"Object {name} is None")
    if len(_shape(a)) != ndim:
        raise RuntimeError(f"Object {name} has {len(_shape(a))} dimensions instead of {ndim}")
    if _dtype_name(a) != dtype:
        raise RuntimeError(f"Object {name} has dtype {_dtype_name(a)}, expected {dtype}")
    if L._is_tensor(a):
        if not a.is_contiguous():
            raise RuntimeError(f"Object {name} is not contiguous")
    elif not a.flags["C_CONTIGUOUS"]:
        raise RuntimeError(f"Object {name} is not contiguous")
    return a


def _intervals(iv):
    if L._is_tensor(iv):
        raise RuntimeError("intervals must be a host array with the Interval dtype")
    iv = np.ascontiguousarray(iv)
    if iv.dtype.itemsize != 32:
        raise RuntimeError("Object intervals does not have the Interval dtype")
    return iv


def _optional(a, n_samp):
    """Reference convention: an optional per-sample array is absent if its length != n_samp."""
    if a is None:
        return None
    if _shape(a)[-1] != n_samp:
        return None
    return a


def _stream(stream):
    return None if stream is None else int(stream)


def pointing_detector(focalplane, boresight, quat_index, quats, intervals, shared_flags,
                      shared_flag_mask, use_accel=False, stream=None):
    """ops_pointing_detector.cpp:78-227."""
    quat_index = L.host(quat_index, np.int32)
    n_det = len(quat_index)
    focalplane = L.host(focalplane, np.float64)
    if focalplane.shape != (n_det, 4):
        raise RuntimeError("Object focalplane has wrong shape")
    _require(boresight, "boresight", "float64", 2)
    n_samp = _shape(boresight)[0]
    _require(quats, "quats", "float64", 3)
    if _shape(quats)[1:] != (n_samp, 4):
        raise RuntimeError("Object quats has wrong shape")
    iv = _intervals(intervals)
    fl = _optional(shared_flags, n_samp)
    L.check(L.load().tb_pointing_detector(
        L.ptr(focalplane), L.ptr(boresight), L.ptr(quat_index), L.ptr(quats), _shape(quats)[0],
        L.ptr(iv), len(iv), L.ptr(fl), shared_flag_mask, n_det, n_samp,
        L.mem_of(quats, use_accel), _stream(stream)))


def pixels_healpix(quat_index, quats, shared_flags, shared_flag_mask, pixel_index, pixels,
                   intervals, hit_submaps, n_pix_submap, nside, nest, use_accel=False,
                   stream=None):
    """ops_pixels_healpix.cpp:1153-1417."""
    quat_index = L.host(quat_index, np.int32)
    pixel_index = L.host(pixel_index, np.int32)
    n_det = len(quat_index)
    if len(pixel_index) != n_det:
        raise RuntimeError("Object pixel_index has wrong shape")
    _require(pixels, "pixels", "int64", 2)
    n_samp = _shape(pixels)[1]
    _require(quats, "quats", "float64", 3)
    if _shape(quats)[1:] != (n_samp, 4):
        raise RuntimeError("Object quats has wrong shape")
    if L._is_tensor(hit_submaps) or hit_submaps.dtype != np.uint8:
        raise RuntimeError("Object hit_submaps must be a host uint8 array")
    iv = _intervals(intervals)
    fl = _optional(shared_flags, n_samp)
    L.check(L.load().tb_pixels_healpix(
        L.ptr(quat_index), L.ptr(quats), _shape(quats)[0], L.ptr(fl), shared_flag_mask,
        L.ptr(pixel_index), L.ptr(pixels), _shape(pixels)[0], L.ptr(iv), len(iv),
        L.ptr(hit_submaps), len(hit_submaps), n_pix_submap, nside, 1 if nest else 0, n_det,
        n_samp, L.mem_of(pixels, use_accel), _stream(stream)))


def pixels_wcs(wcs, quat_index, quats, shared_flags, shared_flag_mask, pixel_index, pixels,
               intervals, hit_submaps, n_pix_submap, use_accel=False, stream=None):
    """ops/pixels_wcs.py:560-620 for all detectors of an observation in one launch.  ``wcs`` is
    a ``toast_b200.wcs.FlatWCS`` (or anything with a ``.desc()`` returning a tb_wcs_desc)."""
    quat_index = L.host(quat_index, np.int32)
    pixel_index = L.host(pixel_index, np.int32)
    n_det = len(quat_index)
    if len(pixel_index) != n_det:
        raise RuntimeError("Object pixel_index has wrong shape")
    _require(pixels, "pixels", "int64", 2)
    n_samp = _shape(pixels)[1]
    _require(quats, "quats", "float64", 3)
    if _shape(quats)[1:] != (n_samp, 4):
        raise RuntimeError("Object quats has wrong shape")
    if hit_submaps is not None and (L._is_tensor(hit_submaps) or hit_submaps.dtype != np.uint8):
        raise RuntimeError("Object hit_submaps must be a host uint8 array")
    iv = _intervals(intervals)
    fl = _optional(shared_flags, n_samp)
    d = wcs.desc()
    import ctypes as ct

    L.check(L.load().tb_pixels_wcs(
        ct.byref(d), L.ptr(quat_index), L.ptr(quats), _shape(quats)[0], L.ptr(fl),
        shared_flag_mask, L.ptr(pixel_index), L.ptr(pixels), _shape(pixels)[0], L.ptr(iv), len(iv),
        L.ptr(hit_submaps), 0 if hit_submaps is None else len(hit_submaps), n_pix_submap, n_det,
        n_samp, L.mem_of(pixels, use_accel), _stream(stream)))


def stokes_weights_IQU(quat_index, quats, weight_index, weights, hwp, intervals, epsilon, gamma,
                       cal, IAU, use_accel=False, stream=None):
    """ops_stokes_weights.cpp:150-392."""
    quat_index = L.host(quat_index, np.int32)
    weight_index = L.host(weight_index, np.int32)
    n_det = len(quat_index)
    _require(weights, "weights", "float64", 3)
    if _shape(weights)[2] != 3:
        raise RuntimeError("Object weights has wrong shape")
    n_samp = _shape(weights)[1]
    _require(quats, "quats", "float64", 3)
    if _shape(quats)[1:] != (n_samp, 4):
        raise RuntimeError("Object quats has wrong shape")
    iv = _intervals(intervals)
    h = _optional(hwp, n_samp)
    eps = L.host(epsilon, np.float64)
    gam = L.host(gamma, np.float64)
    c = L.host(cal, np.float64)
    for a, nm in ((eps, "epsilon"), (gam, "gamma"), (c, "cal"), (weight_index, "weight_index")):
        if len(a) != n_det:
            raise RuntimeError(f"Object {nm} has wrong shape")
    L.check(L.load().tb_stokes_weights_IQU(
        L.ptr(quat_index), L.ptr(quats), _shape(quats)[0], L.ptr(weight_index), L.ptr(weights),
        _shape(weights)[0], L.ptr(h), L.ptr(iv), len(iv), L.ptr(eps), L.ptr(gam), L.ptr(c),
        1 if IAU else 0, n_det, n_samp, L.mem_of(weights, use_accel), _stream(stream)))


def stokes_weights_I(weight_index, weights, intervals, cal, use_accel=False, stream=None):
    """ops_stokes_weights.cpp:397-505."""
    weight_index = L.host(weight_index, np.int32)
    n_det = len(weight_index)
    _require(weights, "weights", "float64", 2)
    n_samp = _shape(weights)[1]
    iv = _intervals(intervals)
    c = L.host(cal, np.float64)
    L.check(L.load().tb_stokes_weights_I(
        L.ptr(weight_index), L.ptr(weights), _shape(weights)[0], L.ptr(iv), len(iv), L.ptr(c),
        n_det, n_samp, L.mem_of(weights, use_accel), _stream(stream)))


def pointing_fused(focalplane, boresight, shared_flags, shared_flag_mask, quat_index, quats,
                   pixel_index, pixels, weight_index, weights, hwp, intervals, hit_submaps,
                   n_pix_submap, nside, nest, epsilon, gamma, cal, IAU, use_accel=False,
                   stream=None):
    """Fused a1+a2+a3 (not in the reference): any of quats / pixels / weights may be None."""
    _require(boresight, "boresight", "float64", 2)
    n_samp = _shape(boresight)[0]
    focalplane = L.host(focalplane, np.float64)
    n_det = focalplane.shape[0]
    iv = _intervals(intervals)
    fl = _optional(shared_flags, n_samp)
    h = _optional(hwp, n_samp)
    qi = L.host(quat_index, np.int32) if quats is not None else None
    pi = L.host(pixel_index, np.int32) if pixels is not None else None
    wi = L.host(weight_index, np.int32) if weights is not None else None
    eps = L.host(epsilon, np.float64)
    gam = L.host(gamma, np.float64)
    c = L.host(cal, np.float64)
    big = pixels if pixels is not None else (weights if weights is not None else quats)
    L.check(L.load().tb_pointing_fused(
        L.ptr(focalplane), L.ptr(boresight), L.ptr(fl), shared_flag_mask,
        L.ptr(qi), L.ptr(quats), _shape(quats)[0] if quats is not None else 0,
        L.ptr(pi), L.ptr(pixels), _shape(pixels)[0] if pixels is not None else 0,
        L.ptr(wi), L.ptr(weights), _shape(weights)[0] if weights is not None else 0,
        L.ptr(h), L.ptr(iv), len(iv), L.ptr(hit_submaps),
        len(hit_submaps) if hit_submaps is not None else 0, n_pix_submap, nside,
        1 if nest else 0, L.ptr(eps), L.ptr(gam), L.ptr(c), 1 if IAU else 0, n_det, n_samp,
        L.mem_of(big, use_accel), _stream(stream)))


def pointing_fused_wcs(wcs, focalplane, boresight, shared_flags, shared_flag_mask, quat_index,
                       quats, pixel_index, pixels, weight_index, weights, hwp, intervals,
                       hit_submaps, n_pix_submap, epsilon, gamma, cal, IAU, use_accel=False,
                       stream=None):
    """``pointing_fused`` onto a flat projection: ``wcs`` is a ``toast_b200.wcs.FlatWCS`` (or
    anything with a ``.desc()`` returning a tb_wcs_desc), as for ``pixels_wcs``."""
    import ctypes as ct

    _require(boresight, "boresight", "float64", 2)
    n_samp = _shape(boresight)[0]
    focalplane = L.host(focalplane, np.float64)
    n_det = focalplane.shape[0]
    iv = _intervals(intervals)
    fl = _optional(shared_flags, n_samp)
    h = _optional(hwp, n_samp)
    qi = L.host(quat_index, np.int32) if quats is not None else None
    pi = L.host(pixel_index, np.int32) if pixels is not None else None
    wi = L.host(weight_index, np.int32) if weights is not None else None
    eps = L.host(epsilon, np.float64)
    gam = L.host(gamma, np.float64)
    c = L.host(cal, np.float64)
    if hit_submaps is not None and (L._is_tensor(hit_submaps) or hit_submaps.dtype != np.uint8):
        raise RuntimeError("Object hit_submaps must be a host uint8 array")
    d = wcs.desc()
    big = pixels if pixels is not None else (weights if weights is not None else quats)
    L.check(L.load().tb_pointing_fused_wcs(
        L.ptr(focalplane), L.ptr(boresight), L.ptr(fl), shared_flag_mask,
        L.ptr(qi), L.ptr(quats), _shape(quats)[0] if quats is not None else 0,
        L.ptr(pi), L.ptr(pixels), _shape(pixels)[0] if pixels is not None else 0,
        L.ptr(wi), L.ptr(weights), _shape(weights)[0] if weights is not None else 0,
        L.ptr(h), L.ptr(iv), len(iv), L.ptr(hit_submaps),
        len(hit_submaps) if hit_submaps is not None else 0, n_pix_submap, ct.byref(d),
        L.ptr(eps), L.ptr(gam), L.ptr(c), 1 if IAU else 0, n_det, n_samp,
        L.mem_of(big, use_accel), _stream(stream)))


def noise_weight(det_data, data_index, intervals, detector_weights, use_accel=False,
                 stream=None):
    """ops_noise_weight.cpp:12-118."""
    data_index = L.host(data_index, np.int32)
    n_det = len(data_index)
    _require(det_data, "det_data", "float64", 2)
    n_samp = _shape(det_data)[1]
    iv = _intervals(intervals)
    w = L.host(detector_weights, np.float64)
    if len(w) != n_det:
        raise RuntimeError("Object detector_weights has wrong shape")
    L.check(L.load().tb_noise_weight(
        L.ptr(det_data), _shape(det_data)[0], L.ptr(data_index), L.ptr(iv), len(iv), L.ptr(w),
        n_det, n_samp, L.mem_of(det_data, use_accel), _stream(stream)))


def build_noise_weighted(global2local, zmap, pixel_index, pixels, weight_index, weights,
                         data_index, det_data, flag_index, det_flags, det_scale, det_flag_mask,
                         intervals, shared_flags, shared_flag_mask, use_accel=False,
                         stream=None):
    """ops_mapmaker_utils.cpp:93-380."""
    pixel_index = L.host(pixel_index, np.int32)
    n_det = len(pixel_index)
    _require(pixels, "pixels", "int64", 2)
    n_samp = _shape(pixels)[1]
    weight_index = L.host(weight_index, np.int32)
    data_index = L.host(data_index, np.int32)
    nd_w = len(_shape(weights))
    if nd_w == 2:
        nnz = 1
        _require(weights, "weights", "float64", 2)
    else:
        _require(weights, "weights", "float64", 3)
        nnz = _shape(weights)[2]
    if _shape(weights)[1] != n_samp:
        raise RuntimeError("Object weights has wrong shape")
    _require(det_data, "det_data", "float64", 2)
    if _shape(det_data)[1] != n_samp:
        raise RuntimeError("Object det_data has wrong shape")
    _require(zmap, "zmap", "float64", 3)
    if _shape(zmap)[2] != nnz:
        raise RuntimeError("Object zmap has wrong shape")
    g2l = L.host(global2local, np.int64)
    scale = L.host(det_scale, np.float64)
    if len(scale) != n_det or len(weight_index) != n_det or len(data_index) != n_det:
        raise RuntimeError("per-detector arrays have inconsistent shapes")
    iv = _intervals(intervals)
    df = det_flags if (det_flags is not None and len(_shape(det_flags)) == 2
                       and _shape(det_flags)[1] == n_samp) else None
    # SURVEY 8b (vii): with det_flags=None the operator passes flag_index=[-1]
    fi = L.host(flag_index, np.int32) if df is not None else None
    if df is not None:
        _require(df, "det_flags", "uint8", 2)
        if len(fi) != n_det:
            raise RuntimeError("Object flag_index has wrong shape")
    sf = _optional(shared_flags, n_samp)
    L.check(L.load().tb_build_noise_weighted(
        L.ptr(g2l), len(g2l), L.ptr(zmap), _shape(zmap)[0], _shape(zmap)[1], nnz,
        L.ptr(pixel_index), L.ptr(pixels), _shape(pixels)[0], L.ptr(weight_index),
        L.ptr(weights), _shape(weights)[0], L.ptr(data_index), L.ptr(det_data),
        _shape(det_data)[0], L.ptr(fi), L.ptr(df), _shape(df)[0] if df is not None else 0,
        L.ptr(scale), det_flag_mask, L.ptr(iv), len(iv), L.ptr(sf), shared_flag_mask, n_det,
        n_samp, L.mem_of(zmap, use_accel), _stream(stream)))


_MAP_DTYPES = {"float64": 0, "float32": 1, "int64": 2, "int32": 3}


def _scan_map(expect):
    def fn(global2local, n_pix_submap, mapdata, det_data, data_index, pixels, pixel_index,
           weights, weight_index, intervals, data_scale, should_zero, should_subtract,
           should_scale, use_accel=False, stream=None):
        """ops_scan_map.cpp:85-292."""
        _require(mapdata, "mapdata", expect, 3)
        nnz = _shape(mapdata)[2]
        data_index = L.host(data_index, np.int32)
        pixel_index = L.host(pixel_index, np.int32)
        weight_index = L.host(weight_index, np.int32)
        n_det = len(data_index)
        _require(pixels, "pixels", "int64", 2)
        n_samp = _shape(pixels)[1]
        _require(det_data, "det_data", "float64", 2)
        if len(_shape(weights)) == 2:
            if nnz != 1:
                raise RuntimeError("Object weights has wrong shape")
        elif _shape(weights)[2] != nnz:
            raise RuntimeError("Object weights has wrong shape")
        if _dtype_name(weights) != "float64":
            raise RuntimeError("Object weights has wrong dtype")
        g2l = L.host(global2local, np.int64)
        iv = _intervals(intervals)
        L.check(L.load().tb_scan_map(
            L.ptr(g2l), len(g2l), n_pix_submap, L.ptr(mapdata), _MAP_DTYPES[expect],
            _shape(mapdata)[0], nnz, L.ptr(det_data), _shape(det_data)[0], L.ptr(data_index),
            L.ptr(pixels), _shape(pixels)[0], L.ptr(pixel_index), L.ptr(weights),
            _shape(weights)[0], L.ptr(weight_index), L.ptr(iv), len(iv), float(data_scale),
            int(bool(should_zero)), int(bool(should_subtract)), int(bool(should_scale)), n_det,
            n_samp, L.mem_of(det_data, use_accel), _stream(stream)))

    fn.__name__ = f"ops_scan_map_{expect}"
    return fn


ops_scan_map_float64 = _scan_map("float64")
ops_scan_map_float32 = _scan_map("float32")
ops_scan_map_int64 = _scan_map("int64")
ops_scan_map_int32 = _scan_map("int32")


def scan_map(global2local, n_pix_submap, mapdata, *args, **kw):
    """Dtype dispatch like ops/scan_map/kernels.py:90-144."""
    return globals()[f"ops_scan_map_{_dtype_name(mapdata)}"](global2local, n_pix_submap, mapdata,
                                                              *args, **kw)


def template_offset_add_to_signal(step_length, amp_offset, n_amp_views, amplitudes,
                                  amplitude_flags, data_index, det_data, intervals,
                                  use_accel=False, stream=None):
    """template_offset.cpp:16-146."""
    _require(amplitudes, "amplitudes", "float64", 1)
    _require(amplitude_flags, "amplitude_flags", "uint8", 1)
    _require(det_data, "det_data", "float64", 2)
    iv = _intervals(intervals)
    nav = L.host(n_amp_views, np.int64)
    if len(nav) != len(iv):
        raise RuntimeError("Object n_amp_views has wrong shape")
    L.check(L.load().tb_template_offset_add_to_signal(
        int(step_length), int(amp_offset), L.ptr(nav), L.ptr(amplitudes), L.ptr(amplitude_flags),
        _shape(amplitudes)[0], int(data_index), L.ptr(det_data), _shape(det_data)[0], L.ptr(iv),
        len(iv), _shape(det_data)[1], L.mem_of(det_data, use_accel), _stream(stream)))


def template_offset_project_signal(data_index, det_data, flag_index, flag_data, flag_mask,
                                   step_length, amp_offset, n_amp_views, amplitudes,
                                   amplitude_flags, intervals, use_accel=False, stream=None):
    """template_offset.cpp:149-331."""
    _require(amplitudes, "amplitudes", "float64", 1)
    _require(amplitude_flags, "amplitude_flags", "uint8", 1)
    _require(det_data, "det_data", "float64", 2)
    n_samp = _shape(det_data)[1]
    iv = _intervals(intervals)
    nav = L.host(n_amp_views, np.int64)
    if len(nav) != len(iv):
        raise RuntimeError("Object n_amp_views has wrong shape")
    fd = None
    if flag_index >= 0 and flag_data is not None and len(_shape(flag_data)) == 2 \
            and _shape(flag_data)[1] == n_samp:
        fd = _require(flag_data, "flag_data", "uint8", 2)
    L.check(L.load().tb_template_offset_project_signal(
        int(data_index), L.ptr(det_data), _shape(det_data)[0], int(flag_index), L.ptr(fd),
        _shape(fd)[0] if fd is not None else 0, flag_mask, int(step_length), int(amp_offset),
        L.ptr(nav), L.ptr(amplitudes), L.ptr(amplitude_flags), _shape(amplitudes)[0], L.ptr(iv),
        len(iv), n_samp, L.mem_of(det_data, use_accel), _stream(stream)))


def template_offset_apply_diag_precond(offset_var, amplitudes_in, amplitude_flags,
                                       amplitudes_out, use_accel=False, stream=None):
    """template_offset.cpp:334-405."""
    _require(amplitudes_in, "amplitudes_in", "float64", 1)
    n = _shape(amplitudes_in)[0]
    for a, nm, dt in ((offset_var, "offset_var", "float64"),
                      (amplitude_flags, "amplitude_flags", "uint8"),
                      (amplitudes_out, "amplitudes_out", "float64")):
        _require(a, nm, dt, 1)
        if _shape(a)[0] != n:
            raise RuntimeError(f"Object {nm} has wrong shape")
    L.check(L.load().tb_template_offset_apply_diag_precond(
        L.ptr(offset_var), L.ptr(amplitudes_in), L.ptr(amplitude_flags), L.ptr(amplitudes_out),
        n, L.mem_of(amplitudes_in, use_accel), _stream(stream)))


def template_offset_add_to_signal_batch(step_length, amp_offsets, n_amp_views, amplitudes,
                                        amplitude_flags, data_index, det_data, intervals,
                                        use_accel=False, stream=None):
    iv = _intervals(intervals)
    nav = L.host(n_amp_views, np.int64)
    ao = L.host(amp_offsets, np.int64)
    di = L.host(data_index, np.int32)
    L.check(L.load().tb_template_offset_add_to_signal_batch(
        int(step_length), L.ptr(ao), L.ptr(nav), L.ptr(amplitudes), L.ptr(amplitude_flags),
        _shape(amplitudes)[0], L.ptr(di), L.ptr(det_data), _shape(det_data)[0], L.ptr(iv),
        len(iv), len(di), _shape(det_data)[1], L.mem_of(det_data, use_accel), _stream(stream)))


def template_offset_project_signal_batch(data_index, det_data, flag_index, flag_data, flag_mask,
                                         step_length, amp_offsets, n_amp_views, amplitudes,
                                         amplitude_flags, intervals, use_accel=False,
                                         stream=None):
    iv = _intervals(intervals)
    nav = L.host(n_amp_views, np.int64)
    ao = L.host(amp_offsets, np.int64)
    di = L.host(data_index, np.int32)
    n_samp = _shape(det_data)[1]
    fd = flag_data if (flag_data is not None and len(_shape(flag_data)) == 2
                       and _shape(flag_data)[1] == n_samp) else None
    fi = L.host(flag_index, np.int32) if fd is not None else None
    L.check(L.load().tb_template_offset_project_signal_batch(
        L.ptr(di), L.ptr(det_data), _shape(det_data)[0], L.ptr(fi), L.ptr(fd),
        _shape(fd)[0] if fd is not None else 0, flag_mask, int(step_length), L.ptr(ao),
        L.ptr(nav), L.ptr(amplitudes), L.ptr(amplitude_flags), _shape(amplitudes)[0], L.ptr(iv),
        len(iv), len(di), n_samp, L.mem_of(det_data, use_accel), _stream(stream)))


def cov_apply_diag(nsub, subsize, nnz, mat, vec, use_accel=False, stream=None):
    """map_cov.cpp:372-423 -> toast_map_cov.cpp:471-528."""
    L.check(L.load().tb_cov_apply_diag(int(nsub), int(subsize), int(nnz), L.ptr(mat), L.ptr(vec),
                                       L.mem_of(vec, use_accel), _stream(stream)))


def cov_accum(global2local, n_local_submap, n_pix_submap, nnz, hits, invcov, pixel_index, pixels,
              weight_index, weights, flag_index, det_flags, det_scale, det_flag_mask, intervals,
              shared_flags, shared_flag_mask, use_accel=False, stream=None):
    """BuildHitMap + BuildInverseCovariance accumulation in one pass."""
    g2l = L.host(global2local, np.int64)
    pi = L.host(pixel_index, np.int32)
    n_det = len(pi)
    n_samp = _shape(pixels)[1]
    wi = L.host(weight_index, np.int32) if invcov is not None else None
    sc = L.host(det_scale, np.float64) if invcov is not None else None
    df = det_flags if (det_flags is not None and len(_shape(det_flags)) == 2
                       and _shape(det_flags)[1] == n_samp) else None
    fi = L.host(flag_index, np.int32) if df is not None else None
    sf = _optional(shared_flags, n_samp)
    iv = _intervals(intervals)
    L.check(L.load().tb_cov_accum(
        L.ptr(g2l), len(g2l), int(n_local_submap), int(n_pix_submap), int(nnz), L.ptr(hits),
        L.ptr(invcov), L.ptr(pi), L.ptr(pixels), _shape(pixels)[0], L.ptr(wi), L.ptr(weights),
        _shape(weights)[0] if weights is not None else 0, L.ptr(fi), L.ptr(df),
        _shape(df)[0] if df is not None else 0, L.ptr(sc), det_flag_mask, L.ptr(iv), len(iv),
        L.ptr(sf), shared_flag_mask, n_det, n_samp, L.mem_of(pixels, use_accel), _stream(stream)))


def cov_invert(npix, nnz, cov, rcond, threshold, use_accel=False, stream=None):
    """cov_eigendecompose_diag(invert=True): toast_map_cov.cpp:246-396."""
    L.check(L.load().tb_cov_invert(int(npix), int(nnz), L.ptr(cov), L.ptr(rcond),
                                   float(threshold), L.mem_of(cov, use_accel), _stream(stream)))


# ---- device memory table (accelerator.cpp:768-1110) ----------------------------------------

def accel_enabled():
    return L.accel_enabled()


def accel_assign_device(node_procs, node_rank, mem_gb, disabled):
    L.check(L.load().tb_accel_assign_device(node_procs, node_rank, float(mem_gb),
                                            1 if disabled else 0))


def accel_get_device():
    return L.load().tb_accel_get_device()


def _nbytes(buf):
    return buf.nbytes


def accel_present(buf, name="unknown"):
    return bool(L.load().tb_accel_present(L.ptr(buf), _nbytes(buf)))


def accel_create(buf, name="unknown"):
    L.check(L.load().tb_accel_create(L.ptr(buf), _nbytes(buf), name.encode()))


def accel_update_device(buf, name="unknown"):
    L.check(L.load().tb_accel_update_device(L.ptr(buf), _nbytes(buf), name.encode()))


def accel_update_host(buf, name="unknown"):
    L.check(L.load().tb_accel_update_host(L.ptr(buf), _nbytes(buf), name.encode()))


def accel_reset(buf, name="unknown"):
    L.check(L.load().tb_accel_reset(L.ptr(buf), _nbytes(buf), name.encode()))


def accel_delete(buf, name="unknown"):
    L.check(L.load().tb_accel_delete(L.ptr(buf), _nbytes(buf), name.encode()))


def accel_dump():
    L.load().tb_accel_dump()
