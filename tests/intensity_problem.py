"""TEST INFRASTRUCTURE ONLY -- never imported by toast_b200.

The oracle's destriping problem with ``nnz`` Stokes values per pixel: 3 (I, Q, U: the problem of
``oracle.toast_oracle.build_problem``) or 1 (intensity only: ``StokesWeights(mode="I")``, whose
weights are ``cal[det]``, ``ops_stokes_weights.cpp:397-505``).  The pointing comes from the oracle's
own kernels, on HEALPix or on a flat WCS map (``tests/wcs_problem.py``); the set-up stages
(pixel distribution, solver flags, CovarianceAndHits, rcond mask, Offset layout and variance)
and the solver's map side are restated here with nnz in place of the oracle's fixed 3.  The oracle's
kernels take nnz = 1 as they are (``build_noise_weighted``, ``scan_map``, ``cov_accum_diag_*``,
``cov_eigendecompose_diag``, ``cov_apply_diag``).  tests/test_intensity_host_logic.py holds the
nnz = 3 form to ``build_problem`` / ``solver_lhs`` bit for bit.
"""

import sys

import numpy as np

import wcs_problem as WP
from oracle import toast_oracle as O


def expand_pointing(pb, K, nnz):
    """Pixels (HEALPix when ``pb.wcs`` is None, else PixelsWCS) and the weights of ``nnz``:
    StokesWeights(mode="IQU") [n_det, n_samp, 3] or (mode="I") [n_det, n_samp]."""
    if getattr(pb, "wcs", None) is None:
        pixels, weights, hits = O.expand_pointing(pb, K)
    else:
        pixels, weights, hits = WP.expand_pointing(pb, K)
    if nnz == 1:
        # (the oracle's: the I weight is cal[det] inside the views, whatever the kernel namespace)
        weights = np.zeros((pb.n_det, pb.n_samp))
        O.stokes_weights_I(np.arange(pb.n_det, dtype=np.int32), weights, pb.intervals, pb.cal,
                           False)
    return pixels, weights, hits


def assemble(pb, obs, nnz, rcond_threshold=1.0e-3, use_flags=True):
    """``wcs_problem.assemble`` (the stages of ``O.build_problem`` after the pointing) with
    ``nnz`` values per pixel: covariance [n_local, n_pix_submap, nnz (nnz + 1) / 2]."""
    ncov = nnz * (nnz + 1) // 2
    pb.local_submaps, pb.global2local = O.pixel_distribution(pb.hit_submaps)
    pb.n_local_submap = len(pb.local_submaps)
    in_view = np.zeros(pb.n_samp, dtype=bool)
    for iv in pb.intervals:
        in_view[iv["first"]:iv["last"]] = True
    sf = np.zeros((pb.n_det, pb.n_samp), dtype=np.uint8)
    if use_flags:
        sf |= ((obs["det_flags"] & pb.det_flag_mask) != 0).astype(np.uint8)
        sf |= ((obs["shared_flags"] & pb.shared_flag_mask) != 0).astype(np.uint8)[None, :]
    sf |= (~in_view).astype(np.uint8)[None, :]
    sf |= (pb.pixels < 0).astype(np.uint8)
    invcov = np.zeros(pb.n_local_submap * pb.n_pix_submap * ncov)
    for d in range(pb.n_det):
        for iv in pb.intervals:
            a, b = int(iv["first"]), int(iv["last"])
            sm, lp = O.global_to_local(pb.pixels[d, a:b], pb.n_pix_submap, pb.global2local)
            lp[sf[d, a:b] != 0] = -1
            O.cov_accum_diag_invnpp(pb.n_local_submap, pb.n_pix_submap, nnz, sm, lp,
                                    np.ascontiguousarray(pb.weights[d, a:b]).reshape(-1),
                                    float(pb.det_scale[d]), invcov)
    pb.invcov = invcov.copy()
    rcond = np.zeros(pb.n_local_submap * pb.n_pix_submap)
    O.cov_eigendecompose_diag(pb.n_local_submap, pb.n_pix_submap, nnz, invcov, rcond,
                              rcond_threshold, True)
    pb.cov = invcov.reshape(pb.n_local_submap, pb.n_pix_submap, ncov)
    pb.rcond = rcond
    badpix = (rcond.reshape(pb.n_local_submap, pb.n_pix_submap) == 0.0)
    for d in range(pb.n_det):
        sm, lp = O.global_to_local(pb.pixels[d], pb.n_pix_submap, pb.global2local)
        ok = sm >= 0
        bad = np.zeros(pb.n_samp, dtype=bool)
        bad[ok] = badpix[sm[ok], lp[ok]]
        sf[d, bad] |= 1
    pb.solver_flags = sf
    pb.shared_flag_mask_solver = 0
    pb.n_amp_views, pb.det_start, pb.n_amp = O.offset_layout(pb.n_det, pb.intervals,
                                                             pb.step_length)
    pb.offset_var, pb.amp_flags = O.offset_variance(
        pb.n_det, pb.n_samp, pb.intervals, pb.step_length, pb.n_amp_views, pb.det_scale,
        pb.solver_flags, pb.det_flag_mask)
    return pb


def build_problem(obs, K=None, nnz=1, wcs=None, submaps=1, rcond_threshold=1.0e-3):
    """The destriping problem of ``obs`` with ``nnz`` values per pixel, on HEALPix (``wcs`` None:
    the observation's nside / nest / nside_submap) or on the flat map ``wcs`` (an
    ``oracle.pixels_wcs.Wcs`` with its shape set) cut into ``submaps`` submaps.  ``pb.nnz`` is
    set; everything else has the attributes of ``O.build_problem``."""
    from toast_b200.synthetic import n_submap_for

    K = K or sys.modules[O.__name__]
    pb = WP._problem(obs, 1, 1, False, None, True)
    if wcs is None:
        pb.nside, pb.nest = obs["nside"], obs["nest"]
        pb.n_submap, pb.n_pix_submap = n_submap_for(pb.nside, obs["nside_submap"])
    else:
        pb.wcs = wcs
        pb.nside = pb.nest = None
        _, pb.n_submap, pb.n_pix_submap = WP.wcs_submaps(wcs, submaps)
    pb.pixels, pb.weights, pb.hit_submaps = expand_pointing(pb, K, nnz)
    assemble(pb, obs, nnz, rcond_threshold)
    pb.nnz = nnz
    return pb


def _nnz(pb):
    return getattr(pb, "nnz", 3)


def _weights3(pb):
    """The weights as [n_det, n_samp, nnz]: the layout every kernel namespace takes."""
    return pb.weights if pb.weights.ndim == 3 else pb.weights[:, :, None]


def bin_map(pb, K, det_data, covapply=None):
    """``O.bin_map`` (BuildNoiseWeighted + covariance_apply) on a map of ``pb.nnz`` values."""
    covapply = covapply or O.cov_apply_diag
    nnz = _nnz(pb)
    idx = np.arange(pb.n_det, dtype=np.int32)
    zmap = np.zeros((pb.n_local_submap, pb.n_pix_submap, nnz))
    K.build_noise_weighted(pb.global2local, zmap, idx, pb.pixels, idx, _weights3(pb), idx,
                           det_data, idx, pb.solver_flags, pb.det_scale, pb.det_flag_mask,
                           pb.intervals, pb.shared_flags, pb.shared_flag_mask, False)
    covapply(pb.n_local_submap, pb.n_pix_submap, nnz, pb.cov.reshape(-1), zmap.reshape(-1))
    return zmap


def _scan_weight_project(pb, K, binned, det_temp, out):
    idx = np.arange(pb.n_det, dtype=np.int32)
    O._scan(K)(pb.global2local, pb.n_pix_submap, binned, det_temp, idx, pb.pixels, idx,
               _weights3(pb), idx, pb.intervals, 1.0, False, True, False, False)
    K.noise_weight(det_temp, idx, pb.intervals, pb.det_scale, False)
    O.template_project(pb, K, det_temp, out)


def solver_lhs(pb, K, amps_in, covapply=None):
    """``O.solver_lhs`` (SolverLHS, mapmaker_solve.py:342-506) on a map of ``pb.nnz`` values."""
    det_temp = np.zeros((pb.n_det, pb.n_samp))
    O.template_add(pb, K, amps_in, det_temp)
    binned = bin_map(pb, K, det_temp, covapply)
    out = np.zeros_like(amps_in)
    det_temp[:] = 0
    O.template_add(pb, K, amps_in, det_temp)
    _scan_weight_project(pb, K, binned, det_temp, out)
    return out


def solver_rhs(pb, K, signal, covapply=None):
    """``O.solver_rhs`` (SolverRHS, mapmaker_solve.py:107-229) on a map of ``pb.nnz`` values."""
    binned = bin_map(pb, K, signal, covapply)
    det_temp = signal.copy()
    rhs = np.zeros(pb.n_amp)
    _scan_weight_project(pb, K, binned, det_temp, rhs)
    return rhs


def solve(pb, K, rhs, convergence=1.0e-12, n_iter_max=100, n_iter_min=3, covapply=None,
          trace=None):
    """``O.solve`` (the PCG of mapmaker_solve.py:524-755) with this module's LHS."""
    covapply = covapply or O.cov_apply_diag
    return O._solve(pb, K, rhs, convergence, n_iter_max, n_iter_min, covapply,
                    lambda pb_, K_, a, c=None: solver_lhs(pb_, K_, a, c), trace)


def lhs_loop(pb, amps):
    """The intensity-only LHS written out sample by sample in numpy (an independent statement of
    what ``solver_lhs`` computes for nnz = 1): F^T N^-1 (1 - P C P^T N^-1) F a."""
    assert _nnz(pb) == 1
    nps = pb.n_pix_submap
    z = np.zeros(pb.n_local_submap * nps)
    todf = np.zeros((pb.n_det, pb.n_samp))     # F a
    ampi = np.full((pb.n_det, pb.n_samp), -1, dtype=np.int64)
    for d in range(pb.n_det):
        off = int(pb.det_start[d])
        for v, iv in enumerate(pb.intervals):
            a, b = int(iv["first"]), int(iv["last"])
            k = off + np.arange(b - a) // pb.step_length
            ampi[d, a:b] = k
            good = pb.amp_flags[k] == 0
            todf[d, a:b] = np.where(good, amps[k], 0.0)
            off += int(pb.n_amp_views[v])
    lpix = np.full((pb.n_det, pb.n_samp), -1, dtype=np.int64)
    for d in range(pb.n_det):
        sm, lp = O.global_to_local(pb.pixels[d], nps, pb.global2local)
        ok = (sm >= 0) & (lp >= 0)
        lpix[d, ok] = sm[ok] * nps + lp[ok]
    use = (ampi >= 0) & (pb.solver_flags & pb.det_flag_mask == 0) & (lpix >= 0)
    for d in range(pb.n_det):
        for s in np.flatnonzero(use[d]):
            z[lpix[d, s]] += todf[d, s] * pb.weights[d, s] * pb.det_scale[d]
    m = z * pb.cov.reshape(-1)
    out = np.zeros(pb.n_amp)
    for d in range(pb.n_det):
        for s in np.flatnonzero(use[d]):
            k = ampi[d, s]
            if pb.amp_flags[k] == 0:
                out[k] += (todf[d, s] - pb.weights[d, s] * m[lpix[d, s]]) * pb.det_scale[d]
    return out
