"""TEST INFRASTRUCTURE ONLY -- never imported by toast_b200.

The oracle's destriping problem on a flat WCS map: ``oracle.toast_oracle.build_problem`` with
PixelsWCS (``oracle.pixels_wcs``) in place of PixelsHealpix.  The pixels come from the oracle's own
detector quaternions; the submaps follow the PixelsWCS rule (``wcs_submaps``).  Everything after
the pointing -- pixel distribution, solver flags, covariance, rcond mask, Offset layout and
variance -- is ``assemble``, which restates the set-up stages of ``build_problem`` on given
pointing; tests/test_mapmaker_wcs_host_logic.py holds it to ``build_problem`` bit for bit on the
HEALPix pointing.
"""

import sys

import numpy as np

from oracle import pixels_wcs as OW
from oracle import toast_oracle as O


def wcs_submaps(wcs, submaps):
    """The PixelsWCS submap rule (pixels_wcs.py:384-389): ``submaps`` submaps of
    ceil(n_pix / submaps) pixels.  Returns (n_pix, n_submap, n_pix_submap)."""
    n_pix = int(wcs.shape[0]) * int(wcs.shape[1])
    nps = n_pix // submaps
    if nps * submaps < n_pix:
        nps += 1
    return n_pix, int(submaps), nps


def pixels_wcs_views(wcs, quats, shared_flags, shared_flag_mask, pixels, intervals, hits,
                     n_pix_submap):
    """PixelsWCS._exec (pixels_wcs.py:590-620) over the views of every detector: the pixels of
    ``oracle.pixels_wcs.pixels_wcs``; samples outside every view are left untouched, the
    hit-submap mask is ORed from the non-negative pixels."""
    n_samp = quats.shape[1]
    fl = shared_flags if (shared_flags is not None and shared_flags.shape[-1] == n_samp) else None
    for d in range(quats.shape[0]):
        for iv in intervals:
            a, b = int(iv["first"]), int(iv["last"])
            p, _, _ = OW.pixels_wcs(wcs, quats[d, a:b], None if fl is None else fl[a:b],
                                    shared_flag_mask)
            pixels[d, a:b] = p
            hits[p[p >= 0] // n_pix_submap] = 1


def expand_pointing(pb, K):
    """PointingDetectorSimple -> PixelsWCS -> StokesWeights (``O.expand_pointing`` with the WCS
    pixel step): ``pb.wcs`` is an ``oracle.pixels_wcs.Wcs``.  Returns (pixels, weights, hits)."""
    n_det, n_samp = pb.n_det, pb.n_samp
    idx = np.arange(n_det, dtype=np.int32)
    quats = np.zeros((n_det, n_samp, 4))
    K.pointing_detector(pb.focalplane, pb.boresight, idx, quats, pb.intervals,
                        pb.shared_flags, pb.shared_flag_mask, False)
    pixels = np.zeros((n_det, n_samp), dtype=np.int64)
    hits = np.zeros(pb.n_submap, dtype=np.uint8)
    pixels_wcs_views(pb.wcs, quats, pb.shared_flags, pb.shared_flag_mask, pixels, pb.intervals,
                     hits, pb.n_pix_submap)
    weights = np.zeros((n_det, n_samp, 3))
    K.stokes_weights_IQU(idx, quats, idx, weights, pb.hwp, pb.intervals, pb.epsilon, pb.gamma,
                         pb.cal, pb.IAU, False)
    return pixels, weights, hits


def _problem(obs, shared_flag_mask, det_flag_mask, IAU, hwp, use_flags):
    """The attributes build_problem sets before expanding the pointing."""
    pb = O.Problem()
    pb.n_det, pb.n_samp = obs["n_det"], obs["n_samp"]
    pb.focalplane, pb.boresight = obs["focalplane"], obs["boresight"]
    pb.intervals = obs["intervals"]
    pb.epsilon, pb.gamma, pb.cal = obs["epsilon"], obs["gamma"], obs["cal"]
    pb.IAU = IAU
    pb.hwp = hwp if hwp is not None else np.zeros(1)
    pb.shared_flags = obs["shared_flags"] if use_flags else np.zeros(1, dtype=np.uint8)
    pb.shared_flag_mask = shared_flag_mask
    pb.det_flag_mask = det_flag_mask
    pb.det_scale = np.ascontiguousarray(obs["detweight"])
    pb.step_length = obs["step_length"]
    return pb


def assemble(pb, obs, rcond_threshold=1.0e-3, use_flags=True):
    """The stages of ``O.build_problem`` after the pointing expansion, on ``pb.pixels`` /
    ``pb.weights`` / ``pb.hit_submaps`` (mapmaker_templates.py:632-990: pixel distribution,
    solver flags, CovarianceAndHits, rcond mask, Offset layout and variance)."""
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
    invcov = np.zeros(pb.n_local_submap * pb.n_pix_submap * 6)
    for d in range(pb.n_det):
        for iv in pb.intervals:
            a, b = int(iv["first"]), int(iv["last"])
            sm, lp = O.global_to_local(pb.pixels[d, a:b], pb.n_pix_submap, pb.global2local)
            lp[sf[d, a:b] != 0] = -1
            O.cov_accum_diag_invnpp(pb.n_local_submap, pb.n_pix_submap, 3, sm, lp,
                                    np.ascontiguousarray(pb.weights[d, a:b]).reshape(-1),
                                    float(pb.det_scale[d]), invcov)
    pb.invcov = invcov.copy()
    rcond = np.zeros(pb.n_local_submap * pb.n_pix_submap)
    O.cov_eigendecompose_diag(pb.n_local_submap, pb.n_pix_submap, 3, invcov, rcond,
                              rcond_threshold, True)
    pb.cov = invcov.reshape(pb.n_local_submap, pb.n_pix_submap, 6)
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


def build_wcs_problem(obs, K=None, wcs=None, submaps=1, shared_flag_mask=1, det_flag_mask=1,
                      rcond_threshold=1.0e-3, IAU=False, hwp=None, use_flags=True):
    """``O.build_problem`` on the flat map ``wcs`` (an ``oracle.pixels_wcs.Wcs`` with its shape
    set) cut into ``submaps`` submaps; ``pb.wcs`` is the projection, ``pb.nside`` / ``pb.nest``
    are None."""
    K = K or sys.modules[O.__name__]
    pb = _problem(obs, shared_flag_mask, det_flag_mask, IAU, hwp, use_flags)
    pb.wcs = wcs
    pb.nside = pb.nest = None
    _, pb.n_submap, pb.n_pix_submap = wcs_submaps(wcs, submaps)
    pb.pixels, pb.weights, pb.hit_submaps = expand_pointing(pb, K)
    return assemble(pb, obs, rcond_threshold, use_flags)


def build_healpix_problem(obs, K=None, rcond_threshold=1.0e-3):
    """``assemble`` on the HEALPix pointing of ``O.expand_pointing``: must be ``O.build_problem``
    bit for bit (the check that ``assemble`` restates it)."""
    from toast_b200.synthetic import n_submap_for

    K = K or sys.modules[O.__name__]
    pb = _problem(obs, 1, 1, False, None, True)
    pb.nside, pb.nest = obs["nside"], obs["nest"]
    pb.n_submap, pb.n_pix_submap = n_submap_for(pb.nside, obs["nside_submap"])
    pb.pixels, pb.weights, pb.hit_submaps = O.expand_pointing(pb, K)
    return assemble(pb, obs, rcond_threshold)
