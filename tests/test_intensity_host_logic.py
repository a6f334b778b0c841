"""Intensity-only destriping (StokesWeights(mode="I")) in the CPU suite.

* tests/intensity_problem.py restates the oracle's problem with nnz values per pixel: its nnz = 3
  form must be ``O.build_problem`` / ``O.solver_lhs`` bit for bit, and its I-only LHS must be
  the RHS of the template timestream (LHS(a) == RHS(F a), as the reference's own test has it,
  tests/ops_mapmaker_solve.py:150-265) and agree with a sample-by-sample numpy loop.
* ``ops.MapMaker`` with mode "I" runs its host logic through the CPU stand-ins of
  tests/fake_device_intensity.py and must give that problem's products bit for bit, with one
  value per pixel.  On the GPU, tests/test_gpu_intensity.py runs the real kernels."""

import numpy as np
import pytest

import fake_device_intensity as FI
import intensity_problem as IP
from helpers import O, S, assert_close_norm
from oracle import pixels_wcs as OW
from test_mapmaker_wcs_host_logic import FOV, _WcsFakeDeviceObservation
from toast_b200 import ops
from toast_b200.data import Data, observation_from_synthetic
from toast_b200.templates import Offset


def _car(obs, res=0.5):
    """A CAR map around the scan of ``obs`` (the oracle's create_wcs)."""
    from toast_b200.ops.pixels_wcs import scan_range_lonlat_deg

    b = scan_range_lonlat_deg(obs["boresight"], obs["shared_flags"], 1, FOV, False)
    wo, shape = OW.create_wcs("CAR", bounds_deg=tuple(float(x) for x in b), res_deg=(res, res))
    wo.shape = tuple(shape)
    return wo


def _amps(pb, seed=3):
    rng = np.random.default_rng(seed)
    a = rng.normal(size=pb.n_amp)
    a[pb.amp_flags != 0] = 0.0
    return a


@pytest.mark.parametrize("name,n_det,n_samp,nside", [("c1", 4, 6000, 16), ("c2", 6, 12000, 64)])
def test_nnz3_problem_is_build_problem(name, n_det, n_samp, nside):
    obs = S.make_observation(name, n_det=n_det, n_samp=n_samp, nside=nside, eps_max=0.03)
    ref = O.build_problem(obs, O, rcond_threshold=1.0e-3)
    got = IP.build_problem(obs, O, nnz=3, rcond_threshold=1.0e-3)
    assert set(ref.__dict__) | {"nnz"} == set(got.__dict__)
    for key, value in ref.__dict__.items():
        if isinstance(value, np.ndarray):
            np.testing.assert_array_equal(getattr(got, key), value, err_msg=key)
        else:
            assert getattr(got, key) == value, key
    a = _amps(ref)
    np.testing.assert_array_equal(IP.solver_lhs(got, O, a), O.solver_lhs(ref, O, a))
    np.testing.assert_array_equal(IP.solver_rhs(got, O, obs["signal"]),
                                  O.solver_rhs(ref, O, obs["signal"]))


@pytest.mark.parametrize("pixelisation", ["healpix", "car"])
def test_intensity_lhs_is_the_rhs_of_the_template_timestream(pixelisation):
    obs = S.make_observation("c2", n_det=6, n_samp=12000, nside=64, eps_max=0.03)
    wcs = _car(obs) if pixelisation == "car" else None
    pb = IP.build_problem(obs, O, nnz=1, wcs=wcs, submaps=8)
    assert pb.weights.shape == (pb.n_det, pb.n_samp) and pb.cov.shape[-1] == 1
    in_view = pb.solver_flags == 0
    np.testing.assert_array_equal(pb.weights[in_view],
                                  np.broadcast_to(pb.cal[:, None], pb.weights.shape)[in_view])
    np.testing.assert_array_equal(pb.rcond, 1.0)   # nnz 1: the reference's rcond
    a = _amps(pb)
    fa = np.zeros((pb.n_det, pb.n_samp))
    O.template_add(pb, O, a, fa)
    lhs = IP.solver_lhs(pb, O, a)
    np.testing.assert_array_equal(lhs, IP.solver_rhs(pb, O, fa))
    assert np.abs(lhs).max() > 0
    assert_close_norm(IP.lhs_loop(pb, a), lhs, rtol=1e-12, what="numpy loop")


def _mapper(pix, obs, mode):
    dp = pix.detector_pointing
    wts = ops.StokesWeights(detector_pointing=dp, mode=mode)
    binning = ops.BinMap(pixel_dist="pixel_dist", covariance="cov", pixel_pointing=pix,
                         stokes_weights=wts, noise_model="noise_model", full_pointing=True)
    tmpl = Offset(name="baselines", step_time=obs["step_time"], times="times",
                  noise_model="noise_model")
    tmat = ops.TemplateMatrix(templates=[tmpl], amplitudes="amplitudes")
    mapper = ops.MapMaker(name="mm", det_data="signal", binning=binning, template_matrix=tmat,
                          solve_rcond_threshold=1.0e-3, map_rcond_threshold=1.0e-3, iter_max=8,
                          convergence=1.0e-30, device="cpu")
    return mapper, tmpl


class _WcsIntensityObservation(FI.IntensityMixin, _WcsFakeDeviceObservation):
    pass


@pytest.mark.parametrize("pixelisation", ["healpix", "car"])
def test_mapmaker_intensity_host_logic_with_oracle_compute(monkeypatch, pixelisation):
    FI.install_intensity(monkeypatch, _WcsIntensityObservation)
    n_det = 6
    obs = S.make_observation("c2", n_det=n_det, n_samp=12000, nside=64, eps_max=0.03)
    data = Data()
    data.obs.append(observation_from_synthetic(obs))
    dp = ops.PointingDetectorSimple(view="scanning", shared_flags="flags", shared_flag_mask=1)
    if pixelisation == "healpix":
        pix = ops.PixelsHealpix(detector_pointing=dp, nside=obs["nside"], nest=obs["nest"],
                                create_dist="pixel_dist")
    else:
        pix = ops.PixelsWCS(detector_pointing=dp, create_dist="pixel_dist", projection="CAR",
                            field_of_view=FOV, resolution=(0.5, 0.5), submaps=8)
    mapper, tmpl = _mapper(pix, obs, "I")
    signal0 = obs["signal"].copy()
    mapper.apply(data)
    if pixelisation == "healpix":
        pb = IP.build_problem(obs, O, nnz=1)
    else:
        wo, shape = OW.create_wcs("CAR", bounds_deg=pix.bounds, res_deg=(0.5, 0.5))
        wo.shape = tuple(shape)
        pb = IP.build_problem(obs, O, nnz=1, wcs=wo, submaps=8)

    dist = data["pixel_dist"]
    np.testing.assert_array_equal(dist.global_submap_to_local, pb.global2local)
    hits_ref = np.zeros(pb.n_local_submap * pb.n_pix_submap, dtype=np.int64)
    sf0 = ((obs["det_flags"] & 1) != 0) | ((obs["shared_flags"] & 1) != 0)[None, :]
    for d in range(n_det):
        for iv in pb.intervals:
            a, b = int(iv["first"]), int(iv["last"])
            sm, lp = O.global_to_local(pb.pixels[d, a:b], pb.n_pix_submap, pb.global2local)
            lp[sf0[d, a:b]] = -1
            O.cov_accum_diag_hits(pb.n_local_submap, pb.n_pix_submap, 1, sm, lp, hits_ref)
    assert hits_ref.sum() > 0
    np.testing.assert_array_equal(data["mm_hits"].raw, hits_ref)
    for key, n_value in (("mm_cov", 1), ("mm_binmap", 1), ("mm_map", 1), ("mm_rcond", 1)):
        assert data[key].n_value == n_value, key
    np.testing.assert_array_equal(data["mm_cov"].data, pb.cov)
    np.testing.assert_array_equal(data["mm_rcond"].raw, pb.rcond)

    np.testing.assert_array_equal(tmpl._amp_flags, pb.amp_flags != 0)
    np.testing.assert_array_equal(tmpl._offsetvar, pb.offset_var)

    covapply = O.cov_apply_diag
    np.testing.assert_array_equal(data["mm_binmap"].data, IP.bin_map(pb, O, signal0, covapply))
    rhs_ref = IP.solver_rhs(pb, O, signal0, covapply)
    amps_ref, hist_ref = IP.solve(pb, O, rhs_ref, convergence=1e-30, n_iter_max=8,
                                  covapply=covapply)
    assert mapper.history == hist_ref
    amps = data["amplitudes"]["baselines"].local
    np.testing.assert_array_equal(amps, amps_ref)
    clean = signal0.copy()
    O.template_add(pb, O, -amps, clean)
    np.testing.assert_array_equal(data.obs[0].detdata["signal"].data, clean)
    assert_close_norm(data["mm_map"].data, IP.bin_map(pb, O, clean, covapply), rtol=1e-15,
                      what="destriped map")


def test_mapmaker_still_refuses_other_modes(monkeypatch):
    FI.install_intensity(monkeypatch)
    obs = S.make_observation("c1", n_det=2, n_samp=2000, nside=16, eps_max=0.03)
    data = Data()
    data.obs.append(observation_from_synthetic(obs))
    dp = ops.PointingDetectorSimple(view="scanning", shared_flags="flags", shared_flag_mask=1)
    pix = ops.PixelsHealpix(detector_pointing=dp, nside=obs["nside"], nest=obs["nest"],
                            create_dist="pixel_dist")
    mapper, _ = _mapper(pix, obs, "IQU")
    mapper.binning.stokes_weights.mode = "QU"
    with pytest.raises(NotImplementedError, match="mode"):
        mapper.apply(data)
