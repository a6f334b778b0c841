"""ops.MapMaker with ops.PixelsWCS: the operator's HOST LOGIC in the CPU suite, against the stand-ins
of tests/fake_device.py (the oracle does the per-sample compute) and the oracle's WCS problem
(tests/wcs_problem.py).  The same assertions as the HEALPix test in
tests/test_mapmaker_host_logic.py; on the GPU, tests/test_gpu_wcs.py runs the real kernels."""

import numpy as np
import pytest

import fake_device
import wcs_problem as WP
from helpers import O, S, assert_close_norm
from oracle import pixels_wcs as OW
from toast_b200 import ops
from toast_b200.data import Data, observation_from_synthetic
from toast_b200.ops.pixels_wcs import _unwrap_together, scan_range_lonlat_deg
from toast_b200.templates import Offset

FOV = 11.0   # degrees: the synthetic focalplane is 10 degrees wide


def _oracle_wcs(flat):
    """The oracle's projection with the numbers of a product FlatWCS (shape and CRPIX as set)."""
    w = OW.Wcs(flat.proj, flat.crval, flat.cdelt, flat.is_azimuth)
    w.crpix = np.array(flat.crpix, dtype=np.float64)
    w.shape = tuple(flat.shape)
    return w


class _WcsFakeDeviceObservation(fake_device.FakeDeviceObservation):
    """FakeDeviceObservation that also takes ``wcs=`` (DeviceObservation's WCS form): the pointing
    expansion is then the oracle's PixelsWCS restatement."""

    def __init__(self, *, wcs=None, nside=None, nest=None, **kw):
        super().__init__(nside=0 if nside is None else nside, nest=bool(nest), **kw)
        self.wcs = wcs

    def expand_pointing(self, hit_submaps=None):
        if self.wcs is None:
            return super().expand_pointing(hit_submaps)
        pb = O.Problem(n_det=self.n_det, n_samp=self.n_samp, wcs=_oracle_wcs(self.wcs),
                       n_submap=self.n_submap, n_pix_submap=self.n_pix_submap,
                       focalplane=self.focalplane, boresight=self.boresight,
                       intervals=self.intervals, epsilon=self.epsilon, gamma=self.gamma,
                       cal=self.cal, IAU=self.IAU,
                       hwp=np.zeros(1) if self.hwp is None else np.asarray(self.hwp),
                       shared_flags=np.zeros(1, dtype=np.uint8) if self.shared_flags is None
                       else self.shared_flags, shared_flag_mask=self.shared_flag_mask)
        import torch

        pixels, weights, hits = WP.expand_pointing(pb, O)
        self.pixels, self.weights = torch.from_numpy(pixels), torch.from_numpy(weights)
        if hit_submaps is not None:
            hit_submaps |= hits


def _install(monkeypatch):
    import toast_b200.solver as SV

    fake_device.install(monkeypatch)
    monkeypatch.setattr(SV, "DeviceObservation", _WcsFakeDeviceObservation)


def _mapper(pix, obs, iter_max=8, **kw):
    dp = pix.detector_pointing
    wts = ops.StokesWeights(detector_pointing=dp, mode="IQU")
    binning = ops.BinMap(pixel_dist="pixel_dist", covariance="cov", pixel_pointing=pix,
                         stokes_weights=wts, noise_model="noise_model", full_pointing=True)
    tmpl = Offset(name="baselines", step_time=obs["step_time"], times="times",
                  noise_model="noise_model")
    tmat = ops.TemplateMatrix(templates=[tmpl], amplitudes="amplitudes")
    mapper = ops.MapMaker(name="mm", det_data="signal", binning=binning, template_matrix=tmat,
                          solve_rcond_threshold=1.0e-6, map_rcond_threshold=1.0e-6,
                          iter_max=iter_max, convergence=1.0e-30, device="cpu", **kw)
    return mapper, tmpl


# CAR sized from the scan (auto bounds); TAN on a fixed image smaller than the scan, so that
# samples fall off every side (negative pixels, and the reference's wrap into the previous row)
CASES = {
    "CAR-auto": dict(projection="CAR", field_of_view=FOV, resolution=(0.5, 0.5), submaps=8),
    "TAN-fixed": dict(projection="TAN", auto_bounds=False, center=(40.0, -30.0),
                      resolution=(0.4, 0.4), dimensions=(40, 24), submaps=7),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_mapmaker_wcs_host_logic_with_oracle_compute(monkeypatch, case):
    _install(monkeypatch)
    n_det = 8
    obs = S.make_observation("c2", n_det=n_det, n_samp=12000, eps_max=0.03)
    data = Data()
    data.obs.append(observation_from_synthetic(obs))
    dp = ops.PointingDetectorSimple(view="scanning", shared_flags="flags", shared_flag_mask=1)
    pix = ops.PixelsWCS(detector_pointing=dp, create_dist="pixel_dist", **CASES[case])
    mapper, tmpl = _mapper(pix, obs)
    signal0 = obs["signal"].copy()
    mapper.apply(data)

    # the operator's projection is the oracle's create_wcs for the same bounds / centre
    cfg = CASES[case]
    if cfg.get("auto_bounds", True):
        assert not pix.auto_bounds and len(pix.bounds) == 4
        wo, shape = OW.create_wcs(cfg["projection"], bounds_deg=pix.bounds,
                                  res_deg=cfg["resolution"])
    else:
        wo, shape = OW.create_wcs(cfg["projection"], center_deg=cfg["center"],
                                  res_deg=cfg["resolution"], dims=cfg["dimensions"])
    assert tuple(shape) == tuple(pix.wcs_shape)
    np.testing.assert_array_equal(wo.crpix, pix.wcs.crpix)
    np.testing.assert_array_equal(wo.cdelt, pix.wcs.cdelt)
    np.testing.assert_array_equal(wo.euler, pix.wcs.euler)
    pb = WP.build_wcs_problem(obs, O, wcs=wo, submaps=cfg["submaps"], rcond_threshold=1.0e-6)
    if case == "TAN-fixed":
        assert (pb.pixels < -1).any(), "no sample fell off the fixed image"

    dist = data["pixel_dist"]
    assert dist.wcs_shape == tuple(pix.wcs_shape) and dist.wcs is pix.wcs
    assert dist.n_pix == shape[0] * shape[1]
    np.testing.assert_array_equal(dist.global_submap_to_local, pb.global2local)
    hits_ref = np.zeros(pb.n_local_submap * pb.n_pix_submap, dtype=np.int64)
    sf0 = ((obs["det_flags"] & 1) != 0) | ((obs["shared_flags"] & 1) != 0)[None, :]
    for d in range(n_det):
        for iv in pb.intervals:
            a, b = int(iv["first"]), int(iv["last"])
            sm, lp = O.global_to_local(pb.pixels[d, a:b], pb.n_pix_submap, pb.global2local)
            lp[sf0[d, a:b]] = -1
            O.cov_accum_diag_hits(pb.n_local_submap, pb.n_pix_submap, 3, sm, lp, hits_ref)
    assert hits_ref.sum() > 0
    np.testing.assert_array_equal(data["mm_hits"].raw, hits_ref)
    np.testing.assert_array_equal(data["mm_cov"].data, pb.cov)
    np.testing.assert_array_equal(data["mm_rcond"].raw, pb.rcond)
    assert (pb.rcond > 0).sum() > 20 and (pb.amp_flags == 0).sum() > 100

    np.testing.assert_array_equal(tmpl._amp_flags, pb.amp_flags != 0)
    np.testing.assert_array_equal(tmpl._offsetvar, pb.offset_var)
    np.testing.assert_array_equal(data["amplitudes"]["baselines"].local_flags != 0,
                                  pb.amp_flags != 0)

    covapply = O.cov_apply_diag
    np.testing.assert_array_equal(data["mm_binmap"].data, O.bin_map(pb, O, signal0, covapply))
    rhs_ref = O.solver_rhs(pb, O, signal0, covapply)
    amps_ref, hist_ref = O.solve(pb, O, rhs_ref, convergence=1e-30, n_iter_max=8,
                                 covapply=covapply)
    assert mapper.history == hist_ref
    amps = data["amplitudes"]["baselines"].local
    np.testing.assert_array_equal(amps, amps_ref)
    clean = signal0.copy()
    O.template_add(pb, O, -amps, clean)
    np.testing.assert_array_equal(data.obs[0].detdata["signal"].data, clean)
    assert_close_norm(data["mm_map"].data, O.bin_map(pb, O, clean, covapply), rtol=1e-15,
                      what="destriped map")


def _bounds_of(observations, is_azimuth=False):
    """The auto bounds as PixelsWCS._exec formed them inline (pixels_wcs.py:436-489)."""
    mm = np.array([scan_range_lonlat_deg(o["boresight"], o["shared_flags"], 1, FOV, is_azimuth)
                   for o in observations]).T
    _unwrap_together(mm[0], mm[1])
    return (float(mm[0].min()), float(mm[1].min()), float(mm[2].min()), float(mm[3].max()))


@pytest.mark.parametrize("n_obs", [1, 2])
def test_wcs_geometry_of_one_and_two_observations(monkeypatch, n_obs):
    """PixelsWCS._geometry (shared by _exec and MapMaker) gives the bounds and the shape the
    operator's auto-bounds code gave, for one observation and for two."""
    obs = S.make_observation("c2", n_det=4, n_samp=12000, with_signal=False)
    parts = [obs] if n_obs == 1 else list(_split(obs, 4500))
    data = Data()
    for k, o in enumerate(parts):
        data.obs.append(observation_from_synthetic(o, name=f"obs{k}"))
    dp = ops.PointingDetectorSimple(view="scanning", shared_flags="flags", shared_flag_mask=1)
    pix = ops.PixelsWCS(detector_pointing=dp, projection="CAR", field_of_view=FOV,
                        resolution=(0.3, 0.3), submaps=5)
    pix._geometry(data)
    bounds = _bounds_of(parts)
    assert pix.bounds == bounds and not pix.auto_bounds
    _, shape = OW.create_wcs("CAR", bounds_deg=bounds, res_deg=(0.3, 0.3))
    assert tuple(pix.wcs_shape) == tuple(shape)
    n_pix = shape[0] * shape[1]
    assert (pix._n_pix, pix._n_submap, pix._n_pix_submap) == WP.wcs_submaps(pix.wcs, 5)
    assert pix._n_pix == n_pix
    # the operator's own run derives the same projection (it calls the same method)
    fake_device.install_operator_kernels(monkeypatch)
    import toast_b200.ops.pixels_wcs as PW
    from test_pixels_wcs import _host_pixels_wcs

    monkeypatch.setattr(PW.K, "pixels_wcs", _host_pixels_wcs)
    pix2 = ops.PixelsWCS(detector_pointing=dp, projection="CAR", field_of_view=FOV,
                         resolution=(0.3, 0.3), submaps=5)
    pix2.apply(data)
    assert pix2.bounds == bounds and tuple(pix2.wcs_shape) == tuple(shape)


def _split(obs, cut):
    iv = [(int(v["first"]), int(v["last"])) for v in obs["intervals"]]
    for a, b, ranges in ((0, cut, [r for r in iv if r[1] <= cut]),
                         (cut, obs["n_samp"], [r for r in iv if r[0] >= cut])):
        o = dict(obs)
        o["n_samp"] = b - a
        o["boresight"] = np.ascontiguousarray(obs["boresight"][a:b])
        o["shared_flags"] = np.ascontiguousarray(obs["shared_flags"][a:b])
        o["det_flags"] = np.ascontiguousarray(obs["det_flags"][:, a:b])
        o["intervals"] = S.make_intervals([(f - a, l - a) for f, l in ranges])
        yield o


@pytest.mark.parametrize("trait,value", [("fits_header", "map.fits"),
                                         ("center_offset", "source")])
def test_mapmaker_wcs_refuses_what_it_does_not_implement(monkeypatch, trait, value):
    _install(monkeypatch)
    obs = S.make_observation("c2", n_det=2, n_samp=4000, eps_max=0.03)
    data = Data()
    data.obs.append(observation_from_synthetic(obs))
    dp = ops.PointingDetectorSimple(view="scanning", shared_flags="flags", shared_flag_mask=1)
    pix = ops.PixelsWCS(detector_pointing=dp, projection="CAR", field_of_view=FOV,
                        resolution=(0.5, 0.5), create_dist="pixel_dist", **{trait: value})
    mapper, _ = _mapper(pix, obs, iter_max=2)
    with pytest.raises(NotImplementedError, match=trait):
        mapper.apply(data)
    assert "mm_map" not in data


@pytest.mark.parametrize("name,n_det,n_samp,nside", [("c1", 4, 6000, 16), ("c2", 6, 12000, 64)])
def test_wcs_problem_assembly_restates_build_problem(name, n_det, n_samp, nside):
    """tests/wcs_problem.py assembles the WCS problem with its own restatement of the set-up
    stages of oracle.build_problem: on the HEALPix pointing it must give build_problem's problem
    bit for bit, attribute by attribute."""
    obs = S.make_observation(name, n_det=n_det, n_samp=n_samp, nside=nside, eps_max=0.03)
    ref = O.build_problem(obs, O, rcond_threshold=1.0e-3)
    got = WP.build_healpix_problem(obs, O, rcond_threshold=1.0e-3)
    assert set(ref.__dict__) == set(got.__dict__)
    for key, value in ref.__dict__.items():
        if isinstance(value, np.ndarray):
            np.testing.assert_array_equal(getattr(got, key), value, err_msg=key)
        else:
            assert getattr(got, key) == value, key
