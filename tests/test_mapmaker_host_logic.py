"""ops.MapMaker's HOST LOGIC in the CPU suite: the operator runs with device="cpu" against the
stand-ins of tests/fake_device.py (the oracle does the per-sample compute), and its products must
be what the oracle's own restatement of the reference stages gives -- the same assertions as
tests/test_gpu_ops.py::test_mapmaker_end_to_end makes on the GPU with the real kernels.  What
this covers is everything between the kernels: solver flags, the pixel distribution, the rcond
mask, amplitude flags and variances, the stage order, the products and where they land."""

import numpy as np
import pytest

import fake_device
import helpers as H
from helpers import O, S, assert_close_norm
from toast_b200 import ops
from toast_b200.data import Data, observation_from_synthetic
from toast_b200.templates import Offset


@pytest.mark.parametrize("name,n_det,n_samp,nside", [("c1", 4, 6000, 64), ("c2", 6, 12000, 64)])
def test_mapmaker_host_logic_with_oracle_compute(monkeypatch, name, n_det, n_samp, nside):
    fake_device.install(monkeypatch)
    obs = S.make_observation(name, n_det=n_det, n_samp=n_samp, nside=nside, eps_max=0.03)
    data = Data()
    data.obs.append(observation_from_synthetic(obs))
    pb = O.build_problem(obs, O, rcond_threshold=1.0e-3)
    dp = ops.PointingDetectorSimple(view="scanning", shared_flags="flags", shared_flag_mask=1)
    pix = ops.PixelsHealpix(detector_pointing=dp, nside=obs["nside"], nest=obs["nest"],
                            create_dist="pixel_dist")
    wts = ops.StokesWeights(detector_pointing=dp, mode="IQU")
    binning = ops.BinMap(pixel_dist="pixel_dist", covariance="cov", pixel_pointing=pix,
                         stokes_weights=wts, noise_model="noise_model", full_pointing=True)
    tmpl = Offset(name="baselines", step_time=obs["step_time"], times="times",
                  noise_model="noise_model")
    tmat = ops.TemplateMatrix(templates=[tmpl], amplitudes="amplitudes")
    mapper = ops.MapMaker(name="mm", det_data="signal", binning=binning, template_matrix=tmat,
                          solve_rcond_threshold=1.0e-3, map_rcond_threshold=1.0e-3, iter_max=8,
                          convergence=1.0e-30, device="cpu")
    signal0 = obs["signal"].copy()
    mapper.apply(data)

    # pixel distribution and the products of CovarianceAndHits
    dist = data["pixel_dist"]
    np.testing.assert_array_equal(dist.global_submap_to_local, pb.global2local)
    hits_ref = np.zeros(pb.n_local_submap * pb.n_pix_submap, dtype=np.int64)
    sf0 = ((obs["det_flags"] & 1) != 0) | ((obs["shared_flags"] & 1) != 0)[None, :]
    for d in range(n_det):
        for iv in pb.intervals:
            a, b = int(iv["first"]), int(iv["last"])
            sm, lp = O.global_to_local(pb.pixels[d, a:b], pb.n_pix_submap, pb.global2local)
            lp[sf0[d, a:b]] = -1
            O.cov_accum_diag_hits(pb.n_local_submap, pb.n_pix_submap, 3, sm, lp, hits_ref)
    np.testing.assert_array_equal(data["mm_hits"].raw, hits_ref)
    assert data["mm_hits"].data.dtype == np.int64
    np.testing.assert_array_equal(data["mm_cov"].data, pb.cov)
    np.testing.assert_array_equal(data["mm_rcond"].raw, pb.rcond)

    # amplitude flags / variance formed by the operator == the oracle's restatement
    # (offset.py:283-344) under the full solver flags, bit for bit
    np.testing.assert_array_equal(tmpl._amp_flags, pb.amp_flags != 0)
    np.testing.assert_array_equal(tmpl._offsetvar, pb.offset_var)
    np.testing.assert_array_equal(data["amplitudes"]["baselines"].local_flags != 0,
                                  pb.amp_flags != 0)

    # raw binned map, PCG history, amplitudes, destriped map, cleaned timestream
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


@pytest.mark.parametrize("traits", ["cal", "hwp_IAU"])
def test_stokes_weights_traits_reach_the_device(monkeypatch, traits):
    """What StokesWeights computes the weights from must be what the device observation gets:
    its `cal` key (ob[cal][det] overrides the focal plane's calibration, stokes_weights.py), its
    half-wave-plate angle, IAU convention and the detectors' gamma.  The operator's products must
    be the oracle's for the problem built with those inputs, and differ from the problem without
    them."""
    fake_device.install(monkeypatch)
    obs = S.make_observation("c1", n_det=4, n_samp=6000, nside=64, eps_max=0.03)
    rng = np.random.default_rng(5)
    plain = dict(obs)
    kw, wkw = {}, {}
    if traits == "cal":
        obs["cal"] = 0.75 + 0.5 * rng.random(obs["n_det"])
        wkw = dict(cal="pointing_cal")
    else:
        obs["gamma"] = 0.3 * rng.random(obs["n_det"])
        kw = dict(hwp=(np.arange(obs["n_samp"]) * 0.0123) % (2 * np.pi), IAU=True)
        wkw = dict(hwp_angle="hwp_angle", IAU=True)
    data = Data()
    data.obs.append(observation_from_synthetic(plain if traits == "cal" else obs))
    ob = data.obs[0]
    if traits == "cal":
        ob["pointing_cal"] = {d: float(c) for d, c in zip(ob.local_detectors, obs["cal"])}
    else:
        ob.shared["hwp_angle"] = kw["hwp"]
    pb = O.build_problem(obs, O, rcond_threshold=1.0e-3, **kw)
    pb_plain = O.build_problem(plain, O, rcond_threshold=1.0e-3)
    dp = ops.PointingDetectorSimple(view="scanning", shared_flags="flags", shared_flag_mask=1)
    pix = ops.PixelsHealpix(detector_pointing=dp, nside=obs["nside"], nest=obs["nest"],
                            create_dist="pixel_dist")
    wts = ops.StokesWeights(detector_pointing=dp, mode="IQU", **wkw)
    binning = ops.BinMap(pixel_dist="pixel_dist", covariance="cov", pixel_pointing=pix,
                         stokes_weights=wts, noise_model="noise_model", full_pointing=True)
    tmpl = Offset(name="baselines", step_time=obs["step_time"], times="times",
                  noise_model="noise_model")
    tmat = ops.TemplateMatrix(templates=[tmpl], amplitudes="amplitudes")
    mapper = ops.MapMaker(name="mm", det_data="signal", binning=binning, template_matrix=tmat,
                          solve_rcond_threshold=1.0e-3, map_rcond_threshold=1.0e-3, iter_max=6,
                          convergence=1.0e-30, device="cpu")
    signal0 = obs["signal"].copy()
    mapper.apply(data)
    assert not np.array_equal(pb.cov, pb_plain.cov)
    np.testing.assert_array_equal(data["mm_cov"].data, pb.cov)
    np.testing.assert_array_equal(data["mm_binmap"].data,
                                  O.bin_map(pb, O, signal0, O.cov_apply_diag))
    rhs_ref = O.solver_rhs(pb, O, signal0)
    amps_ref, hist_ref = O.solve(pb, O, rhs_ref, convergence=1e-30, n_iter_max=6)
    assert mapper.history == hist_ref
    np.testing.assert_array_equal(data["amplitudes"]["baselines"].local, amps_ref)


def test_single_precision_weights_are_refused(monkeypatch):
    fake_device.install(monkeypatch)
    obs = S.make_observation("c1", n_det=2, n_samp=2000, nside=16)
    data = Data()
    data.obs.append(observation_from_synthetic(obs))
    dp = ops.PointingDetectorSimple(view="scanning", shared_flags="flags", shared_flag_mask=1)
    pix = ops.PixelsHealpix(detector_pointing=dp, nside=16, nest=obs["nest"],
                            create_dist="pixel_dist")
    wts = ops.StokesWeights(detector_pointing=dp, mode="IQU", single_precision=True)
    binning = ops.BinMap(pixel_dist="pixel_dist", covariance="cov", pixel_pointing=pix,
                         stokes_weights=wts, noise_model="noise_model", full_pointing=True)
    tmat = ops.TemplateMatrix(templates=[Offset(name="baselines", step_time=obs["step_time"],
                                                times="times", noise_model="noise_model")],
                              amplitudes="amplitudes")
    mapper = ops.MapMaker(name="mm", det_data="signal", binning=binning, template_matrix=tmat,
                          iter_max=2, device="cpu")
    with pytest.raises(NotImplementedError, match="single_precision"):
        mapper.apply(data)


def test_final_products_use_the_map_threshold_and_the_input_flags(monkeypatch):
    """ops/mapmaker.py:386-470, 502-594: the final covariance and maps are made with the binning
    flags (input flags, bad pointing, view) and map_rcond_threshold -- NOT with the solver's
    rcond mask.  With a looser map threshold the products must keep the pixels the solve masked."""
    fake_device.install(monkeypatch)
    obs = S.make_observation("c2", n_det=6, n_samp=12000, nside=64, eps_max=0.03)
    data = Data()
    data.obs.append(observation_from_synthetic(obs))
    solve_thr, map_thr = 1.0e-2, 1.0e-6
    pb_solve = O.build_problem(obs, O, rcond_threshold=solve_thr)
    pb_map = O.build_problem(obs, O, rcond_threshold=map_thr)
    assert (pb_map.rcond > 0).sum() > (pb_solve.rcond > 0).sum()   # the thresholds differ in effect
    dp = ops.PointingDetectorSimple(view="scanning", shared_flags="flags", shared_flag_mask=1)
    pix = ops.PixelsHealpix(detector_pointing=dp, nside=obs["nside"], nest=obs["nest"],
                            create_dist="pixel_dist")
    wts = ops.StokesWeights(detector_pointing=dp, mode="IQU")
    binning = ops.BinMap(pixel_dist="pixel_dist", covariance="cov", pixel_pointing=pix,
                         stokes_weights=wts, noise_model="noise_model", full_pointing=True)
    tmpl = Offset(name="baselines", step_time=obs["step_time"], times="times",
                  noise_model="noise_model")
    tmat = ops.TemplateMatrix(templates=[tmpl], amplitudes="amplitudes")
    mapper = ops.MapMaker(name="mm", det_data="signal", binning=binning, template_matrix=tmat,
                          solve_rcond_threshold=solve_thr, map_rcond_threshold=map_thr,
                          iter_max=5, convergence=1.0e-30, device="cpu")
    signal0 = obs["signal"].copy()
    mapper.apply(data)
    # the solve saw the strict mask ...
    np.testing.assert_array_equal(tmpl._amp_flags, pb_solve.amp_flags != 0)
    rhs_ref = O.solver_rhs(pb_solve, O, signal0)
    _, hist_ref = O.solve(pb_solve, O, rhs_ref, convergence=1e-30, n_iter_max=5)
    assert mapper.history == hist_ref
    # ... the products the loose one, on the input flags
    np.testing.assert_array_equal(data["mm_cov"].data, pb_map.cov)
    np.testing.assert_array_equal(data["mm_rcond"].raw, pb_map.rcond)
    in_view = np.zeros(pb_map.n_samp, dtype=bool)
    for iv in pb_map.intervals:
        in_view[iv["first"]:iv["last"]] = True
    base = (((obs["det_flags"] & 1) != 0) | ((obs["shared_flags"] & 1) != 0)[None, :]
            | ~in_view[None, :] | (pb_map.pixels < 0)).astype(np.uint8)
    pbx = O.Problem(**pb_map.__dict__)
    pbx.solver_flags = base
    np.testing.assert_array_equal(data["mm_binmap"].data,
                                  O.bin_map(pbx, O, signal0, O.cov_apply_diag))
    kept_only_by_map = (pb_map.rcond > 0) & (pb_solve.rcond == 0)
    hit = data["mm_binmap"].data.reshape(-1, 3)[kept_only_by_map]
    assert np.any(hit != 0.0)


def test_a_cut_detector_is_left_out_and_left_alone(monkeypatch):
    """Per-detector cut flags (det_mask): MapMaker solves and maps with the remaining detector
    rows only (gathered from / scattered back to the detdata buffer), the cut detector's
    timestream stays as it was, and the result is the oracle's for the problem without it."""
    fake_device.install(monkeypatch)
    n_det, cut = 6, 2
    obs = S.make_observation("c2", n_det=n_det, n_samp=12000, nside=64, eps_max=0.03)
    data = Data()
    data.obs.append(observation_from_synthetic(obs))
    ob = data.obs[0]
    ob.det_flags[ob.local_detectors[cut]] = 1
    keep = [d for d in range(n_det) if d != cut]
    sub = dict(obs)
    sub["n_det"] = len(keep)
    for key in ("focalplane", "epsilon", "gamma", "cal", "detweight", "sigma", "det_flags",
                "signal"):
        sub[key] = np.ascontiguousarray(obs[key][keep])
    pb = O.build_problem(sub, O, rcond_threshold=1.0e-3)
    dp = ops.PointingDetectorSimple(view="scanning", shared_flags="flags", shared_flag_mask=1)
    pix = ops.PixelsHealpix(detector_pointing=dp, nside=obs["nside"], nest=obs["nest"],
                            create_dist="pixel_dist")
    wts = ops.StokesWeights(detector_pointing=dp, mode="IQU")
    binning = ops.BinMap(pixel_dist="pixel_dist", covariance="cov", pixel_pointing=pix,
                         stokes_weights=wts, noise_model="noise_model", full_pointing=True)
    tmpl = Offset(name="baselines", step_time=obs["step_time"], times="times",
                  noise_model="noise_model")
    tmat = ops.TemplateMatrix(templates=[tmpl], amplitudes="amplitudes")
    mapper = ops.MapMaker(name="mm", det_data="signal", binning=binning, template_matrix=tmat,
                          solve_rcond_threshold=1.0e-3, map_rcond_threshold=1.0e-3, iter_max=5,
                          convergence=1.0e-30, device="cpu")
    mapper.apply(data)
    np.testing.assert_array_equal(data["mm_cov"].data, pb.cov)
    rhs_ref = O.solver_rhs(pb, O, sub["signal"])
    amps_ref, hist_ref = O.solve(pb, O, rhs_ref, convergence=1e-30, n_iter_max=5)
    assert mapper.history == hist_ref
    np.testing.assert_array_equal(data["amplitudes"]["baselines"].local, amps_ref)
    clean = sub["signal"].copy()
    O.template_add(pb, O, -amps_ref, clean)
    got = ob.detdata["signal"].data
    np.testing.assert_array_equal(got[keep], clean)
    np.testing.assert_array_equal(got[cut], obs["signal"][cut])       # untouched


def _split_observation(obs, cut):
    """The synthetic observation cut into two at sample ``cut`` (which lies between two views):
    the same detectors, the same baselines in the same detector-major order."""
    def part(a, b, ranges):
        o = dict(obs)
        o["n_samp"] = b - a
        o["boresight"] = np.ascontiguousarray(obs["boresight"][a:b])
        o["shared_flags"] = np.ascontiguousarray(obs["shared_flags"][a:b])
        o["det_flags"] = np.ascontiguousarray(obs["det_flags"][:, a:b])
        o["signal"] = np.ascontiguousarray(obs["signal"][:, a:b])
        o["intervals"] = S.make_intervals([(f - a, l - a) for f, l in ranges])
        return o

    iv = [(int(v["first"]), int(v["last"])) for v in obs["intervals"]]
    first = [r for r in iv if r[1] <= cut]
    second = [r for r in iv if r[0] >= cut]
    assert len(first) + len(second) == len(iv) and first and second
    return part(0, cut, first), part(cut, obs["n_samp"], second)


def test_two_observations_equal_the_one_they_were_cut_from(monkeypatch):
    """Several observations in one MapMaker call (the usual TOAST job): every observation bins
    into the same map and owns its slice of every detector's amplitudes
    (templates/offset/offset.py:166-253).  One observation cut in two between views is the SAME
    destriping problem -- same baselines, same amplitude order -- so hits, covariance, maps,
    amplitudes and cleaned timestreams must agree with the uncut run (sums re-associated)."""
    fake_device.install(monkeypatch)
    obs = S.make_observation("c2", n_det=4, n_samp=12000, nside=64, eps_max=0.03)

    def run(parts):
        data = Data()
        for k, o in enumerate(parts):
            data.obs.append(observation_from_synthetic(o, name=f"obs{k}"))
        dp = ops.PointingDetectorSimple(view="scanning", shared_flags="flags", shared_flag_mask=1)
        pix = ops.PixelsHealpix(detector_pointing=dp, nside=obs["nside"], nest=obs["nest"],
                                create_dist="pixel_dist")
        wts = ops.StokesWeights(detector_pointing=dp, mode="IQU")
        binning = ops.BinMap(pixel_dist="pixel_dist", covariance="cov", pixel_pointing=pix,
                             stokes_weights=wts, noise_model="noise_model", full_pointing=True)
        tmpl = Offset(name="baselines", step_time=obs["step_time"], times="times",
                      noise_model="noise_model")
        tmat = ops.TemplateMatrix(templates=[tmpl], amplitudes="amplitudes")
        mapper = ops.MapMaker(name="mm", det_data="signal", binning=binning,
                              template_matrix=tmat, solve_rcond_threshold=1.0e-3,
                              map_rcond_threshold=1.0e-3, iter_max=6, iter_min=6,
                              convergence=1.0e-30, device="cpu")
        mapper.apply(data)
        return data, mapper, tmpl

    one, m1, t1 = run([obs])
    two, m2, t2 = run(_split_observation(obs, 4500))
    assert t2._n_local == t1._n_local
    np.testing.assert_array_equal(two["pixel_dist"].global_submap_to_local,
                                  one["pixel_dist"].global_submap_to_local)
    np.testing.assert_array_equal(two["mm_hits"].raw, one["mm_hits"].raw)
    np.testing.assert_array_equal(t2._amp_flags, t1._amp_flags)
    np.testing.assert_array_equal(t2._offsetvar, t1._offsetvar)
    assert_close_norm(two["mm_cov"].data, one["mm_cov"].data, rtol=1e-12, what="covariance")
    assert_close_norm(two["mm_binmap"].data, one["mm_binmap"].data, rtol=1e-12, what="binned map")
    np.testing.assert_allclose(m2.history, m1.history, rtol=1e-10)
    assert_close_norm(two["amplitudes"]["baselines"].local, one["amplitudes"]["baselines"].local,
                      what="amplitudes")
    assert_close_norm(two["mm_map"].data, one["mm_map"].data, what="destriped map")
    cleaned = np.hstack([ob.detdata["signal"].data for ob in two.obs])
    assert_close_norm(cleaned, one.obs[0].detdata["signal"].data, what="cleaned timestreams")


@pytest.mark.parametrize("precond_width,nside,rcond,flags",
                         [(20, 16, 1.0e-6, False),    # banded: needs unflagged baselines
                          (1, 32, 1.0e-3, True)])     # Toeplitz: with flagged baselines
def test_mapmaker_with_the_offset_noise_prior(monkeypatch, precond_width, nside, rcond, flags):
    """MapMaker(use_noise_prior): baselines span the observation, the view only flags samples
    (offset.py:136-141), the prior is built from the variance under the FULL solver flags, the
    LHS gains the inverse amplitude covariance and the preconditioner becomes the banded /
    Toeplitz solve (mapmaker_solve.py:395-412, offset.py:884-1010) -- against the oracle's PCG
    with its restatement of the prior.  (The banded form cannot be built with flagged baselines,
    in the reference as here: 1 / offsetvar = inf fails cholesky_banded, offset.py:520-531.)"""
    from oracle import offset_prior as OP
    from toast_b200.data import NoiseModel

    fake_device.install(monkeypatch, oracle_prior=True)
    obs = S.make_observation("c1", n_det=4, n_samp=6000, nside=nside, eps_max=0.03, flags=flags)
    data = Data()
    ob = observation_from_synthetic(obs)
    data.obs.append(ob)
    dets = ob.local_detectors
    psdfreq, psds = OP.analytic_psd(obs["sigma"], obs["rate"], fknee=0.05, fmin=1e-4, alpha=1.5,
                                    n_freq=300)
    ob["noise_model"] = NoiseModel({d: float(w) for d, w in zip(dets, obs["detweight"])},
                                   {d: psdfreq for d in dets},
                                   {d: psds[i] for i, d in enumerate(dets)})
    pb = O.build_problem(obs, O, rcond_threshold=rcond)
    assert (pb.amp_flags != 0).any() == flags
    dp = ops.PointingDetectorSimple(view="scanning", shared_flags="flags", shared_flag_mask=1)
    pix = ops.PixelsHealpix(detector_pointing=dp, nside=obs["nside"], nest=obs["nest"],
                            create_dist="pixel_dist")
    wts = ops.StokesWeights(detector_pointing=dp, mode="IQU")
    binning = ops.BinMap(pixel_dist="pixel_dist", covariance="cov", pixel_pointing=pix,
                         stokes_weights=wts, noise_model="noise_model", full_pointing=True)
    tmpl = Offset(name="baselines", step_time=obs["step_time"], times="times",
                  noise_model="noise_model", use_noise_prior=True, precond_width=precond_width)
    tmat = ops.TemplateMatrix(templates=[tmpl], amplitudes="amplitudes")
    mapper = ops.MapMaker(name="mm", det_data="signal", binning=binning, template_matrix=tmat,
                          solve_rcond_threshold=rcond, map_rcond_threshold=rcond, iter_max=8,
                          convergence=1.0e-30, device="cpu")
    signal0 = obs["signal"].copy()
    mapper.apply(data)
    np.testing.assert_array_equal(tmpl._offsetvar, pb.offset_var)
    t = ob.shared["times"]
    oprior = OP.build_prior(psdfreq, psds, obs["detweight"], pb.offset_var, pb.n_amp_views,
                            float(t[-1] - t[0]), obs["step_time"], tmpl._obs_rate[0],
                            precond_width=precond_width)
    rhs_ref = O.solver_rhs(pb, O, signal0)
    amps_ref, hist_ref = O.solve(pb, O, rhs_ref, convergence=1e-30, n_iter_max=8, prior=oprior)
    assert mapper.history == hist_ref
    np.testing.assert_array_equal(data["amplitudes"]["baselines"].local, amps_ref)
    # the prior changes the solution (the test is not vacuous)
    amps_plain, _ = O.solve(pb, O, rhs_ref, convergence=1e-30, n_iter_max=8)
    assert np.max(np.abs(amps_plain - amps_ref)) > 1e-6 * np.max(np.abs(amps_ref))


def test_without_the_stand_ins_the_operator_refuses_a_cpu():
    """The product has no CPU path: the same call without tests/fake_device.py fails loudly."""
    import torch

    if torch.cuda.is_available():
        pytest.skip("meaningful on a machine without a device only")
    obs = S.make_observation("c1", n_det=2, n_samp=2000, nside=16)
    data = Data()
    data.obs.append(observation_from_synthetic(obs))
    dp = ops.PointingDetectorSimple(view="scanning", shared_flags="flags", shared_flag_mask=1)
    pix = ops.PixelsHealpix(detector_pointing=dp, nside=16, nest=obs["nest"],
                            create_dist="pixel_dist")
    wts = ops.StokesWeights(detector_pointing=dp, mode="IQU")
    binning = ops.BinMap(pixel_dist="pixel_dist", covariance="cov", pixel_pointing=pix,
                         stokes_weights=wts, noise_model="noise_model", full_pointing=True)
    tmpl = Offset(name="baselines", step_time=obs["step_time"], times="times",
                  noise_model="noise_model")
    tmat = ops.TemplateMatrix(templates=[tmpl], amplitudes="amplitudes")
    for device in ("cpu", "cuda"):
        mapper = ops.MapMaker(name="mm", det_data="signal", binning=binning,
                              template_matrix=tmat, iter_max=2, device=device)
        with pytest.raises(Exception):
            mapper.apply(data)
        assert "mm_map" not in data
