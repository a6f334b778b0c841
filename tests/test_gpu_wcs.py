"""Destriping onto flat-sky WCS maps on the device: the fused WCS pointing expansion
(tb_pointing_fused_wcs), WCS solver observations (tb_obs_create_wcs) with stored and regenerated
pointing, and ops.MapMaker with ops.PixelsWCS, against the three-launch chain and the oracle."""

import ctypes as ct

import numpy as np
import pytest
import torch

import helpers as H
import wcs_problem as WP
from helpers import O, S, assert_close_norm
from oracle import pixels_wcs as OW
from toast_b200 import kernels as K
from toast_b200 import lib as L
from toast_b200 import ops
from toast_b200 import wcs as W
from toast_b200.data import Data, observation_from_synthetic
from toast_b200.solver import DeviceObservation, Destriper
from toast_b200.templates import Offset

pytestmark = pytest.mark.gpu

CENTER = (40.0, -30.0)   # the centre of the synthetic ground scans (synthetic.ground_boresight)
BLOCK_PIX = 128


def _projection(proj, coord="EQU", center=CENTER, res=0.1, dims=(120, 80), bounds=None):
    """The product's FlatWCS and the oracle's Wcs for the same arguments (asserted equal)."""
    azel = coord == "AZEL"
    if bounds is not None:
        wp, _ = W.create_wcs(coord, proj, bounds_deg=bounds, res_deg=(res, res))
        wo, _ = OW.create_wcs(proj, bounds_deg=bounds, res_deg=(res, res), is_azimuth=azel)
    else:
        wp, _ = W.create_wcs(coord, proj, center_deg=center, res_deg=(res, res), dims=dims)
        wo, _ = OW.create_wcs(proj, center_deg=center, res_deg=(res, res), dims=dims,
                              is_azimuth=azel)
    assert tuple(wp.shape) == tuple(wo.shape)
    for a in ("crpix", "cdelt", "euler"):
        np.testing.assert_array_equal(getattr(wp, a), getattr(wo, a))
    return wp, wo


# ---- 1. the fused expansion against the three-launch chain ---------------------------------------
@pytest.mark.parametrize("with_quats", [False, True])
@pytest.mark.parametrize("hwp", [False, True])
@pytest.mark.parametrize("coord", ["EQU", "AZEL"])
@pytest.mark.parametrize("proj", OW.PROJECTIONS)
def test_fused_wcs_matches_the_three_launch_chain(proj, coord, hwp, with_quats):
    obs = S.make_observation("c2", n_det=5, n_samp=9000, with_signal=False, eps_max=0.03)
    n_det, n_samp = obs["n_det"], obs["n_samp"]
    center = CENTER if coord == "EQU" else (360.0 - CENTER[0], CENTER[1])
    # smaller than the scan: samples fall off every side
    wp, _ = _projection(proj, coord, center=center, res=0.1, dims=(120, 80))
    n_pix = wp.shape[0] * wp.shape[1]
    n_submap = 7
    nps = (n_pix + n_submap - 1) // n_submap
    idx = np.arange(n_det, dtype=np.int32)
    iv = obs["intervals"]
    bore = torch.from_numpy(obs["boresight"]).cuda()
    flags = torch.from_numpy(obs["shared_flags"]).cuda()
    h = np.random.default_rng(1).uniform(0, 2 * np.pi, n_samp) if hwp else None
    h_d = None if h is None else torch.from_numpy(h).cuda()
    args = (obs["epsilon"], obs["gamma"], obs["cal"], False)

    quats = torch.full((n_det, n_samp, 4), float("nan"), dtype=torch.float64, device="cuda")
    pix_c = torch.full((n_det, n_samp), -7, dtype=torch.int64, device="cuda")
    w_c = torch.full((n_det, n_samp, 3), float("nan"), dtype=torch.float64, device="cuda")
    hits_c = np.zeros(n_submap, dtype=np.uint8)
    K.pointing_detector(obs["focalplane"], bore, idx, quats, iv, flags, 1)
    K.pixels_wcs(wp, idx, quats, flags, 1, idx, pix_c, iv, hits_c, nps)
    K.stokes_weights_IQU(idx, quats, idx, w_c, h_d if hwp else np.zeros(1), iv, *args)

    q_f = torch.full_like(quats, float("nan")) if with_quats else None
    pix_f = torch.full_like(pix_c, -7)
    w_f = torch.full_like(w_c, float("nan"))
    hits_f = np.zeros(n_submap, dtype=np.uint8)
    K.pointing_fused_wcs(wp, obs["focalplane"], bore, flags, 1, idx if with_quats else None, q_f,
                         idx, pix_f, idx, w_f, h_d, iv, hits_f, nps, *args)

    pc, pf = pix_c.cpu().numpy(), pix_f.cpu().numpy()
    np.testing.assert_array_equal(pf, pc)
    np.testing.assert_array_equal(w_f.cpu().numpy(), w_c.cpu().numpy())   # (NaN == NaN here)
    np.testing.assert_array_equal(hits_f, hits_c)
    if with_quats:
        np.testing.assert_array_equal(q_f.cpu().numpy(), quats.cpu().numpy())
    in_view = np.zeros(n_samp, dtype=bool)
    for v in iv:
        in_view[int(v["first"]):int(v["last"])] = True
    assert np.all(pf[:, ~in_view] == -7)                         # outside every view: untouched
    assert np.all(np.isnan(w_f.cpu().numpy()[:, ~in_view]))
    flagged = in_view & ((obs["shared_flags"] & 1) != 0)
    assert flagged.any() and np.all(pf[:, flagged] == -1)
    good = pf[:, in_view & ~flagged]
    assert (good >= 0).any() and (good == -1).any() and (good < -1).any()   # on and off the map
    assert hits_f.any()


# ---- 2. device pixels == oracle pixels ------------------------------------------------------------
@pytest.mark.parametrize("proj", ["CAR", "TAN", "ZEA"])
def test_fused_wcs_pixels_equal_the_oracle(proj):
    obs = S.make_observation("c2", n_det=6, n_samp=12000, with_signal=False, eps_max=0.03)
    wp, wo = _projection(proj, res=0.11, dims=(200, 140))
    n_det, n_samp = obs["n_det"], obs["n_samp"]
    idx = np.arange(n_det, dtype=np.int32)
    quats = np.zeros((n_det, n_samp, 4))
    O.pointing_detector(obs["focalplane"], obs["boresight"], idx, quats, obs["intervals"],
                        obs["shared_flags"], 1)
    pix = torch.full((n_det, n_samp), -7, dtype=torch.int64, device="cuda")
    w = torch.zeros((n_det, n_samp, 3), dtype=torch.float64, device="cuda")
    K.pointing_fused_wcs(wp, obs["focalplane"], torch.from_numpy(obs["boresight"]).cuda(),
                         torch.from_numpy(obs["shared_flags"]).cuda(), 1, None, None, idx, pix,
                         idx, w, None,
                         obs["intervals"], None, 0, obs["epsilon"], obs["gamma"], obs["cal"],
                         False)
    got = pix.cpu().numpy()
    n_checked = 0
    for d in range(n_det):
        for v in obs["intervals"]:
            a, b = int(v["first"]), int(v["last"])
            ref, dc, dr = OW.pixels_wcs(wo, quats[d, a:b], obs["shared_flags"][a:b], 1)
            ok = (obs["shared_flags"][a:b] & 1) == 0
            # no unflagged sample lies within 1e-9 of a rounding boundary: the comparison is exact
            dist = np.minimum(np.abs(np.abs(dc - np.floor(dc)) - 0.5),
                              np.abs(np.abs(dr - np.floor(dr)) - 0.5))
            assert dist[ok].min() > 1e-9
            np.testing.assert_array_equal(got[d, a:b], ref)
            n_checked += int(ok.sum())
    assert n_checked > 50000


# ---- 3. MapMaker end to end -----------------------------------------------------------------------
CASES = {
    "CAR-auto": dict(projection="CAR", field_of_view=11.0, resolution=(0.5, 0.5), submaps=8),
    "TAN-fixed": dict(projection="TAN", auto_bounds=False, center=CENTER, resolution=(0.4, 0.4),
                      dimensions=(40, 24), submaps=7),
}


@pytest.mark.parametrize("regen", [False, True])
@pytest.mark.parametrize("case", sorted(CASES))
def test_mapmaker_wcs_end_to_end(case, regen):
    ck = H.checker()
    covapply = ck.cov_apply_diag
    n_det, thr, n_iter = 8, 1.0e-6, 12
    obs = S.make_observation("c2", n_det=n_det, n_samp=12000, eps_max=0.03)
    data = Data()
    data.obs.append(observation_from_synthetic(obs))
    dp = ops.PointingDetectorSimple(view="scanning", shared_flags="flags", shared_flag_mask=1)
    cfg = CASES[case]
    pix = ops.PixelsWCS(detector_pointing=dp, create_dist="pixel_dist", **cfg)
    wts = ops.StokesWeights(detector_pointing=dp, mode="IQU")
    binning = ops.BinMap(pixel_dist="pixel_dist", covariance="cov", pixel_pointing=pix,
                         stokes_weights=wts, noise_model="noise_model", full_pointing=True)
    tmpl = Offset(name="baselines", step_time=obs["step_time"], times="times",
                  noise_model="noise_model")
    tmat = ops.TemplateMatrix(templates=[tmpl], amplitudes="amplitudes")
    mapper = ops.MapMaker(name="mm", det_data="signal", binning=binning, template_matrix=tmat,
                          solve_rcond_threshold=thr, map_rcond_threshold=thr, iter_max=n_iter,
                          convergence=1.0e-30, regenerate_pointing=regen)
    signal0 = obs["signal"].copy()
    mapper.apply(data)
    if cfg.get("auto_bounds", True):
        wo, shape = OW.create_wcs(cfg["projection"], bounds_deg=pix.bounds,
                                  res_deg=cfg["resolution"])
    else:
        wo, shape = OW.create_wcs(cfg["projection"], center_deg=cfg["center"],
                                  res_deg=cfg["resolution"], dims=cfg["dimensions"])
    assert tuple(shape) == tuple(pix.wcs_shape)
    np.testing.assert_array_equal(wo.crpix, pix.wcs.crpix)
    pb = WP.build_wcs_problem(obs, ck, wcs=wo, submaps=cfg["submaps"], rcond_threshold=thr)
    assert data["pixel_dist"].wcs_shape == tuple(shape)
    np.testing.assert_array_equal(data["pixel_dist"].global_submap_to_local, pb.global2local)

    hits_ref = np.zeros(pb.n_local_submap * pb.n_pix_submap, dtype=np.int64)
    sf0 = ((obs["det_flags"] & 1) != 0) | ((obs["shared_flags"] & 1) != 0)[None, :]
    for d in range(n_det):
        for iv in pb.intervals:
            a, b = int(iv["first"]), int(iv["last"])
            sm, lp = O.global_to_local(pb.pixels[d, a:b], pb.n_pix_submap, pb.global2local)
            lp[sf0[d, a:b]] = -1
            O.cov_accum_diag_hits(pb.n_local_submap, pb.n_pix_submap, 3, sm, lp, hits_ref)
    np.testing.assert_array_equal(data["mm_hits"].raw, hits_ref)
    assert_close_norm(data["mm_cov"].data, pb.cov, what="covariance")
    np.testing.assert_array_equal(data["mm_rcond"].raw > 0, pb.rcond > 0)
    assert_close_norm(data["mm_binmap"].data, O.bin_map(pb, ck, signal0, covapply),
                      what="binned map")
    rhs_ref = O.solver_rhs(pb, ck, signal0, covapply)
    amps_ref, hist_ref = O.solve(pb, ck, rhs_ref, convergence=1e-30, n_iter_max=n_iter,
                                 covapply=covapply)
    H.assert_history_matches(mapper.history, hist_ref, H.pcg_envelope(pb, rhs_ref, n_iter),
                             what=case)
    amps = data["amplitudes"]["baselines"].local
    clean = signal0.copy()
    O.template_add(pb, O, -amps, clean)
    assert_close_norm(data["mm_map"].data, O.bin_map(pb, ck, clean, covapply),
                      what="destriped map")
    dev = np.abs(amps - amps_ref).max() / np.abs(amps_ref).max()
    assert dev < max(1e-10, 1e3 * H.pcg_envelope(pb, rhs_ref, n_iter)[-1] ** 0.5), dev
    assert_close_norm(data.obs[0].detdata["signal"].data, clean, what="cleaned TOD")


# ---- 4. the solver LHS on WCS pixels -------------------------------------------------------------
# (observation, projection arguments, submaps)
LHS_PROBLEMS = {
    # a fixed image smaller than the scan: samples fall off every side
    "fixed": (dict(n_det=8, n_samp=24000), dict(proj="CAR", res=0.11, dims=(120, 70)), 1),
    # 7 submaps: the last one runs past n_pix, the local map is not a multiple of the block
    "submaps7": (dict(n_det=8, n_samp=24000), dict(proj="TAN", res=0.15, dims=(150, 110)), 7),
    # ~1 degree pixels on a long scan: blocks with more records than one work unit holds
    "coarse": (dict(n_det=32, n_samp=120000), dict(proj="CAR", res=1.0, dims=(40, 30)), 2),
}


def _wcs_problem(pid, ck):
    okw, pkw, submaps = LHS_PROBLEMS[pid]
    obs = S.make_observation("c2", eps_max=0.03, **okw)
    wp, wo = _projection(pkw["proj"], res=pkw["res"], dims=pkw["dims"])
    pb = WP.build_wcs_problem(obs, ck, wcs=wo, submaps=submaps, rcond_threshold=1e-3)
    return obs, wp, pb


def _wcs_device_observation(obs, wp, pb):
    dobs = DeviceObservation(
        focalplane=obs["focalplane"], boresight=obs["boresight"], intervals=obs["intervals"],
        det_scale=pb.det_scale, step_length=pb.step_length, wcs=wp,
        n_pix_submap=pb.n_pix_submap, n_submap=pb.n_submap, global2local=pb.global2local,
        epsilon=obs["epsilon"], gamma=obs["gamma"], cal=obs["cal"],
        shared_flags=pb.shared_flags, shared_flag_mask=pb.shared_flag_mask,
        solver_flags=pb.solver_flags, solver_flag_mask=pb.det_flag_mask)
    hits = np.zeros(pb.n_submap, dtype=np.uint8)
    dobs.expand_pointing(hits)
    np.testing.assert_array_equal(dobs.pixels.cpu().numpy(), pb.pixels)
    np.testing.assert_array_equal(hits, pb.hit_submaps)
    return dobs


def _lhs(ds, a_d):
    q = torch.full_like(a_d, float("nan"))
    ds.lhs(a_d, q)
    return q.cpu().numpy()


@pytest.mark.parametrize("pid", sorted(LHS_PROBLEMS))
def test_lhs_on_wcs_pixels(pid):
    ck = H.checker()
    obs, wp, pb = _wcs_problem(pid, ck)
    n_local = pb.n_local_submap * pb.n_pix_submap
    if pid == "fixed":
        assert (pb.pixels < -1).any() and (pb.pixels == -1).any()
        # the reference's wrap: samples left of column 0 land at the end of the previous row
        idx = np.arange(pb.n_det, dtype=np.int32)
        quats = np.zeros((pb.n_det, pb.n_samp, 4))
        O.pointing_detector(obs["focalplane"], obs["boresight"], idx, quats, pb.intervals,
                            pb.shared_flags, 1)
        in_view = np.zeros(pb.n_samp, dtype=bool)
        for v in pb.intervals:
            in_view[int(v["first"]):int(v["last"])] = True
        in_view &= (pb.shared_flags & 1) == 0
        p, dc, _ = OW.pixels_wcs(pb.wcs, quats[:, in_view].reshape(-1, 4))
        assert np.any((np.around(dc) < 0) & (p >= 0)), "no sample wrapped into the previous row"
    if pid == "submaps7":
        assert pb.n_submap * pb.n_pix_submap > wp.shape[0] * wp.shape[1]
        assert pb.hit_submaps[-1] == 1 and n_local % BLOCK_PIX != 0
    dobs = _wcs_device_observation(obs, wp, pb)
    lib = L.load()
    h = dobs.handle().h
    assert lib.tb_obs_blocked(h) == 1
    n_rec, n_units, n_multi, n_blocks = (ct.c_int64(0) for _ in range(4))
    L.check(lib.tb_obs_blocked_stats(h, ct.byref(n_rec), ct.byref(n_units), ct.byref(n_multi),
                                     ct.byref(n_blocks)))
    print(f"WCS_BLOCKED_STATS {pid}: n_local {n_local} n_records {n_rec.value} "
          f"n_units {n_units.value} n_multi_units {n_multi.value} n_blocks {n_blocks.value}")
    assert n_blocks.value == (n_local + BLOCK_PIX - 1) // BLOCK_PIX
    if pid == "coarse":
        assert n_multi.value > 0
    covapply = ck.cov_apply_diag
    a = np.where(pb.amp_flags == 0, np.random.default_rng(3).standard_normal(pb.n_amp), 0.0)
    ref = O.solver_lhs(pb, ck, a, covapply=covapply)
    a_d = torch.from_numpy(a).cuda()
    ds = Destriper([dobs], pb.n_local_submap, pb.n_pix_submap, pb.cov, pb.offset_var,
                   pb.amp_flags)
    assert ds._blocked()
    got = {}
    for fused in (True, False):
        ds.fuse_lhs = fused
        got[fused] = _lhs(ds, a_d)
        assert_close_norm(got[fused], ref, what=f"{pid} LHS (fused={fused})")
    ds_r = Destriper([dobs], pb.n_local_submap, pb.n_pix_submap, pb.cov, pb.offset_var,
                     pb.amp_flags, regen=True)
    reg = _lhs(ds_r, a_d)
    assert_close_norm(reg, ref, what=f"{pid} LHS (regenerated pointing)")
    assert_close_norm(reg, got[True], what=f"{pid} LHS regenerated vs stored")
    sig = torch.from_numpy(obs["signal"]).cuda()
    assert_close_norm(ds_r.bin_signal([sig]).cpu().numpy(),
                      O.bin_map(pb, ck, obs["signal"], covapply), what=f"{pid} binned (regen)")


# ---- 5. refusals ------------------------------------------------------------------------------------
def _bad_descs(wp):
    out = []
    for field, value in (("projection", 6), ("projection", -1), ("cdelt0", 0.0),
                         ("cdelt1", 0.0), ("n_col", 0), ("n_row", -3)):
        d = wp.desc()
        if field.startswith("cdelt"):
            d.cdelt[int(field[-1])] = value
        else:
            setattr(d, field, value)
        out.append((field, d))
    return out


def test_wcs_entry_points_refuse_bad_projections():
    obs = S.make_observation("c2", n_det=2, n_samp=3000, with_signal=False)
    wp, wo = _projection("CAR", res=0.2, dims=(60, 40))
    lib = L.load()
    n_det, n_samp = 2, 3000
    idx = np.arange(n_det, dtype=np.int32)
    iv = obs["intervals"]
    bore = torch.from_numpy(obs["boresight"]).cuda()
    pix = torch.full((n_det, n_samp), -7, dtype=torch.int64, device="cuda")
    w = torch.zeros((n_det, n_samp, 3), dtype=torch.float64, device="cuda")
    ones, zeros = np.ones(n_det), np.zeros(n_det)
    n_pix = 60 * 40

    def fused(desc, hits, nps):
        return lib.tb_pointing_fused_wcs(
            L.ptr(obs["focalplane"]), L.ptr(bore), None, 0, None, None, 0, L.ptr(idx),
            L.ptr(pix), n_det, L.ptr(idx), L.ptr(w), n_det, None, L.ptr(iv), len(iv),
            L.ptr(hits), len(hits), nps, ct.byref(desc), L.ptr(zeros), L.ptr(zeros),
            L.ptr(ones), 0, n_det, n_samp, L.TB_MEM_DEVICE, None)

    hits = np.zeros(4, dtype=np.uint8)
    launches = lib.tb_launch_count()
    for field, d in _bad_descs(wp):
        assert fused(d, hits, n_pix // 4) != 0, field
    assert fused(wp.desc(), hits, n_pix // 4 - 1) != 0             # hit_submaps too small
    assert "too small" in L.last_error()
    torch.cuda.synchronize()
    assert lib.tb_launch_count() == launches
    assert np.all(pix.cpu().numpy() == -7) and not hits.any()
    assert fused(wp.desc(), hits, n_pix // 4) == 0                 # the good descriptor runs
    assert lib.tb_launch_count() > launches

    # tb_obs_create_wcs
    dobs = DeviceObservation(
        focalplane=obs["focalplane"], boresight=obs["boresight"], intervals=iv,
        det_scale=np.ones(n_det), step_length=100, wcs=wp, n_pix_submap=n_pix // 4, n_submap=4,
        global2local=np.arange(4, dtype=np.int64))
    assert dobs.handle().h                                            # the good one is accepted
    for field, d in _bad_descs(wp):
        dobs.wcs = _Fixed(d)
        dobs.invalidate()
        with pytest.raises(RuntimeError):
            dobs.handle()
    dobs.wcs = wp
    dobs.n_pix_submap = n_pix // 4 - 1
    dobs.invalidate()
    with pytest.raises(RuntimeError, match="cover"):
        dobs.handle()
    assert lib.tb_obs_create_wcs(None, None) is None


class _Fixed:
    """A projection whose descriptor is given as it is."""

    def __init__(self, d):
        self.d = d

    def desc(self):
        return self.d


def test_device_observation_takes_one_pixelisation():
    obs = S.make_observation("c2", n_det=2, n_samp=3000, with_signal=False)
    wp, _ = _projection("CAR", res=0.2, dims=(60, 40))
    kw = dict(focalplane=obs["focalplane"], boresight=obs["boresight"],
              intervals=obs["intervals"], det_scale=np.ones(2), step_length=100,
              n_pix_submap=600, n_submap=4, global2local=np.arange(4, dtype=np.int64))
    with pytest.raises(ValueError):
        DeviceObservation(wcs=wp, nside=64, nest=True, **kw)
    with pytest.raises(ValueError):
        DeviceObservation(**kw)
