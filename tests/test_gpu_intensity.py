"""Intensity-only destriping on the device: observations made by tb_obs_create_intensity
(DeviceObservation(nnz=1), StokesWeights(mode="I")) through every layer that takes them.

* Exact comparisons on the dyadic problems of tests/test_gpu_blocked.py (split blocks, a partial
  last block, an odd detector count) and on the same focalplane with the pair partners pointing
  apart, where the crossing list keeps one row per detector: the block-ordered list's counts
  against the numpy model, and every form of the LHS bit for bit against the numpy reference
  (with one value per pixel, the LHS of the dyadic inputs IS that reference's I-only LHS).
* Oracle parity on the I-only problem of tests/intensity_problem.py: HEALPix NEST and RING, a
  CAR map, and two observations on one GPU.
* ops.MapMaker(mode="I") end to end, and two ranks on the NCCL path."""

import ctypes as ct
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import helpers as H
import intensity_problem as IP
import test_gpu_blocked as GB
from helpers import O, S, assert_close_norm
from oracle import pixels_wcs as OW
from test_gpu_peer import _collect, _free_port, _need
from test_gpu_wcs import _projection
from toast_b200 import lib as L
from toast_b200 import ops
from toast_b200.data import Data, observation_from_synthetic
from toast_b200.solver import DeviceObservation, Destriper
from toast_b200.templates import Offset

pytestmark = pytest.mark.gpu

# the problems of test_gpu_blocked.py, and "apart": `split` with the focalplane rolled by one
# detector, so that the two detectors of every row belong to different polarisation pairs
CASES = list(GB.PROBLEMS) + ["apart"]


def _observation(case, det_first=0, dyadic=True):
    obs = GB._observation("split" if case == "apart" else case, det_first, dyadic)
    if case == "apart":
        obs["focalplane"] = np.ascontiguousarray(np.roll(obs["focalplane"], 1, axis=0))
    return obs


def _device_observation(obs, pb, g2l=None, amp_offset=0, expand=True, wcs=None):
    pix = dict(wcs=wcs) if wcs is not None else dict(nside=pb.nside, nest=pb.nest)
    dobs = DeviceObservation(
        focalplane=obs["focalplane"], boresight=obs["boresight"], intervals=obs["intervals"],
        det_scale=pb.det_scale, step_length=pb.step_length, n_pix_submap=pb.n_pix_submap,
        n_submap=pb.n_submap, global2local=pb.global2local if g2l is None else g2l,
        amp_offset=amp_offset, epsilon=obs["epsilon"], gamma=obs["gamma"], cal=obs["cal"],
        shared_flags=pb.shared_flags, shared_flag_mask=pb.shared_flag_mask,
        solver_flags=pb.solver_flags, solver_flag_mask=pb.det_flag_mask, nnz=1, **pix)
    if expand:
        hits = np.zeros(pb.n_submap, dtype=np.uint8)
        dobs.expand_pointing(hits)
        np.testing.assert_array_equal(dobs.pixels.cpu().numpy(), pb.pixels)
        np.testing.assert_array_equal(hits, pb.hit_submaps)
        w = np.zeros((pb.n_det, pb.n_samp))
        O.stokes_weights_I(np.arange(pb.n_det, dtype=np.int32), w, pb.intervals, obs["cal"])
        np.testing.assert_array_equal(dobs.weights.cpu().numpy(), w)
    assert L.load().tb_obs_nnz(dobs.handle().h) == 1
    return dobs


def _check_block_list(case, dobs, pb, g2l=None):
    """The device built the intensity block-ordered list the numpy model predicts, in the row
    layout with fewer entries: detector pairs for the synthetic (co-pointed) pairs, one row per
    detector when the partners point apart.  Returns the model's entries per block."""
    lib = L.load()
    h = dobs.handle().h
    assert lib.tb_obs_blocked(h) == 1, f"{case}: no block-ordered list"
    n_rec, n_rows, paired = ct.c_int64(0), ct.c_int64(0), ct.c_int(0)
    L.check(lib.tb_obs_crossing_stats(h, ct.byref(n_rec), ct.byref(n_rows), ct.byref(paired)))
    e_pair, e_det = GB._block_entries(pb, True, g2l), GB._block_entries(pb, False, g2l)
    want_paired = int(e_pair.sum() < e_det.sum())
    assert want_paired == (0 if case == "apart" else 1), (case, e_pair.sum(), e_det.sum())
    assert paired.value == want_paired
    assert n_rows.value == ((pb.n_det + 1) // 2 if want_paired else pb.n_det)
    entries = e_pair if want_paired else e_det
    units = GB._units(entries)
    n_rec, n_units, n_multi, n_blocks = (ct.c_int64(0) for _ in range(4))
    L.check(lib.tb_obs_blocked_stats(h, ct.byref(n_rec), ct.byref(n_units), ct.byref(n_multi),
                                     ct.byref(n_blocks)))
    print(f"INTENSITY_BLOCKED_STATS {case}: paired {paired.value} n_records {n_rec.value} "
          f"(pairs {int(e_pair.sum())}, detectors {int(e_det.sum())}) n_units {n_units.value} "
          f"n_multi_units {n_multi.value} n_blocks {n_blocks.value}")
    assert n_blocks.value == len(entries)
    assert (n_rec.value, n_units.value, n_multi.value) == \
        (int(entries.sum()), int(units.sum()), int(units[units > 1].sum())), f"{case}: model"
    assert n_multi.value > 0
    if case in GB.TAILS:
        g2l = pb.global2local if g2l is None else g2l
        assert int(np.sum(g2l >= 0)) * pb.n_pix_submap % GB.BLOCK_PIX != 0 and entries[-1] > 0
    return entries


def _cov1(cii, n_local, nps):
    return np.ascontiguousarray(cii.reshape(n_local, nps, 1))


@pytest.fixture(scope="module", params=CASES)
def dyadic(request):
    """A dyadic problem on the device as an intensity observation, with its numpy reference (the
    flags and amplitude layout are those of the problem's oracle set-up)."""
    case = request.param
    obs = _observation(case)
    pb = O.build_problem(obs, O, rcond_threshold=1e-3)
    cii = GB._dyadic_cov(pb)[..., 0].reshape(-1)
    amps, aflags = GB._dyadic_amplitudes(pb)
    n_pix = pb.n_local_submap * pb.n_pix_submap
    ref = GB.DyadicReference([(pb, pb.global2local, 0)], n_pix, amps, aflags)
    zI, lhs = ref.lhs(cii)
    dobs = _device_observation(obs, pb)
    entries = _check_block_list(case, dobs, pb)
    if case in GB.TAILS:
        assert np.any(zI[(len(entries) - 1) * GB.BLOCK_PIX:] != 0.0)
    cov = _cov1(cii, pb.n_local_submap, pb.n_pix_submap)
    ds = Destriper([dobs], pb.n_local_submap, pb.n_pix_submap, cov, pb.offset_var, aflags)
    assert ds._blocked() and ds.nnz == 1
    assert tuple(ds.zmap.shape) == (pb.n_local_submap, pb.n_pix_submap, 1)
    return SimpleNamespace(case=case, obs=obs, pb=pb, cov=cov, cii=cii, amps=amps, aflags=aflags,
                           n_pix=n_pix, ref=ref, zI=zI, lhs=lhs, dobs=dobs, ds=ds,
                           h=dobs.handle().h, entries=entries,
                           a_d=torch.from_numpy(amps).cuda())


def _lhs(ds, a_d):
    q = torch.full_like(a_d, float("nan"))
    ds.lhs(a_d, q)
    return q.cpu().numpy()


# ---- exact references on dyadic inputs -----------------------------------------------------------
@pytest.mark.parametrize("fused", [True, False])
def test_intensity_lhs_is_exact_and_repeatable(dyadic, fused):
    ds = dyadic.ds
    ds.fuse_lhs = fused
    try:
        ds.zmap.fill_(float("nan"))
        first = _lhs(ds, dyadic.a_d)
        second = _lhs(ds, dyadic.a_d)
    finally:
        ds.fuse_lhs = True
    np.testing.assert_array_equal(first, dyadic.lhs)
    np.testing.assert_array_equal(second, dyadic.lhs)
    if not fused:
        np.testing.assert_array_equal(ds.zmap.cpu().numpy().reshape(-1), dyadic.cii * dyadic.zI)


def test_intensity_pass1_and_pass2_alone(dyadic):
    lib = L.load()
    d, z = dyadic, dyadic.ds.zmap
    aflags_d = dyadic.ds.amp_flags
    z.fill_(float("nan"))
    L.check(lib.tb_bx_pass1(d.h, L.ptr(d.a_d), L.ptr(aflags_d), L.ptr(z), 0, -1, None))
    np.testing.assert_array_equal(z.cpu().numpy().reshape(-1), d.zI)
    rng = np.random.default_rng(1)
    known = rng.integers(-64, 65, d.n_pix) * 0.25
    z.copy_(torch.from_numpy(known.reshape(z.shape)))
    L.check(lib.tb_bx_pass1(d.h, L.ptr(d.a_d), L.ptr(aflags_d), L.ptr(z), 1, -1, None))
    np.testing.assert_array_equal(z.cpu().numpy().reshape(-1), known + d.zI)
    m = rng.integers(-512, 513, d.n_pix) * 2.0 ** -8
    z.copy_(torch.from_numpy(m.reshape(z.shape)))
    q = torch.zeros_like(d.a_d)
    L.check(lib.tb_bx_pass2(d.h, L.ptr(z), L.ptr(q), -1, None))
    np.testing.assert_array_equal(q.cpu().numpy(), d.ref.pass2(m))


def test_intensity_pixel_chunked_passes(dyadic):
    lib = L.load()
    d, ds = dyadic, dyadic.ds
    split = np.flatnonzero(GB._units(d.entries) > 1)
    around = np.unique(np.minimum(d.n_pix, np.concatenate(
        [[0, d.n_pix], split * GB.BLOCK_PIX, (split + 1) * GB.BLOCK_PIX])))
    every = list(range(0, d.n_pix, GB.BLOCK_PIX)) + [d.n_pix]
    try:
        for bounds in (around, every):
            b = np.ascontiguousarray(bounds, dtype=np.int64)
            n_chunks = len(b) - 1
            L.check(lib.tb_obs_set_pixel_chunks(d.h, n_chunks, L.ptr(b)))
            ds.zmap.fill_(float("nan"))
            for c in range(n_chunks):
                L.check(lib.tb_bx_pass1(d.h, L.ptr(d.a_d), L.ptr(ds.amp_flags), L.ptr(ds.zmap), 0,
                                        c, None))
            ds.reduce_and_apply_cov()
            q = torch.zeros_like(d.a_d)
            for c in reversed(range(n_chunks)):
                L.check(lib.tb_bx_pass2(d.h, L.ptr(ds.zmap), L.ptr(q), c, None))
            np.testing.assert_array_equal(q.cpu().numpy(), d.lhs,
                                          err_msg=f"chunk bounds {b.tolist()}")
    finally:
        whole = np.array([0, d.n_pix], dtype=np.int64)
        L.check(lib.tb_obs_set_pixel_chunks(d.h, 1, L.ptr(whole)))


def test_intensity_per_sample_and_regenerated_lhs_are_exact(dyadic):
    """blocked = 0 (k_bin / k_project on the stored I weights) and regenerated pointing (w = cal)."""
    lib = L.load()
    d = dyadic
    try:
        L.check(lib.tb_set_option(b"blocked", 0))
        dobs = _device_observation(d.obs, d.pb)
        ds = Destriper([dobs], d.pb.n_local_submap, d.pb.n_pix_submap, d.cov, d.pb.offset_var,
                       d.aflags)
        assert not ds._blocked()
        np.testing.assert_array_equal(_lhs(ds, d.a_d), d.lhs, err_msg="blocked=0")
    finally:
        lib.tb_set_option(b"blocked", 1)
    dobs = _device_observation(d.obs, d.pb, expand=False)
    ds = Destriper([dobs], d.pb.n_local_submap, d.pb.n_pix_submap, d.cov, d.pb.offset_var,
                   d.aflags, regen=True)
    np.testing.assert_array_equal(_lhs(ds, d.a_d), d.lhs, err_msg="regen")


@pytest.mark.parametrize("pid", ["split", "split_tail"])
def test_intensity_two_observations_accumulate(pid):
    n_det = GB.PROBLEMS[pid][1]
    obs = [_observation(pid, det_first=k * n_det) for k in range(2)]
    pbs = [O.build_problem(o, O, rcond_threshold=1e-3) for o in obs]
    hit = pbs[0].hit_submaps | pbs[1].hit_submaps
    _, g2l = O.pixel_distribution(hit)
    n_local, nps = int(np.sum(hit != 0)), pbs[0].n_pix_submap
    n_pix = n_local * nps
    keep = np.zeros((n_local, nps), dtype=bool)
    for pb in pbs:
        keep[g2l[pb.local_submaps]] |= pb.rcond.reshape(-1, nps) > 0
    cii = np.where(keep, GB.COV_II, 0.0).reshape(-1)
    offsets = [0, pbs[0].n_amp]
    amps = np.concatenate([GB._dyadic_amplitudes(pb, seed=k)[0] for k, pb in enumerate(pbs)])
    aflags = np.concatenate([pb.amp_flags for pb in pbs])
    aflags[::7] = 1
    ref = GB.DyadicReference([(pb, g2l, off) for pb, off in zip(pbs, offsets)], n_pix, amps,
                             aflags)
    zI, lhs = ref.lhs(cii)
    dobs = []
    for o, pb, off in zip(obs, pbs, offsets):
        dobs.append(_device_observation(o, pb, g2l=g2l, amp_offset=off))
        _check_block_list(pid, dobs[-1], pb, g2l)
    ds = Destriper(dobs, n_local, nps, _cov1(cii, n_local, nps),
                   np.concatenate([pb.offset_var for pb in pbs]), aflags)
    assert ds._blocked()
    a_d = torch.from_numpy(amps).cuda()
    ds.zmap.fill_(float("nan"))
    np.testing.assert_array_equal(_lhs(ds, a_d), lhs)
    np.testing.assert_array_equal(ds.zmap.cpu().numpy().reshape(-1), cii * zI)
    np.testing.assert_array_equal(_lhs(ds, a_d), lhs)


def test_mixed_nnz_is_refused():
    obs = GB._observation("split_partial")
    pb = O.build_problem(obs, O, rcond_threshold=1e-3)
    d1 = _device_observation(obs, pb, expand=False)
    d3 = GB._device_observation(obs, pb, expand=False)
    cov = np.zeros((pb.n_local_submap, pb.n_pix_submap, 1))
    with pytest.raises(ValueError, match="nnz"):
        Destriper([d1, d3], pb.n_local_submap, pb.n_pix_submap, cov,
                  np.concatenate([pb.offset_var] * 2), np.concatenate([pb.amp_flags] * 2))


# ---- oracle parity on the I-only problem ---------------------------------------------------------
PARITY = {
    "nest": dict(nest=True),
    "ring": dict(nest=False),
    "car": dict(wcs=dict(proj="CAR", res=0.15, dims=(150, 110)), submaps=7),
}


def _parity_problem(case, ck, n_det=8, n_samp=24000, det_first=0):
    cfg = PARITY[case]
    obs = S.make_observation("c2", n_det=n_det, n_samp=n_samp, det_first=det_first, nside=64,
                             eps_max=0.03)
    wp = None
    if "wcs" in cfg:
        w = cfg["wcs"]
        wp, wo = _projection(w["proj"], res=w["res"], dims=w["dims"])
        pb = IP.build_problem(obs, ck, nnz=1, wcs=wo, submaps=cfg["submaps"])
    else:
        obs["nest"] = cfg["nest"]
        pb = IP.build_problem(obs, ck, nnz=1)
    return obs, pb, wp


@pytest.mark.parametrize("case", sorted(PARITY))
def test_intensity_oracle_parity(case):
    """LHS (fused and three-launch), RHS, binned map and ten restarted PCG iterations against
    the I-only oracle problem."""
    ck = H.checker()
    obs, pb, wp = _parity_problem(case, ck)
    dobs = _device_observation(obs, pb, wcs=wp)
    assert L.load().tb_obs_blocked(dobs.handle().h) == 1
    ds = Destriper([dobs], pb.n_local_submap, pb.n_pix_submap, pb.cov, pb.offset_var,
                   pb.amp_flags)
    assert ds._blocked()
    covapply = ck.cov_apply_diag
    rng = np.random.default_rng(3)
    a = np.where(pb.amp_flags == 0, rng.standard_normal(pb.n_amp), 0.0)
    ref = IP.solver_lhs(pb, ck, a, covapply)
    a_d = torch.from_numpy(a).cuda()
    for fused in (True, False):
        ds.fuse_lhs = fused
        assert_close_norm(_lhs(ds, a_d), ref, what=f"{case} LHS (fused={fused})")
    ds.fuse_lhs = True
    sig = torch.from_numpy(obs["signal"]).cuda()
    rhs_ref = IP.solver_rhs(pb, ck, obs["signal"], covapply)
    assert_close_norm(ds.rhs([sig]).cpu().numpy(), rhs_ref, what=f"{case} RHS")
    assert_close_norm(ds.bin_signal([sig]).cpu().numpy(), IP.bin_map(pb, ck, obs["signal"],
                                                                      covapply),
                      what=f"{case} binned map")
    trace = []
    IP.solve(pb, ck, rhs_ref, n_iter_max=10, covapply=covapply, trace=trace)
    assert len(trace) == 10
    H.restart_parity(ds, pb, trace, what=case)


def test_intensity_oracle_parity_two_observations():
    """Two observations on one GPU sharing the union of their submaps, against the oracle's
    LHS of the two observations on that map (the sum of their noise-weighted maps)."""
    ck = H.checker()
    parts = [_parity_problem("nest", ck, det_first=8 * k) for k in range(2)]
    hit = parts[0][1].hit_submaps | parts[1][1].hit_submaps
    _, g2l = O.pixel_distribution(hit)
    n_local, nps = int(np.sum(hit != 0)), parts[0][1].n_pix_submap
    # the covariance of the union: both observations' inverse covariances, inverted
    inv = np.zeros(n_local * nps)
    for obs, pb, _ in parts:
        sub = np.zeros((n_local, nps))
        sub[g2l[pb.local_submaps]] = pb.invcov.reshape(-1, nps)
        inv += sub.reshape(-1)
    cov = inv.copy()
    O.cov_eigendecompose_diag(n_local, nps, 1, cov, None, 1e-3, True)
    offsets = [0, parts[0][1].n_amp]
    rng = np.random.default_rng(4)
    amps, aflags, dobs = [], [], []
    for (obs, pb, _), off in zip(parts, offsets):
        amps.append(np.where(pb.amp_flags == 0, rng.standard_normal(pb.n_amp), 0.0))
        aflags.append(pb.amp_flags)
        dobs.append(_device_observation(obs, pb, g2l=g2l, amp_offset=off))
    amps, aflags = np.concatenate(amps), np.concatenate(aflags)
    ds = Destriper(dobs, n_local, nps, cov.reshape(n_local, nps, 1),
                   np.concatenate([p[1].offset_var for p in parts]), aflags)
    assert ds._blocked()
    # the oracle: bin both observations into one map, apply C, scan back per observation
    z = np.zeros((n_local, nps, 1))
    tods = []
    for (obs, pb, _), off in zip(parts, offsets):
        pbu = SimpleNamespace(**pb.__dict__)
        pbu.global2local, pbu.n_local_submap = g2l, n_local
        pbu.det_start = pb.det_start + off
        pbu.amp_flags = aflags
        tod = np.zeros((pb.n_det, pb.n_samp))
        O.template_add(pbu, ck, amps, tod)
        idx = np.arange(pb.n_det, dtype=np.int32)
        ck.build_noise_weighted(g2l, z, idx, pb.pixels, idx, IP._weights3(pb), idx, tod, idx,
                                pb.solver_flags, pb.det_scale, pb.det_flag_mask, pb.intervals,
                                pb.shared_flags, pb.shared_flag_mask, False)
        tods.append((pbu, tod))
    ck.cov_apply_diag(n_local, nps, 1, cov, z.reshape(-1))
    ref = np.zeros_like(amps)
    for pbu, tod in tods:
        IP._scan_weight_project(pbu, ck, z, tod, ref)
    for fused in (True, False):   # (several observations: the fused kernel is not used)
        ds.fuse_lhs = fused
        assert_close_norm(_lhs(ds, torch.from_numpy(amps).cuda()), ref, what="two observations")


# ---- MapMaker(mode="I") end to end ---------------------------------------------------------------
def _envelope(pb, rhs, n_iter):
    """helpers.pcg_envelope for the I-only problem."""
    rng = np.random.default_rng(0)
    rhs2 = rhs * (1.0 + 2.2e-16 * rng.choice([-1.0, 1.0], size=rhs.shape))
    _, h1 = IP.solve(pb, O, rhs, n_iter_max=n_iter)
    _, h2 = IP.solve(pb, O, rhs2, n_iter_max=n_iter)
    n = min(len(h1), len(h2))
    return np.maximum.accumulate(np.abs(np.array(h2[:n]) - np.array(h1[:n])) / np.array(h1[:n]))


@pytest.mark.parametrize("regen", [False, True])
@pytest.mark.parametrize("pixelisation", ["healpix", "car"])
def test_mapmaker_intensity_end_to_end(pixelisation, regen):
    ck = H.checker()
    covapply = ck.cov_apply_diag
    n_det, n_iter = 8, 12
    obs = S.make_observation("c2", n_det=n_det, n_samp=12000, nside=64, eps_max=0.03)
    data = Data()
    data.obs.append(observation_from_synthetic(obs))
    dp = ops.PointingDetectorSimple(view="scanning", shared_flags="flags", shared_flag_mask=1)
    if pixelisation == "healpix":
        pix = ops.PixelsHealpix(detector_pointing=dp, nside=obs["nside"], nest=obs["nest"],
                                create_dist="pixel_dist")
    else:
        pix = ops.PixelsWCS(detector_pointing=dp, create_dist="pixel_dist", projection="CAR",
                            field_of_view=11.0, resolution=(0.5, 0.5), submaps=8)
    wts = ops.StokesWeights(detector_pointing=dp, mode="I")
    binning = ops.BinMap(pixel_dist="pixel_dist", covariance="cov", pixel_pointing=pix,
                         stokes_weights=wts, noise_model="noise_model", full_pointing=True)
    tmpl = Offset(name="baselines", step_time=obs["step_time"], times="times",
                  noise_model="noise_model")
    tmat = ops.TemplateMatrix(templates=[tmpl], amplitudes="amplitudes")
    mapper = ops.MapMaker(name="mm", det_data="signal", binning=binning, template_matrix=tmat,
                          solve_rcond_threshold=1e-3, map_rcond_threshold=1e-3, iter_max=n_iter,
                          convergence=1.0e-30, regenerate_pointing=regen)
    signal0 = obs["signal"].copy()
    mapper.apply(data)
    if pixelisation == "healpix":
        pb = IP.build_problem(obs, ck, nnz=1)
    else:
        wo, shape = OW.create_wcs("CAR", bounds_deg=pix.bounds, res_deg=(0.5, 0.5))
        wo.shape = tuple(shape)
        pb = IP.build_problem(obs, ck, nnz=1, wcs=wo, submaps=8)
    np.testing.assert_array_equal(data["pixel_dist"].global_submap_to_local, pb.global2local)
    hits_ref = np.zeros(pb.n_local_submap * pb.n_pix_submap, dtype=np.int64)
    sf0 = ((obs["det_flags"] & 1) != 0) | ((obs["shared_flags"] & 1) != 0)[None, :]
    for d in range(n_det):
        for iv in pb.intervals:
            a, b = int(iv["first"]), int(iv["last"])
            sm, lp = O.global_to_local(pb.pixels[d, a:b], pb.n_pix_submap, pb.global2local)
            lp[sf0[d, a:b]] = -1
            O.cov_accum_diag_hits(pb.n_local_submap, pb.n_pix_submap, 1, sm, lp, hits_ref)
    np.testing.assert_array_equal(data["mm_hits"].raw, hits_ref)
    for key in ("mm_cov", "mm_binmap", "mm_map"):
        assert data[key].n_value == 1, key
    assert_close_norm(data["mm_cov"].data, pb.cov, what="covariance")
    np.testing.assert_array_equal(data["mm_rcond"].raw, pb.rcond)
    assert_close_norm(data["mm_binmap"].data, IP.bin_map(pb, ck, signal0, covapply),
                      what="binned map")
    rhs_ref = IP.solver_rhs(pb, ck, signal0, covapply)
    amps_ref, hist_ref = IP.solve(pb, ck, rhs_ref, convergence=1e-30, n_iter_max=n_iter,
                                  covapply=covapply)
    env = _envelope(pb, rhs_ref, n_iter)
    H.assert_history_matches(mapper.history, hist_ref, env, what=pixelisation)
    amps = data["amplitudes"]["baselines"].local
    dev = np.abs(amps - amps_ref).max() / np.abs(amps_ref).max()
    assert dev < max(1e-10, 1e3 * env[-1] ** 0.5), dev
    clean = signal0.copy()
    O.template_add(pb, O, -amps, clean)
    assert_close_norm(data["mm_map"].data, IP.bin_map(pb, ck, clean, covapply),
                      what="destriped map")


# ---- two ranks on the NCCL path ------------------------------------------------------------------
def _nccl_worker(rank, world, port, out):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ["OMP_NUM_THREADS"] = "1"
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world,
                            device_id=torch.device("cuda", rank))
    try:
        obs = S.make_observation("c4", n_det=6, n_samp=24000, nside=64, eps_max=0.03)
        pb = IP.build_problem(obs, O, nnz=1)
        per = pb.n_det // world
        sl = slice(rank * per, (rank + 1) * per)
        nad = int(pb.n_amp_views.sum())
        asl = slice(rank * per * nad, (rank + 1) * per * nad)
        dobs = DeviceObservation(
            focalplane=obs["focalplane"][sl], boresight=obs["boresight"],
            intervals=obs["intervals"], det_scale=pb.det_scale[sl], step_length=pb.step_length,
            nside=pb.nside, nest=pb.nest, n_pix_submap=pb.n_pix_submap, n_submap=pb.n_submap,
            global2local=pb.global2local, epsilon=obs["epsilon"][sl], gamma=obs["gamma"][sl],
            cal=obs["cal"][sl], shared_flags=pb.shared_flags, shared_flag_mask=1,
            solver_flags=np.ascontiguousarray(pb.solver_flags[sl]), solver_flag_mask=1, nnz=1,
            device=torch.device("cuda", rank))
        dobs.expand_pointing(np.zeros(pb.n_submap, dtype=np.uint8))
        ds = Destriper([dobs], pb.n_local_submap, pb.n_pix_submap, pb.cov, pb.offset_var[asl],
                       pb.amp_flags[asl], device=torch.device("cuda", rank))
        assert ds.peer is None and not ds.pipeline
        rhs = ds.rhs([torch.from_numpy(np.ascontiguousarray(obs["signal"][sl])).cuda()])
        _, hist = ds.solve(rhs, n_iter_max=8)
        rhs_all = [torch.zeros_like(rhs) for _ in range(world)]
        dist.all_gather(rhs_all, rhs)
        if rank == 0:
            out.put((torch.cat(rhs_all).cpu().numpy(), hist))
        dist.barrier()
    except BaseException:
        import sys
        import traceback

        traceback.print_exc()
        sys.stderr.flush()
        os._exit(1)
    finally:
        dist.destroy_process_group()


def test_intensity_two_ranks_nccl_match_single_process_oracle():
    import torch.multiprocessing as mp

    world = 2
    _need(world)
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_nccl_worker, args=(r, world, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    rhs, hist = _collect(procs, out, 180)
    obs = S.make_observation("c4", n_det=6, n_samp=24000, nside=64, eps_max=0.03)
    pb = IP.build_problem(obs, O, nnz=1)
    rhs_ref = IP.solver_rhs(pb, O, obs["signal"])
    assert_close_norm(rhs, rhs_ref, what="RHS (2 ranks)")
    _, hist_ref = IP.solve(pb, O, rhs_ref, n_iter_max=8)
    H.assert_history_matches(hist, hist_ref, _envelope(pb, rhs_ref, 8), what="2-rank NCCL")
