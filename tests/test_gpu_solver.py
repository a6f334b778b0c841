"""GPU parity tests for the fused destriper passes and the device-resident PCG: against the
oracle's restatement of SolverRHS / SolverLHS / solve() (ops/mapmaker_solve.py) driven by the
compiled reference kernels, and against the committed golden fixtures."""

import numpy as np
import pytest
import torch

import helpers as H
from helpers import O, S, assert_close_norm
from toast_b200 import lib as L
from toast_b200.solver import DeviceObservation, Destriper

pytestmark = pytest.mark.gpu


def _device_problem(obs, pb, regen=False):
    dobs = DeviceObservation(
        focalplane=obs["focalplane"], boresight=obs["boresight"], intervals=obs["intervals"],
        det_scale=pb.det_scale, step_length=pb.step_length, nside=pb.nside, nest=pb.nest,
        n_pix_submap=pb.n_pix_submap, n_submap=pb.n_submap, global2local=pb.global2local,
        epsilon=obs["epsilon"], gamma=obs["gamma"], cal=obs["cal"],
        shared_flags=pb.shared_flags, shared_flag_mask=pb.shared_flag_mask,
        solver_flags=pb.solver_flags, solver_flag_mask=pb.det_flag_mask)
    hits = np.zeros(pb.n_submap, dtype=np.uint8)
    if not regen:
        dobs.expand_pointing(hits)
    ds = Destriper([dobs], pb.n_local_submap, pb.n_pix_submap, pb.cov, pb.offset_var,
                   pb.amp_flags, regen=regen)
    return dobs, ds, hits


# rcond threshold per case: the few-detector satellite slices (c1, c4) see most pixels with one
# polarisation-pair orientation only; at the 1e-3 default 96-98 % of their samples would be cut
# and the passes under test would run on almost nothing.  1e-5 keeps 84-97 % of the samples.
CASES = [("c1", 4, 6000, 64, 1e-5), ("c2", 6, 24000, 64, 1e-3), ("c5", 6, 24000, 64, 1e-3),
         ("c4", 4, 40000, 128, 1e-5)]


@pytest.mark.parametrize("name,n_det,n_samp,nside,rcond", CASES)
@pytest.mark.parametrize("regen", [False, True])
def test_lhs_rhs_and_pcg_history(name, n_det, n_samp, nside, rcond, regen):
    ck = H.checker()
    covapply = getattr(ck, "cov_apply_diag")
    obs = S.make_observation(name, n_det=n_det, n_samp=n_samp, eps_max=0.03, nside=nside)
    pb = O.build_problem(obs, ck, rcond_threshold=rcond)
    assert np.mean((pb.solver_flags & pb.det_flag_mask) == 0) > 0.25  # the passes have work
    dobs, ds, hits = _device_problem(obs, pb, regen)
    if not regen:
        np.testing.assert_array_equal(dobs.pixels.cpu().numpy(), pb.pixels)
        np.testing.assert_array_equal(hits, pb.hit_submaps)
        assert_close_norm(dobs.weights.cpu().numpy(), pb.weights, what="weights")

    # RHS
    rhs_ref = O.solver_rhs(pb, ck, obs["signal"], covapply=covapply)
    sig = torch.from_numpy(obs["signal"]).cuda()
    rhs = ds.rhs([sig])
    assert_close_norm(rhs.cpu().numpy(), rhs_ref, what="RHS")
    binned_ref = O.bin_map(pb, ck, obs["signal"], covapply)
    assert_close_norm(ds.bin_signal([sig]).cpu().numpy(), binned_ref, what="binned map")

    # LHS on a random amplitude vector
    rng = np.random.default_rng(9)
    a = np.where(pb.amp_flags == 0, rng.standard_normal(pb.n_amp), 0.0)
    lhs_ref = O.solver_lhs(pb, ck, a, covapply=covapply)
    q = torch.zeros(pb.n_amp, dtype=torch.float64, device="cuda")
    ds.lhs(torch.from_numpy(a).cuda(), q)
    assert_close_norm(q.cpu().numpy(), lhs_ref, what="LHS")

    # PCG: amplitudes after 3 iterations (before CG amplifies rounding noise) ...
    amps_ref, hist3_ref = O.solve(pb, ck, rhs_ref, n_iter_max=3, covapply=covapply)
    amps, hist3 = ds.solve(torch.from_numpy(rhs_ref).cuda(), n_iter_max=3)
    assert_close_norm(amps.cpu().numpy(), amps_ref, what="amplitudes after 3 iterations")
    # ... and the residual history over 12 iterations
    _, hist_ref = O.solve(pb, ck, rhs_ref, n_iter_max=12, covapply=covapply)
    _, hist = ds.solve(torch.from_numpy(rhs_ref).cuda(), n_iter_max=12)
    H.assert_history_matches(hist, hist_ref, H.pcg_envelope(pb, rhs_ref, 12), what=name)


@pytest.mark.parametrize("fixture", ["c1_tiny", "c2_slice", "c5_slice"])
def test_against_golden_reference_outputs(fixture):
    """Committed outputs of the reference's compiled kernels (tests/golden/make_golden.py)."""
    g = np.load(f"{H.GOLDEN}/{fixture}.npz")
    obs = S.make_observation(str(g["workload"]), n_det=int(g["n_det"]), n_samp=int(g["n_samp"]),
                             eps_max=0.05, nside=int(g["nside"]))
    # the setup stages (flags, covariance, layout) come from the oracle restatement; the
    # pointing, maps, RHS/LHS and PCG under test come from the GPU
    pb = O.build_problem(obs, O)
    dobs, ds, hits = _device_problem(obs, pb, regen=False)
    np.testing.assert_array_equal(dobs.pixels.cpu().numpy(), g["pixels"])
    np.testing.assert_array_equal(hits, g["hit_submaps"])
    assert_close_norm(dobs.weights.cpu().numpy(), g["weights"], what="weights")

    from toast_b200 import kernels as K
    idx = np.arange(pb.n_det, dtype=np.int32)
    zmap = torch.zeros((pb.n_local_submap, pb.n_pix_submap, 3), dtype=torch.float64, device="cuda")
    K.build_noise_weighted(pb.global2local, zmap, idx, dobs.pixels, idx, dobs.weights, idx,
                           torch.from_numpy(obs["signal"]).cuda(), idx,
                           torch.from_numpy(pb.solver_flags).cuda(), pb.det_scale, 1,
                           pb.intervals, torch.from_numpy(pb.shared_flags).cuda(), 1)
    z = zmap.cpu().numpy().reshape(-1, 3)
    zg = np.zeros_like(z)
    zg[g["zmap_index"]] = g["zmap_values"]
    assert_close_norm(z, zg, what="zmap")

    sig = torch.from_numpy(obs["signal"]).cuda()
    assert_close_norm(ds.rhs([sig]).cpu().numpy(), g["rhs"], what="RHS")
    ones = torch.from_numpy(np.where(pb.amp_flags == 0, 1.0, 0.0)).cuda()
    q = torch.zeros_like(ones)
    ds.lhs(ones, q)
    assert_close_norm(q.cpu().numpy(), g["lhs_of_ones"], what="LHS(1)")
    # amplitudes after 2 iterations: before the tiny case reaches its fp64 noise floor, where
    # the (singular) destriping system lets the null-space component drift
    amps2, _ = ds.solve(torch.from_numpy(g["rhs"]).cuda(), n_iter_max=2)
    assert_close_norm(amps2.cpu().numpy(), g["amplitudes_iter2"], what="amplitudes (2 it)")
    _, hist = ds.solve(torch.from_numpy(g["rhs"]).cuda(), n_iter_max=12)
    H.assert_history_matches(hist, g["history"], H.pcg_envelope(pb, g["rhs"], 12), what=fixture)


@pytest.mark.parametrize("fixture", ["c1_wide", "c2_wide", "c4_wide", "c5_wide"])
def test_against_wide_golden_reference_outputs(fixture):
    """The committed reference outputs with thousands of hit pixels
    (tests/golden/make_golden_wide.py): 16-64 detectors, 1282-4564 non-zero map pixels."""
    g = np.load(f"{H.GOLDEN}/{fixture}.npz")
    obs = S.make_observation(str(g["workload"]), n_det=int(g["n_det"]), n_samp=int(g["n_samp"]),
                             eps_max=0.05, nside=int(g["nside"]))
    pb = O.build_problem(obs, O)
    dobs, ds, hits = _device_problem(obs, pb, regen=False)
    np.testing.assert_array_equal(dobs.pixels.cpu().numpy(), g["pixels"].astype(np.int64))
    np.testing.assert_array_equal(hits, g["hit_submaps"])
    ws = int(g["weight_stride"])
    w = dobs.weights.cpu().numpy()
    # the fixture pins the strided weights by digest: the oracle's are those values bit for bit
    H.assert_packed(g, "weights_strided", pb.weights[:, ::ws, :])
    assert_close_norm(w[:, ::ws, :], pb.weights[:, ::ws, :], what="weights")
    assert_close_norm(w.sum(axis=1), g["weights_colsum"], what="weight column sums")

    from toast_b200 import kernels as K
    idx = np.arange(pb.n_det, dtype=np.int32)
    zmap = torch.zeros((pb.n_local_submap, pb.n_pix_submap, 3), dtype=torch.float64, device="cuda")
    K.build_noise_weighted(pb.global2local, zmap, idx, dobs.pixels, idx, dobs.weights, idx,
                           torch.from_numpy(obs["signal"]).cuda(), idx,
                           torch.from_numpy(pb.solver_flags).cuda(), pb.det_scale, 1,
                           pb.intervals, torch.from_numpy(pb.shared_flags).cuda(), 1)
    z = zmap.cpu().numpy().reshape(-1, 3)
    zg = np.zeros_like(z)
    zg[g["zmap_index"]] = g["zmap_values"]
    assert len(g["zmap_index"]) >= 1000
    assert_close_norm(z, zg, what="zmap")
    sig = torch.from_numpy(obs["signal"]).cuda()
    assert_close_norm(ds.rhs([sig]).cpu().numpy(), g["rhs"], what="RHS")
    ones = torch.from_numpy(np.where(pb.amp_flags == 0, 1.0, 0.0)).cuda()
    q = torch.zeros_like(ones)
    ds.lhs(ones, q)
    assert_close_norm(q.cpu().numpy(), g["lhs_of_ones"], what="LHS(1)")
    amps2, _ = ds.solve(torch.from_numpy(g["rhs"]).cuda(), n_iter_max=2)
    assert_close_norm(amps2.cpu().numpy(), g["amplitudes_iter2"], what="amplitudes (2 it)")
    _, hist = ds.solve(torch.from_numpy(g["rhs"]).cuda(), n_iter_max=12)
    H.assert_history_matches(hist, g["history"], H.pcg_envelope(pb, g["rhs"], 12), what=fixture)


@pytest.mark.parametrize("name,n_det,n_samp,nside,rcond", [("c1", 8, 20000, 64, 1e-3),
                                                           ("c2", 16, 24000, 128, 1e-8),
                                                           ("c4", 8, 40000, 128, 1e-8),
                                                           ("c5", 16, 30000, 256, 1e-8)])
def test_pcg_restart_parity_every_iteration(name, n_det, n_samp, nside, rcond):
    """helpers.restart_parity for k = 0 .. 19: the oracle's state before iteration k, ONE device
    iteration, 1e-10 on q, alpha, r.r, x and r -- at the production rcond threshold."""
    ck = H.checker()
    obs = S.make_observation(name, n_det=n_det, n_samp=n_samp, eps_max=0.03, nside=nside)
    pb = O.build_problem(obs, ck, rcond_threshold=rcond)
    assert np.mean((pb.solver_flags & pb.det_flag_mask) == 0) > 0.25
    dobs, ds, _ = _device_problem(obs, pb)
    rhs_ref = O.solver_rhs(pb, ck, obs["signal"], covapply=ck.cov_apply_diag)
    trace = []
    _, hist_ref = O.solve(pb, ck, rhs_ref, n_iter_max=20, covapply=ck.cov_apply_diag, trace=trace)
    # 1e-10, or the reference's own summation-order dependence at this rcond if that is larger
    d0 = trace[0]["d"]
    tol, self_diff = H.order_tolerance(
        trace[0]["q"], O.solver_lhs(pb, ck, d0, covapply=ck.cov_apply_diag, reverse=True),
        rcond=rcond)
    worst = H.restart_parity(ds, pb, trace, rtol=tol, what=name)
    _, hist = ds.solve(torch.from_numpy(rhs_ref).cuda(), n_iter_max=20)
    first, dev = H.first_iteration_over(hist, hist_ref)
    print(f"PARITY_REPORT {name}: restart parity worst {max(worst):.2e} over {len(trace)} "
          f"iterations (bar {tol:.1e}; the reference differs from itself by {self_diff:.1e} when "
          f"it sums the detectors in reverse order); free-running history leaves 1e-10 at "
          f"iteration {first}")


def test_lhs_equals_rhs_of_template_signal():
    """tests/ops_mapmaker_solve.py:150-265: LHS(a) == RHS(F a)."""
    obs = S.make_observation("c1", n_det=4, n_samp=6000, nside=64)
    pb = O.build_problem(obs, O)
    dobs, ds, _ = _device_problem(obs, pb)
    rng = np.random.default_rng(1)
    a = np.where(pb.amp_flags == 0, rng.standard_normal(pb.n_amp), 0.0)
    sig = np.zeros((pb.n_det, pb.n_samp))
    O.template_add(pb, O, a, sig)
    q = torch.zeros(pb.n_amp, dtype=torch.float64, device="cuda")
    ds.lhs(torch.from_numpy(a).cuda(), q)
    r = ds.rhs([torch.from_numpy(sig).cuda()])
    assert_close_norm(q.cpu().numpy(), r.cpu().numpy(), what="LHS(a) vs RHS(Fa)")


def test_destriping_recovers_baselines():
    """End-to-end property at a size the oracle does not need: the solved offsets remove the
    injected random-walk baselines (map-domain residual shrinks by orders of magnitude)."""
    obs = S.make_observation("c1", n_det=4, n_samp=6000, nside=64)
    pb = O.build_problem(obs, O)
    dobs, ds, _ = _device_problem(obs, pb)
    sig = torch.from_numpy(obs["signal"]).cuda()
    rhs = ds.rhs([sig])
    amps, hist = ds.solve(rhs, n_iter_max=50)
    assert hist[-1] < 1e-10
    # residual RHS after subtracting the solved template must vanish: F^T N^-1 Z (d - F a) = 0
    clean = obs["signal"].copy()
    O.template_add(pb, O, -amps.cpu().numpy(), clean)
    r2 = ds.rhs([torch.from_numpy(clean).cuda()])
    assert float(torch.abs(r2).max()) < 1e-6 * float(torch.abs(rhs).max())


def _permuted(obs, perm):
    out = dict(obs)
    for k in ("focalplane", "epsilon", "gamma", "cal", "sigma", "detweight", "signal",
              "det_flags"):
        out[k] = np.ascontiguousarray(obs[k][perm])
    out["n_det"] = len(perm)
    return out


@pytest.mark.parametrize("perm,eps_max", [([0, 2, 1, 3, 4], 0.03), ([0, 1, 2, 3, 4], 0.03),
                                          ([3, 0, 4], 0.03), ([0, 1, 2, 3, 4], 0.0),
                                          ([0, 2, 1, 3, 4], 0.0)])
def test_lhs_path_variants_agree(perm, eps_max):
    """The shipped detector-pair kernels (co-pointed rows share a RED / gather) against the
    oracle and against the block-ordered, crossing-list and general kernels -- including an odd
    detector count and rows whose neighbours do NOT point at the same pixel."""
    ck = H.checker()
    # eps_max = 0: every pair has the same weight rotation (-1, 0) -> the constants of the
    # block-ordered passes are kernel arguments; eps_max > 0: per-pair table
    obs = _permuted(S.make_observation("c4", n_det=6, n_samp=30000, eps_max=eps_max, nside=128),
                    perm)
    pb = O.build_problem(obs, ck, rcond_threshold=1e-5)  # 30-83 % of the samples unflagged
    assert np.mean((pb.solver_flags & pb.det_flag_mask) == 0) > 0.25
    rng = np.random.default_rng(4)
    a = np.where(pb.amp_flags == 0, rng.standard_normal(pb.n_amp), 0.0)
    ref = O.solver_lhs(pb, ck, a, covapply=ck.cov_apply_diag)
    lib = L.load()
    results = {}
    try:
        for name, opts in (("blocked", dict(blocked=1, crossings=1, pair=1, pairw=1)),
                           ("blocked2", dict(blocked=1, crossings=1, pair=1, pairw=1)),
                           ("crossings", dict(blocked=0, crossings=1, pair=1, pairw=1)),
                           ("pairw", dict(blocked=0, crossings=0, pair=1, pairw=1)),
                           ("pair", dict(blocked=0, crossings=0, pair=1, pairw=0)),
                           ("general", dict(blocked=0, crossings=0, pair=0))):
            for k, v in opts.items():
                L.check(lib.tb_set_option(k.encode(), v))
            dobs, ds, _ = _device_problem(obs, pb)
            if name.startswith("blocked"):
                # "blocked": one fused kernel; "blocked2": pass 1 / covariance / pass 2 launches
                assert lib.tb_obs_blocked(dobs.handle().h) == 1
                ds.fuse_lhs = name == "blocked"
            q = torch.zeros(pb.n_amp, dtype=torch.float64, device="cuda")
            ds.lhs(torch.from_numpy(a).cuda(), q)
            results[name] = q.cpu().numpy()
            assert_close_norm(results[name], ref, what=f"LHS ({name})")
            if name == "crossings":
                import ctypes as ct

                n_rec, n_rows, paired = ct.c_int64(0), ct.c_int64(0), ct.c_int(0)
                L.check(lib.tb_obs_crossing_stats(dobs.handle().h, ct.byref(n_rec),
                                                  ct.byref(n_rows), ct.byref(paired)))
                # nside 128 at 50 Hz: dozens of samples per pixel crossing -> the list is built
                assert 0 < n_rec.value < pb.n_det * pb.n_samp // 4
                assert n_rows.value == ((len(perm) + 1) // 2 if paired.value else len(perm))
            if name == "pairw":
                # the shared-weight form is only taken when every pair (2p, 2p+1) is a real
                # polarisation pair (fixed weight rotation, verified sample by sample)
                co_pointed = all(perm[i] // 2 == perm[i + 1] // 2
                                 for i in range(0, len(perm) - 1, 2))
                assert bool(lib.tb_obs_has_pair_weights(dobs.handle().h)) == co_pointed
    finally:
        for k, v in dict(blocked=1, crossings=1, pair=1, pairw=1).items():
            lib.tb_set_option(k.encode(), v)
    for name in ("blocked", "blocked2", "crossings", "pairw", "general"):
        # (pixels with rcond down to 1e-5 amplify the summation-order differences of the variants)
        assert_close_norm(results[name], results["pair"], rtol=1e-11, what=f"{name} vs pair")


def test_block_ordered_pixel_chunks_sum_to_the_whole():
    """tb_bx_pass1 / tb_bx_pass2 chunk by chunk (the units the multi-GPU pipeline overlaps with
    the map reduction): any chunking of the local pixel range on block boundaries gives the
    un-chunked LHS, and flagged amplitudes receive nothing."""
    ck = H.checker()
    obs = S.make_observation("c4", n_det=6, n_samp=30000, eps_max=0.03, nside=128)
    pb = O.build_problem(obs, ck, rcond_threshold=1e-5)
    pb.amp_flags[::7] = 1  # make sure flagged baselines are exercised
    rng = np.random.default_rng(5)
    a = np.where(pb.amp_flags == 0, rng.standard_normal(pb.n_amp), 0.0)
    ref = O.solver_lhs(pb, ck, a, covapply=ck.cov_apply_diag)
    dobs, ds, _ = _device_problem(obs, pb)
    lib = L.load()
    h = dobs.handle().h
    n_pix = pb.n_local_submap * pb.n_pix_submap
    a_d = torch.from_numpy(a).cuda()
    # bounds on block boundaries; pass 1 writes (does not add to) every block of its chunk, so
    # the map starts from garbage
    assert lib.tb_obs_blocked(h) == 1
    bp = int(lib.tb_bx_block_pixels())
    for bounds in ([0, n_pix], [0, bp, 2 * bp, n_pix], list(range(0, n_pix, bp)) + [n_pix],
                   [0, 3 * bp, 3 * bp, n_pix]):
        b = np.array(bounds, dtype=np.int64)
        n_chunks = len(b) - 1
        L.check(lib.tb_obs_set_pixel_chunks(h, n_chunks, L.ptr(b)))
        ds.zmap.fill_(float("nan"))
        for c in range(n_chunks):
            L.check(lib.tb_bx_pass1(h, L.ptr(a_d), L.ptr(ds.amp_flags), L.ptr(ds.zmap), 0, c, None))
        ds.reduce_and_apply_cov()
        q = torch.full((pb.n_amp,), 0.0, dtype=torch.float64, device="cuda")
        for c in reversed(range(n_chunks)):
            L.check(lib.tb_bx_pass2(h, L.ptr(ds.zmap), L.ptr(q), c, None))
        qh = q.cpu().numpy()
        assert_close_norm(qh, ref, what=f"chunked blocked LHS ({n_chunks} chunks)")
        assert np.all(qh[pb.amp_flags != 0] == 0.0)
    with pytest.raises(RuntimeError):
        L.check(lib.tb_bx_pass2(h, L.ptr(ds.zmap), L.ptr(q), n_chunks, None))
    # bounds off the block grid: the chunked block-ordered calls are refused
    b = np.array([0, bp // 2, n_pix], dtype=np.int64)
    L.check(lib.tb_obs_set_pixel_chunks(h, 2, L.ptr(b)))
    with pytest.raises(RuntimeError):
        L.check(lib.tb_bx_pass1(h, L.ptr(a_d), L.ptr(ds.amp_flags), L.ptr(ds.zmap), 0, 0, None))


def test_off_map_samples_run_both_passes_on_the_time_ordered_list():
    """Unflagged samples whose submap is not local have no pixel block: the block-ordered list
    is not built and both passes stay on the time-ordered crossing list (the reference itself
    indexes out of bounds there, ops_scan_map.cpp:44-52, so the checker is the general per-sample
    kernel)."""
    obs = S.make_observation("c4", n_det=4, n_samp=30000, eps_max=0.0, nside=128)
    pb = O.build_problem(obs, O, rcond_threshold=1e-5)
    drop = int(np.flatnonzero(pb.global2local >= 0)[1])
    g2l = pb.global2local.copy()
    g2l[drop] = -1
    keep = g2l >= 0
    g2l[keep] = np.arange(int(keep.sum()))
    cov = np.delete(pb.cov, pb.global2local[drop], axis=0)
    rng = np.random.default_rng(6)
    a = np.where(pb.amp_flags == 0, rng.standard_normal(pb.n_amp), 0.0)
    lib = L.load()
    out = {}
    try:
        for name, opts in (("crossings", dict(crossings=1)),
                           ("general", dict(crossings=0, pair=0))):
            for k, v in opts.items():
                L.check(lib.tb_set_option(k.encode(), v))
            dobs, _, _ = _device_problem(obs, pb)
            dobs.set_global2local(g2l)
            ds = Destriper([dobs], int(keep.sum()), pb.n_pix_submap, cov, pb.offset_var,
                           pb.amp_flags)
            h = dobs.handle().h
            if name == "crossings":
                import ctypes as ct

                assert lib.tb_obs_blocked(h) == 0
                n_rec = ct.c_int64(0)
                L.check(lib.tb_obs_crossing_stats(h, ct.byref(n_rec), None, None))
                assert n_rec.value > 0
                # no block-ordered list: the pixel chunks of the multi-GPU pipeline are refused
                b = np.array([0, ds.zmap.shape[0] * ds.zmap.shape[1]], dtype=np.int64)
                assert lib.tb_obs_set_pixel_chunks(h, 1, L.ptr(b)) != 0
            q = torch.zeros(pb.n_amp, dtype=torch.float64, device="cuda")
            ds.lhs(torch.from_numpy(a).cuda(), q)
            out[name] = q.cpu().numpy()
    finally:
        for k, v in dict(crossings=1, pair=1).items():
            lib.tb_set_option(k.encode(), v)
    assert_close_norm(out["crossings"], out["general"], what="off-map samples")


def test_full_size_properties_c4_shard():
    """BASELINE full size (128 det x 2.16e6 samples, nside 2048: the bench workload), where the
    oracle is too slow to be the checker: size-independent properties instead.
      * hit map total == number of unflagged samples (integer, exact)
      * pixels in range; fused pointing == 3-kernel chain on a detector subset (bit-exact)
      * LHS is linear and symmetric (F^T N^-1 Z F), to 1e-10
      * stored-pointing and regenerated-pointing LHS agree to 1e-10
    """
    from toast_b200 import kernels as K

    n_det, n_samp = 128, 2160000
    obs = S.make_observation("c4", n_det=n_det, n_samp=n_samp, with_signal=False)
    nside, nest = obs["nside"], obs["nest"]
    n_submap, nps = S.n_submap_for(nside, 16)
    dev = torch.device("cuda")
    sflags = torch.from_numpy(obs["shared_flags"]).to(dev)
    solver_flags = torch.from_numpy(obs["det_flags"]).to(dev)
    solver_flags |= sflags[None, :]
    dobs = DeviceObservation(
        focalplane=obs["focalplane"], boresight=obs["boresight"], intervals=obs["intervals"],
        det_scale=obs["detweight"], step_length=obs["step_length"], nside=nside, nest=nest,
        n_pix_submap=nps, n_submap=n_submap, global2local=np.zeros(n_submap, dtype=np.int64),
        epsilon=obs["epsilon"], gamma=obs["gamma"], cal=obs["cal"], shared_flags=sflags,
        shared_flag_mask=1, solver_flags=solver_flags, solver_flag_mask=1)
    hits = np.zeros(n_submap, dtype=np.uint8)
    dobs.expand_pointing(hits)
    pix = dobs.pixels
    assert int(pix.max()) < 12 * nside * nside and int(pix.min()) == -1
    np.testing.assert_array_equal((pix < 0).any(dim=0).cpu().numpy(), obs["shared_flags"] != 0)

    # fused == chain, bit-exact, on 4 detectors
    sub = np.arange(4, dtype=np.int32)
    q = torch.zeros((4, n_samp, 4), dtype=torch.float64, device=dev)
    K.pointing_detector(obs["focalplane"][:4], dobs.boresight, sub, q, obs["intervals"], sflags, 1)
    p2 = torch.zeros((4, n_samp), dtype=torch.int64, device=dev)
    K.pixels_healpix(sub, q, sflags, 1, sub, p2, obs["intervals"],
                     np.zeros(n_submap, dtype=np.uint8), nps, nside, nest)
    assert torch.equal(p2, pix[:4])
    w2 = torch.zeros((4, n_samp, 3), dtype=torch.float64, device=dev)
    K.stokes_weights_IQU(sub, q, sub, w2, None, obs["intervals"], obs["epsilon"][:4],
                         obs["gamma"][:4], obs["cal"][:4], False)
    assert torch.equal(w2, dobs.weights[:4])
    del q, p2, w2

    local = np.flatnonzero(hits).astype(np.int64)
    g2l = np.full(n_submap, -1, dtype=np.int64)
    g2l[local] = np.arange(len(local))
    dobs.set_global2local(g2l)
    n_loc = len(local)
    idx = np.arange(n_det, dtype=np.int32)
    dobs.solver_flags |= (pix < 0).to(torch.uint8)
    hmap = torch.zeros(n_loc * nps, dtype=torch.int64, device=dev)
    inv = torch.zeros((n_loc, nps, 6), dtype=torch.float64, device=dev)
    K.cov_accum(g2l, n_loc, nps, 3, hmap, inv, idx, pix, idx, dobs.weights, idx,
                dobs.solver_flags, obs["detweight"], 1, obs["intervals"], None, 0)
    assert int(hmap.sum()) == int((dobs.solver_flags == 0).sum())   # checksum of the hit map
    rc = torch.zeros(n_loc * nps, dtype=torch.float64, device=dev)
    # rcond >= 1e-3: pixels with condition numbers up to 1e8 (the 1e-8 production threshold)
    # amplify the order-dependent fp64 rounding of the binning to ~1e-10 of the result
    K.cov_invert(n_loc * nps, 3, inv, rc, 1e-3)

    n_amp = dobs.n_amp
    g = torch.Generator(device=dev)
    g.manual_seed(3)
    var = torch.rand(n_amp, generator=g, device=dev, dtype=torch.float64)
    aflags = torch.zeros(n_amp, dtype=torch.uint8, device=dev)
    ds = Destriper([dobs], n_loc, nps, inv, var, aflags)
    a = torch.randn(n_amp, generator=g, device=dev, dtype=torch.float64)
    b = torch.randn(n_amp, generator=g, device=dev, dtype=torch.float64)
    Aa, Ab, Aab = (torch.zeros_like(a) for _ in range(3))
    ds.lhs(a, Aa)
    ds.lhs(b, Ab)
    ds.lhs(2.5 * a - 0.75 * b, Aab)
    lin = 2.5 * Aa - 0.75 * Ab
    e_lin = float((Aab - lin).abs().max() / lin.abs().max())
    assert e_lin < 1e-10, f"linearity {e_lin}"
    ab, ba = float(torch.dot(a, Ab)), float(torch.dot(b, Aa))
    scale = float(torch.sqrt(torch.dot(a, a) * torch.dot(Ab, Ab)))
    assert abs(ab - ba) <= 1e-10 * scale, f"symmetry {ab} {ba} {scale}"
    # regenerated pointing gives the same operator
    ds_r = Destriper([dobs], n_loc, nps, inv, var, aflags, regen=True)
    Ar = torch.zeros_like(a)
    ds_r.lhs(a, Ar)
    e_regen = float((Ar - Aa).abs().max() / Aa.abs().max())
    assert e_regen < 1e-10, f"stored vs regenerated {e_regen}"
