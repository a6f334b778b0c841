"""MapMaker(mc_mode=True) on the device: three realisations in a row on one Data, each later one
against a fresh mc_mode=False call on the same timestream and against the oracle, with the kept
destriper's fused LHS, device memory that does not grow, and two ranks on NCCL."""

import gc
import os

import numpy as np
import pytest
import torch

import helpers as H
import intensity_problem as IP
import wcs_problem as WP
from helpers import O, S, assert_close_norm
from oracle import pixels_wcs as OW
from test_gpu_intensity import _envelope as _envelope_intensity
from test_gpu_peer import _collect, _free_port, _need
from toast_b200 import ops
from toast_b200.data import Data, observation_from_synthetic
from toast_b200.templates import Offset

pytestmark = pytest.mark.gpu

N_ITER = 12

# name: (workload, n_det, n_samp, regenerate_pointing, mode, pixels, solve / map rcond thresholds)
CASES = {
    "c1": ("c1", 4, 6000, False, "IQU", "healpix", 1.0e-3, 1.0e-3),
    "c1_regen": ("c1", 4, 6000, True, "IQU", "healpix", 1.0e-3, 1.0e-3),
    "c2": ("c2", 6, 24000, False, "IQU", "healpix", 1.0e-3, 1.0e-3),
    "c2_regen": ("c2", 6, 24000, True, "IQU", "healpix", 1.0e-3, 1.0e-3),
    "c2_thresholds": ("c2", 6, 24000, False, "IQU", "healpix", 1.0e-3, 1.0e-5),
    "c2_stricter_map": ("c2", 6, 24000, False, "IQU", "healpix", 1.0e-5, 1.0e-3),
    "c2_intensity": ("c2", 8, 12000, False, "I", "healpix", 1.0e-3, 1.0e-3),
    "c2_car": ("c2", 8, 12000, False, "IQU", "car", 1.0e-6, 1.0e-6),
}


def _signal(obs, seed):
    rng = np.random.default_rng(seed)
    n_det, n_samp = obs["signal"].shape
    return obs["signal"] + rng.normal(size=(n_det, 1)) + 0.3 * rng.normal(size=(n_det, n_samp))


def _mapper(case, obs, mc_mode):
    _, _, _, regen, mode, pixels, solve_thr, map_thr = CASES[case]
    dp = ops.PointingDetectorSimple(view="scanning", shared_flags="flags", shared_flag_mask=1)
    if pixels == "healpix":
        pix = ops.PixelsHealpix(detector_pointing=dp, nside=obs["nside"], nest=obs["nest"],
                                create_dist="pixel_dist")
    else:
        pix = ops.PixelsWCS(detector_pointing=dp, create_dist="pixel_dist", projection="CAR",
                            field_of_view=11.0, resolution=(0.5, 0.5), submaps=8)
    wts = ops.StokesWeights(detector_pointing=dp, mode=mode)
    binning = ops.BinMap(pixel_dist="pixel_dist", covariance="cov", pixel_pointing=pix,
                         stokes_weights=wts, noise_model="noise_model", full_pointing=True)
    tmpl = Offset(name="baselines", step_time=obs["step_time"], times="times",
                  noise_model="noise_model")
    tmat = ops.TemplateMatrix(templates=[tmpl], amplitudes="amplitudes")
    return ops.MapMaker(name="mm", det_data="signal", binning=binning, template_matrix=tmat,
                        solve_rcond_threshold=solve_thr, map_rcond_threshold=map_thr,
                        iter_max=N_ITER, convergence=1.0e-30, regenerate_pointing=regen,
                        mc_mode=mc_mode)


def _apply(mapper, data, signal):
    data.obs[0].detdata["signal"].data[:] = signal
    mapper.apply(data)
    return dict(hits=data["mm_hits"], binmap=data["mm_binmap"].data.copy(),
                map=data["mm_map"].data.copy(),
                amps=data["amplitudes"]["baselines"].local.copy(),
                history=list(mapper.history), tod=data.obs[0].detdata["signal"].data.copy())


def _fresh(case, obs, signal):
    data = Data()
    data.obs.append(observation_from_synthetic(obs))
    return _apply(_mapper(case, obs, False), data, signal)


def _clean(pb, signal, amps):
    clean = signal.copy()
    O.template_add(pb, O, -amps, clean)
    return clean


def _oracle(case, obs, pix, signal, ck):
    """(history, amplitudes, reproducibility envelope) of the oracle's solve of ``signal``, and
    the oracle's binned map of ``signal`` cleaned with given amplitudes."""
    _, _, _, _, mode, pixels, solve_thr, _ = CASES[case]
    covapply = ck.cov_apply_diag
    if mode == "I":
        pb = IP.build_problem(obs, ck, nnz=1)
        rhs = IP.solver_rhs(pb, ck, signal, covapply)
        amps, hist = IP.solve(pb, ck, rhs, convergence=1e-30, n_iter_max=N_ITER,
                              covapply=covapply)
        return hist, amps, _envelope_intensity(pb, rhs, N_ITER), \
            lambda a: IP.bin_map(pb, ck, _clean(pb, signal, a), covapply)
    if pixels == "car":
        wo, shape = OW.create_wcs("CAR", bounds_deg=pix.bounds, res_deg=(0.5, 0.5))
        wo.shape = tuple(shape)
        pb = WP.build_wcs_problem(obs, ck, wcs=wo, submaps=8, rcond_threshold=solve_thr)
    else:
        pb = O.build_problem(obs, ck, rcond_threshold=solve_thr)
    rhs = O.solver_rhs(pb, ck, signal, covapply)
    amps, hist = O.solve(pb, ck, rhs, convergence=1e-30, n_iter_max=N_ITER, covapply=covapply)
    return hist, amps, H.pcg_envelope(pb, rhs, N_ITER), \
        lambda a: O.bin_map(pb, ck, _clean(pb, signal, a), covapply)


@pytest.mark.parametrize("case", list(CASES))
def test_realisations_match_fresh_calls(case):
    ck = H.checker()
    name, n_det, n_samp, regen = CASES[case][:4]
    obs = S.make_observation(name, n_det=n_det, n_samp=n_samp, nside=64, eps_max=0.03)
    data = Data()
    data.obs.append(observation_from_synthetic(obs))
    mapper = _mapper(case, obs, True)
    first = _apply(mapper, data, _signal(obs, 1))
    ds = mapper._mc_state.ds
    allocated = []
    for k in (2, 3):
        signal = _signal(obs, k)
        got = _apply(mapper, data, signal)
        assert mapper._mc_state.ds is ds
        torch.cuda.synchronize()
        gc.collect()
        allocated.append(torch.cuda.memory_allocated())
        if k == 2 and not regen:
            # one observation on one GPU: the kept destriper runs the fused LHS on the direction
            # its PCG update prescaled
            assert ds._fused_lhs() and ds._direction_prescale()
        ref = _fresh(case, obs, signal)
        what = f"{case}, realisation {k}"
        assert got["hits"] is first["hits"]
        np.testing.assert_array_equal(got["hits"].raw, ref["hits"].raw)
        assert_close_norm(got["binmap"], ref["binmap"], what=f"binned map ({what})")
        hist_ref, amps_ref, env, bin_clean = _oracle(case, obs, mapper.binning.pixel_pointing,
                                                     signal, ck)
        H.assert_history_matches(got["history"], hist_ref, env, what=what)
        H.assert_history_matches(got["history"], ref["history"], env, what=f"{what} vs fresh")
        bound = max(1e-10, 1e3 * env[-1] ** 0.5)
        dev = np.abs(got["amps"] - amps_ref).max() / np.abs(amps_ref).max()
        assert dev < bound, (what, dev)
        # the destriped map and timestream: 1e-10 against the oracle's cleaning and binning with
        # the realisation's own amplitudes; against the fresh call (whose solve sums in another
        # order: the binning kernels accumulate with atomics) to the level the amplitudes agree
        if CASES[case][6] == CASES[case][7]:   # (the oracle's problem has the solve's threshold)
            assert_close_norm(got["map"], bin_clean(got["amps"]),
                              what=f"destriped map ({what})")
        assert_close_norm(got["map"], ref["map"], rtol=bound, what=f"map vs fresh ({what})")
        assert_close_norm(got["tod"], ref["tod"], rtol=bound, what=f"cleaned TOD ({what})")
        del ref
    # the previous realisation's timestreams and PCG vectors are released
    assert allocated[1] == allocated[0], allocated


# ---- two ranks on the NCCL path ------------------------------------------------------------------
def _mc_worker(rank, world, port, out):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ["OMP_NUM_THREADS"] = "1"
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world,
                            device_id=torch.device("cuda", rank))
    try:
        full = S.make_observation("c1", n_det=4, n_samp=6000, nside=64, eps_max=0.03)
        per = full["n_det"] // world
        sl = slice(rank * per, (rank + 1) * per)
        obs = dict(full)
        obs["n_det"] = per
        for key in ("focalplane", "epsilon", "gamma", "cal", "detweight", "sigma", "det_flags",
                    "signal"):
            obs[key] = np.ascontiguousarray(full[key][sl])
        data = Data()
        data.obs.append(observation_from_synthetic(obs))
        mapper = _mapper("c1", obs, True)
        mapper.device = f"cuda:{rank}"
        _apply(mapper, data, _signal(full, 1)[sl])
        ds = mapper._mc_state.ds
        got = _apply(mapper, data, _signal(full, 2)[sl])
        assert mapper._mc_state.ds is ds
        res = dict(history=got["history"], map=got["map"], amps=got["amps"])
        gathered = [None] * world
        dist.all_gather_object(gathered, res)
        if rank == 0:
            out.put(gathered)
        dist.barrier()
    except BaseException:
        import sys
        import traceback

        traceback.print_exc()
        sys.stderr.flush()
        os._exit(1)
    finally:
        dist.destroy_process_group()


def test_two_ranks_second_realisation_matches_the_oracle():
    import torch.multiprocessing as mp

    world = 2
    _need(world)
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_mc_worker, args=(r, world, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    ranks = _collect(procs, out, 300)
    ck = H.checker()
    full = S.make_observation("c1", n_det=4, n_samp=6000, nside=64, eps_max=0.03)
    s2 = _signal(full, 2)
    pb = O.build_problem(full, ck, rcond_threshold=1.0e-3)
    rhs = O.solver_rhs(pb, ck, s2, ck.cov_apply_diag)
    amps_ref, hist_ref = O.solve(pb, ck, rhs, convergence=1e-30, n_iter_max=N_ITER,
                                 covapply=ck.cov_apply_diag)
    env = H.pcg_envelope(pb, rhs, N_ITER)
    per = pb.n_amp // world
    for r, got in enumerate(ranks):
        H.assert_history_matches(got["history"], hist_ref, env, what=f"rank {r}")
        dev = np.abs(got["amps"] - amps_ref[r * per:(r + 1) * per]).max() / \
            np.abs(amps_ref).max()
        assert dev < max(1e-10, 1e3 * env[-1] ** 0.5), (r, dev)
    assert_close_norm(ranks[0]["map"], ranks[1]["map"], what="maps of the two ranks")
