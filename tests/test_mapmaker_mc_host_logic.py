"""MapMaker(mc_mode=True) in the CPU suite: repeated realisations on one Data reuse the set-up of
the first call (tests/fake_device.py stands in for the device; it reads the solver flags and the
destriper's covariance live, so a realisation solved on the wrong flags or covariance gives
wrong products).  Every product of a later realisation must be, bit for bit, what a fresh
mc_mode=False call on a fresh Data gives for the same timestream, and the set-up stages must
not run again."""

import os

import numpy as np
import pytest
import torch.multiprocessing as mp

import fake_device
import fake_device_intensity as FI
import helpers as H
from helpers import O, S
from test_distributed_gloo import _free_port, _shard
from test_intensity_host_logic import _WcsIntensityObservation
from test_mapmaker_host_logic import _split_observation
from test_mapmaker_wcs_host_logic import FOV
from toast_b200 import ops
from toast_b200.data import Data, NoiseModel, observation_from_synthetic
from toast_b200.templates import Offset


def _signal(obs, seed):
    """A new realisation of the timestream of ``obs``: its signal plus seeded per-detector
    offsets and white noise."""
    rng = np.random.default_rng(seed)
    n_det, n_samp = obs["signal"].shape
    return obs["signal"] + rng.normal(size=(n_det, 1)) + 0.3 * rng.normal(size=(n_det, n_samp))


def _with_prior(ob, obs):
    from oracle import offset_prior as OP

    dets = ob.local_detectors
    psdfreq, psds = OP.analytic_psd(obs["sigma"], obs["rate"], fknee=0.05, fmin=1e-4, alpha=1.5,
                                    n_freq=300)
    ob["noise_model"] = NoiseModel({d: float(w) for d, w in zip(dets, obs["detweight"])},
                                   {d: psdfreq for d in dets},
                                   {d: psds[i] for i, d in enumerate(dets)})


def _data(parts, prior=False):
    data = Data()
    for k, o in enumerate(parts):
        ob = observation_from_synthetic(o, name=f"obs{k}")
        if prior:
            _with_prior(ob, o)
        data.obs.append(ob)
    return data


def _mapper(obs, solve_thr=1.0e-3, map_thr=1.0e-3, prior=False, mode="IQU", pixels="healpix",
            mc_mode=True, iter_max=6):
    dp = ops.PointingDetectorSimple(view="scanning", shared_flags="flags", shared_flag_mask=1)
    if pixels == "healpix":
        pix = ops.PixelsHealpix(detector_pointing=dp, nside=obs["nside"], nest=obs["nest"],
                                create_dist="pixel_dist")
    else:
        pix = ops.PixelsWCS(detector_pointing=dp, create_dist="pixel_dist", projection="CAR",
                            field_of_view=FOV, resolution=(0.5, 0.5), submaps=8)
    wts = ops.StokesWeights(detector_pointing=dp, mode=mode)
    binning = ops.BinMap(pixel_dist="pixel_dist", covariance="cov", pixel_pointing=pix,
                         stokes_weights=wts, noise_model="noise_model", full_pointing=True)
    tmpl = Offset(name="baselines", step_time=obs["step_time"], times="times",
                  noise_model="noise_model", use_noise_prior=prior, precond_width=20)
    tmat = ops.TemplateMatrix(templates=[tmpl], amplitudes="amplitudes")
    return ops.MapMaker(name="mm", det_data="signal", binning=binning, template_matrix=tmat,
                        solve_rcond_threshold=solve_thr, map_rcond_threshold=map_thr,
                        iter_max=iter_max, iter_min=iter_max, convergence=1.0e-30, device="cpu",
                        mc_mode=mc_mode)


def _apply(mapper, data, signals):
    for ob, s in zip(data.obs, signals):
        ob.detdata["signal"].data[:] = s
    mapper.apply(data)
    amps = data["amplitudes"]["baselines"]
    return dict(binmap=data["mm_binmap"].data.copy(), map=data["mm_map"].data.copy(),
                amps=amps.local.copy(), amp_flags=amps.local_flags.copy(),
                history=list(mapper.history),
                tod=[ob.detdata["signal"].data.copy() for ob in data.obs],
                hits=data["mm_hits"], cov=data["mm_cov"], rcond=data["mm_rcond"])


def _fresh(parts, signals, prior=False, **kw):
    """The products of a fresh mc_mode=False call on a fresh Data."""
    data = _data(parts, prior)
    return _apply(_mapper(parts[0], prior=prior, mc_mode=False, **kw), data, signals)


def _assert_same(got, ref):
    for key in ("binmap", "map", "amps", "amp_flags"):
        np.testing.assert_array_equal(got[key], ref[key], err_msg=key)
    assert got["history"] == ref["history"]
    for a, b in zip(got["tod"], ref["tod"]):
        np.testing.assert_array_equal(a, b, err_msg="cleaned timestream")
    for key in ("hits", "cov", "rcond"):
        np.testing.assert_array_equal(got[key].data, ref[key].data, err_msg=key)


def _parts(case):
    if case == "prior":
        return [S.make_observation("c1", n_det=4, n_samp=6000, nside=16, eps_max=0.03,
                                   flags=False)]
    obs = S.make_observation("c2", n_det=6, n_samp=12000, nside=64, eps_max=0.03)
    if case == "two_obs":
        return list(_split_observation(obs, 4500))
    return [obs]


# (a stricter map threshold zeroes pixels of the map covariance that the solve uses: a solve on
# the map covariance goes wrong)
_CASES = {"equal": dict(), "looser_map_threshold": dict(map_thr=1.0e-5),
          "stricter_map_threshold": dict(solve_thr=1.0e-5, map_thr=1.0e-3),
          "prior": dict(solve_thr=1.0e-6, map_thr=1.0e-6, prior=True), "two_obs": dict()}


class _Counters:
    """Counts the set-up stages: pointing expansion, covariance accumulation, destriper
    construction, template initialisation, noise-prior construction and the amplitude-flag
    projection."""

    def __init__(self, monkeypatch):
        import toast_b200.ops.mapmaker as MM

        self.n = {}
        for owner, name in ((fake_device.FakeDeviceObservation, "expand_pointing"),
                            (MM.KC, "cov_accum"), (fake_device.FakeDestriper, "__init__"),
                            (Offset, "initialize"), (Offset, "_build_prior"),
                            (MM.KC, "template_offset_project_signal_batch")):
            self._wrap(monkeypatch, owner, name)

    def _wrap(self, monkeypatch, owner, name):
        fn = getattr(owner, name)
        self.n[name] = 0

        def counted(*a, **kw):
            self.n[name] += 1
            return fn(*a, **kw)

        monkeypatch.setattr(owner, name, counted)

    def reset(self):
        for k in self.n:
            self.n[k] = 0

    def all_ran(self, prior=False):
        return all(v > 0 for k, v in self.n.items() if prior or k != "_build_prior")


@pytest.mark.parametrize("case", list(_CASES))
def test_second_realisation_equals_a_fresh_call(monkeypatch, case):
    kw = _CASES[case]
    fake_device.install(monkeypatch, oracle_prior=kw.get("prior", False))
    parts = _parts(case)
    if case.endswith("map_threshold"):
        # the two thresholds mask different pixels: the map covariance is not the solve's
        pb_s = O.build_problem(parts[0], O, rcond_threshold=kw.get("solve_thr", 1.0e-3))
        pb_m = O.build_problem(parts[0], O, rcond_threshold=kw["map_thr"])
        assert (pb_m.rcond > 0).sum() != (pb_s.rcond > 0).sum()
    s1 = [_signal(o, 11 + k) for k, o in enumerate(parts)]
    s2 = [_signal(o, 22 + k) for k, o in enumerate(parts)]
    data = _data(parts, kw.get("prior", False))
    mapper = _mapper(parts[0], **kw)
    first = _apply(mapper, data, s1)
    _assert_same(first, _fresh(parts, s1, **kw))
    second = _apply(mapper, data, s2)
    ref = _fresh(parts, s2, **kw)
    _assert_same(second, ref)
    assert not np.array_equal(second["map"], first["map"])
    # a third realisation on the state the second one left
    s3 = [_signal(o, 33 + k) for k, o in enumerate(parts)]
    _assert_same(_apply(mapper, data, s3), _fresh(parts, s3, **kw))


def test_the_set_up_is_not_repeated(monkeypatch):
    fake_device.install(monkeypatch, oracle_prior=True)
    count = _Counters(monkeypatch)
    parts = _parts("prior")
    data = _data(parts, prior=True)
    mapper = _mapper(parts[0], solve_thr=1.0e-6, map_thr=1.0e-5, prior=True)
    first = _apply(mapper, data, [_signal(parts[0], 1)])
    assert count.all_ran(prior=True), count.n
    count.reset()
    second = _apply(mapper, data, [_signal(parts[0], 2)])
    assert all(v == 0 for v in count.n.values()), count.n
    for key in ("hits", "cov", "rcond"):
        assert second[key] is first[key], key
    _assert_same(second, _fresh(parts, [_signal(parts[0], 2)], solve_thr=1.0e-6, map_thr=1.0e-5,
                                prior=True))


def test_flags_are_part_of_the_set_up(monkeypatch):
    """A realisation with other detector flags is destriped with the first call's flags."""
    fake_device.install(monkeypatch)
    parts = _parts("equal")
    data = _data(parts)
    mapper = _mapper(parts[0])
    _apply(mapper, data, [_signal(parts[0], 1)])
    s2 = [_signal(parts[0], 2)]
    changed = data.obs[0].detdata["flags"].data
    changed[:, ::7] |= 1
    got = _apply(mapper, data, s2)
    _assert_same(got, _fresh(parts, s2))
    # (the change matters: a fresh call with the new flags gives other products)
    moved = dict(parts[0])
    moved["det_flags"] = changed.copy()
    assert not np.array_equal(_fresh([moved], s2)["map"], got["map"])


@pytest.mark.parametrize("change", ["new_data", "solve_rcond_threshold", "mc_mode_off"])
def test_a_changed_set_up_is_rebuilt(monkeypatch, change):
    fake_device.install(monkeypatch)
    count = _Counters(monkeypatch)
    parts = _parts("equal")
    data = _data(parts)
    mapper = _mapper(parts[0])
    _apply(mapper, data, [_signal(parts[0], 1)])
    kw = {}
    if change == "new_data":
        data = _data(parts)
    elif change == "solve_rcond_threshold":
        mapper.solve_rcond_threshold = kw["solve_thr"] = 1.0e-2
    else:
        mapper.mc_mode = False
        _apply(mapper, data, [_signal(parts[0], 5)])
        mapper.mc_mode = True
    count.reset()
    s2 = [_signal(parts[0], 2)]
    got = _apply(mapper, data, s2)
    assert count.all_ran(), count.n
    _assert_same(got, _fresh(parts, s2, **kw))
    # ... and the rebuilt set-up is the one kept
    s3 = [_signal(parts[0], 3)]
    ref = _fresh(parts, s3, **kw)
    count.reset()
    got = _apply(mapper, data, s3)
    assert all(v == 0 for v in count.n.values()), count.n
    _assert_same(got, ref)


def test_mc_mode_off_keeps_nothing(monkeypatch):
    fake_device.install(monkeypatch)
    parts = _parts("equal")
    data = _data(parts)
    mapper = _mapper(parts[0])
    _apply(mapper, data, [_signal(parts[0], 1)])
    assert mapper._mc_state is not None
    mapper.mc_mode = False
    _apply(mapper, data, [_signal(parts[0], 2)])
    assert mapper._mc_state is None


@pytest.mark.parametrize("pixels", ["healpix", "car"])
def test_intensity_realisations(monkeypatch, pixels):
    FI.install_intensity(monkeypatch, _WcsIntensityObservation)
    parts = _parts("equal")
    kw = dict(mode="I", pixels=pixels)
    data = _data(parts)
    mapper = _mapper(parts[0], **kw)
    _apply(mapper, data, [_signal(parts[0], 1)])
    s2 = [_signal(parts[0], 2)]
    got = _apply(mapper, data, s2)
    assert got["map"].shape[-1] == 1
    _assert_same(got, _fresh(parts, s2, **kw))


# ------------------------------------------------------------------------------------------------
# two gloo ranks, detector-sharded (the harness of tests/test_distributed_gloo.py)
# ------------------------------------------------------------------------------------------------
def _mc_worker(rank, world, port, n_det_total, n_samp, out):
    import pytest as _pytest
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ["OMP_NUM_THREADS"] = "1"
    dist.init_process_group("gloo", rank=rank, world_size=world)
    mp_ = _pytest.MonkeyPatch()
    try:
        fake_device.install(mp_)
        n_ds = [0]
        init = fake_device.FakeDestriper.__init__

        def counted(self, *a, **kw):
            n_ds[0] += 1
            init(self, *a, **kw)

        mp_.setattr(fake_device.FakeDestriper, "__init__", counted)
        full = S.make_observation("c1", n_det=n_det_total, n_samp=n_samp, nside=32, eps_max=0.03)
        per = n_det_total // world
        obs = _shard(full, rank * per, per)
        data = _data([obs])
        assert data.comm.world_size == world
        mapper = _mapper(obs, iter_max=4)
        rows = slice(rank * per, (rank + 1) * per)
        _apply(mapper, data, [_signal(full, 1)[rows]])
        got = _apply(mapper, data, [_signal(full, 2)[rows]])
        res = dict(hits=got["hits"].raw.copy(), cov=got["cov"].data.copy(), binmap=got["binmap"],
                   map=got["map"], amps=got["amps"], history=got["history"], n_destriper=n_ds[0])
        gathered = [None] * world
        dist.all_gather_object(gathered, res)
        if rank == 0:
            out.put(gathered)
    finally:
        mp_.undo()
        dist.destroy_process_group()


def test_two_rank_second_realisation_matches_the_single_rank_oracle():
    world, n_det_total, n_samp = 2, 4, 6000
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_mc_worker, args=(r, world, port, n_det_total, n_samp, out))
             for r in range(world)]
    for p in procs:
        p.start()
    ranks = out.get(timeout=300)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0

    full = S.make_observation("c1", n_det=n_det_total, n_samp=n_samp, nside=32, eps_max=0.03)
    s2 = _signal(full, 2)
    pb = O.build_problem(full, O, rcond_threshold=1.0e-3)
    rhs_ref = O.solver_rhs(pb, O, s2)
    amps_ref, hist_ref = O.solve(pb, O, rhs_ref, convergence=1e-30, n_iter_max=4, n_iter_min=4)
    clean = s2.copy()
    O.template_add(pb, O, -amps_ref, clean)
    per = pb.n_amp // world
    for r, got in enumerate(ranks):
        assert got["n_destriper"] == 1   # the second realisation reused the set-up
        H.assert_close_norm(got["cov"], pb.cov, rtol=1e-12, what=f"covariance (rank {r})")
        H.assert_close_norm(got["binmap"], O.bin_map(pb, O, s2, O.cov_apply_diag), rtol=1e-12,
                            what=f"binned map (rank {r})")
        np.testing.assert_allclose(got["history"], hist_ref, rtol=1e-10)
        H.assert_close_norm(got["amps"], amps_ref[r * per:(r + 1) * per],
                            what=f"amplitudes of rank {r}")
        H.assert_close_norm(got["map"], O.bin_map(pb, O, clean, O.cov_apply_diag),
                            what=f"destriped map (rank {r})")
    np.testing.assert_array_equal(ranks[0]["map"], ranks[1]["map"])
    np.testing.assert_array_equal(ranks[0]["hits"], ranks[1]["hits"])
