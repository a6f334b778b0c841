"""CPU tests of the host-side logic: synthetic workloads, data model, Offset layout, operator
plumbing and argument validation (no GPU needed; compute entry points must fail loudly)."""

import numpy as np
import pytest

import helpers as H
from helpers import O, S
from toast_b200 import kernels as KC
from toast_b200 import lib as L
from toast_b200.data import Data, DetDataManager, make_intervals, observation_from_synthetic
from toast_b200.pixels import PixelData, PixelDistribution
from toast_b200.templates import Amplitudes, AmplitudesMap


def test_synthetic_workloads_are_deterministic_and_shardable():
    a = S.make_observation("c4", n_det=4, n_samp=5000)
    b = S.make_observation("c4", n_det=4, n_samp=5000)
    for k in ("focalplane", "boresight", "signal", "det_flags", "shared_flags"):
        np.testing.assert_array_equal(a[k], b[k])
    # detector blocks of one focalplane: rank r of a sharded job draws detectors [r*n, (r+1)*n)
    full = S.make_observation("c4", n_det=8, n_samp=100, with_signal=False)
    lo = S.make_observation("c4", n_det=4, n_samp=100, det_first=0, with_signal=False)
    hi = S.make_observation("c4", n_det=4, n_samp=100, det_first=4, with_signal=False)
    np.testing.assert_array_equal(full["focalplane"][:4], lo["focalplane"])
    np.testing.assert_array_equal(full["focalplane"][4:], hi["focalplane"])
    np.testing.assert_array_equal(lo["boresight"], hi["boresight"])
    assert np.allclose(np.linalg.norm(full["boresight"], axis=1), 1.0)
    g = S.make_observation("c2", n_det=2, n_samp=40000, with_signal=False)
    iv = g["intervals"]
    assert len(iv) > 4 and np.all(iv["last"][:-1] <= iv["first"][1:])
    cover = np.sum(iv["last"] - iv["first"]) / 40000
    assert 0.85 < cover < 0.95
    for name, cfg in S.CONFIGS.items():
        n_submap, nps = S.n_submap_for(cfg["nside"])
        assert n_submap * nps == 12 * cfg["nside"] ** 2


def test_offset_layout_and_variance_match_reference_rules():
    iv = make_intervals([(0, 250), (300, 1000)])
    nav, det_start, n_amp = O.offset_layout(3, iv, 100)
    np.testing.assert_array_equal(nav, [3, 7])
    np.testing.assert_array_equal(det_start, [0, 10, 20])
    assert n_amp == 30
    flags = np.zeros((3, 1000), dtype=np.uint8)
    flags[1, 0:60] = 1          # first step of det 1: 40 % good -> flagged
    flags[2, 300:349] = 1       # 51 % good -> kept
    var, fl = O.offset_variance(3, 1000, iv, 100, nav, np.array([2.0, 2.0, 0.0]), flags, 1)
    assert fl[10] == 1 and var[10] == 0.0
    assert fl[0] == 0 and var[0] == 1.0 / (2.0 * 100)
    assert var[2] == 1.0 / (2.0 * 50)           # last, short step of the first view
    assert np.all(fl[20:] == 1)                 # detector with zero noise weight is cut


def test_detdata_ensure_semantics():
    m = DetDataManager(100)
    assert m.ensure("pixels", dtype=np.int64, detectors=["a", "b"]) is False
    assert m["pixels"].data.shape == (2, 100)
    assert m.ensure("pixels", dtype=np.int64, detectors=["b"]) is True   # exists => skip
    with pytest.raises(RuntimeError):
        m.ensure("pixels", dtype=np.int32, detectors=["a"])
    np.testing.assert_array_equal(m["pixels"].indices(["b", "a"]), [1, 0])
    assert m["pixels"].indices(["a"]).dtype == np.int32


def test_pixel_distribution_and_amplitudes():
    dist = PixelDistribution(12 * 64 * 64, 16, [3, 7, 8])
    assert dist.n_pix_submap == 3072
    np.testing.assert_array_equal(dist.global_submap_to_local[[3, 7, 8, 0]], [0, 1, 2, -1])
    sm, lp = dist.global_pixel_to_submap(np.array([3 * 3072 + 5, -1, 8 * 3072]))
    np.testing.assert_array_equal(sm, [0, -1, 2])
    np.testing.assert_array_equal(lp, [5, -1, 0])
    p = PixelData(dist, np.float64, n_value=3)
    assert p.data.shape == (3, 3072, 3) and p.raw.base is not None

    a = Amplitudes(None, 6, 6)
    b = a.duplicate()
    a.local[:] = np.arange(6)
    b.local[:] = 2.0
    a.local_flags[1] = 1
    b.local_flags[:] = a.local_flags
    assert a.dot(b) == 2.0 * (0 + 2 + 3 + 4 + 5)
    m = AmplitudesMap()
    m["x"] = a
    m2 = m.duplicate()
    m2 *= 2.0
    m += m2
    np.testing.assert_array_equal(m["x"].local, 3.0 * np.arange(6))


def test_finished_maps_land_in_the_pixeldata_buffer():
    """MapMaker's products: one copy from the (device) tensor straight into PixelData.data,
    whatever the tensor's shape (flat hit / rcond maps, [n_loc, n_pix_submap, nnz] maps)."""
    import torch

    from toast_b200.ops.mapmaker import _pixdata_from_device

    dist = PixelDistribution(12 * 64 * 64, 16, [3, 7, 8])
    hits = torch.arange(3 * 3072, dtype=torch.int64)
    p = _pixdata_from_device(dist, hits, np.int64, 1)
    assert p.data.shape == (3, 3072, 1) and p.data.dtype == np.int64
    np.testing.assert_array_equal(p.raw, hits.numpy())
    cov = torch.randn((3, 3072, 6), dtype=torch.float64)
    p = _pixdata_from_device(dist, cov, np.float64, 6)
    np.testing.assert_array_equal(p.data, cov.numpy())
    assert p.raw.base is not None and p.distribution is dist


def test_amplitude_flags_and_variance_helpers_match_the_numpy_form():
    """MapMaker forms the Offset amplitude flags / preconditioner (offset.py:283-344) with torch
    element-wise ops on the device; the same functions on CPU tensors must give the bits of the
    numpy form in templates/offset.py, and the layout fill must equal the per-detector loop."""
    import torch

    from toast_b200.ops.mapmaker import _amp_flags_and_variance, _fill_amp_layout

    rng = np.random.default_rng(3)
    nad, n_det = 37, 5
    n = nad * n_det + 25
    lens = np.minimum(50, 1830 - 50 * np.arange(nad)).astype(np.float64)
    scale = rng.uniform(0.5, 2.0, n_det)
    scale[3] = 0.0                                   # a detector with zero weight is cut
    for offs in (7 + nad * np.arange(n_det), np.array([40, 0, 120, 80, 160]) + 3):
        amplen, detnoise = np.zeros(n), np.ones(n)
        for k, o in enumerate(offs):
            amplen[o:o + nad] = lens
            detnoise[o:o + nad] = scale[k]
        a_t, d_t = torch.zeros(n, dtype=torch.float64), torch.ones(n, dtype=torch.float64)
        _fill_amp_layout(a_t, d_t, offs, nad, lens, scale)
        np.testing.assert_array_equal(a_t.numpy(), amplen)
        np.testing.assert_array_equal(d_t.numpy(), detnoise)
        ng = np.floor(rng.uniform(0.0, 1.0, n) * amplen)
        ng[::7] = 0.0
        with np.errstate(divide="ignore", invalid="ignore"):
            keep = (np.where(amplen > 0, ng / amplen, 0.0) > 0.5) & (detnoise > 0)
            var = np.where(keep, 1.0 / (detnoise * ng), 0.0)
        flagged, var_t = _amp_flags_and_variance(torch.from_numpy(ng), a_t, d_t, 0.5)
        np.testing.assert_array_equal(flagged.numpy(), ~keep)
        np.testing.assert_array_equal(var_t.numpy(), var)
        assert keep.any() and (~keep).any() and np.all(np.isfinite(var_t.numpy()))


def test_median_spacing_on_a_torch_device_equals_numpy():
    """The sample spacing behind the Offset step length (utils.py:655-685): the torch form used
    for long time vectors gives numpy's value, for odd and even counts and jittered stamps."""
    import torch

    from toast_b200.templates.offset import median_spacing

    rng = np.random.default_rng(9)
    cpu = torch.device("cpu")
    for n in ((1 << 18) + 1, (1 << 18) + 2, (1 << 18) + 7):
        t = np.arange(n, dtype=np.float64) / 37.0
        for tt in (t, t + rng.normal(0.0, 1e-4, n), np.cumsum(rng.uniform(0.01, 0.03, n))):
            ref = float(np.median(np.diff(tt)))
            assert median_spacing(tt, cpu) == ref
            assert median_spacing(tt) == ref
    assert median_spacing(np.arange(100.0) / 10.0, cpu) == float(np.median(np.diff(np.arange(100.0) / 10.0)))


def test_argument_validation_happens_before_the_device():
    obs = S.make_observation("c1", n_det=4, n_samp=600)
    idx = np.arange(4, dtype=np.int32)
    from toast_b200 import _libtoast as KP

    for K in (KC, KP):
        with pytest.raises(RuntimeError, match="format|dtype"):
            K.pointing_detector(obs["focalplane"], obs["boresight"].astype(np.float32), idx,
                                np.zeros((4, 600, 4)), obs["intervals"], obs["shared_flags"], 1,
                                False)
        with pytest.raises(RuntimeError, match="shape|length"):
            K.pointing_detector(obs["focalplane"], obs["boresight"], idx, np.zeros((4, 599, 4)),
                                obs["intervals"], obs["shared_flags"], 1, False)
        with pytest.raises(RuntimeError):
            K.noise_weight(np.zeros((4, 600))[:, ::2], idx, obs["intervals"], np.ones(4), False)
    if not L.accel_enabled():
        # and with valid arguments the call refuses to compute without a GPU
        with pytest.raises(RuntimeError, match="no usable CUDA device"):
            KP.noise_weight(np.zeros((4, 600)), idx, obs["intervals"], np.ones(4), False)


def test_operator_mirror_has_reference_names_and_traits():
    from toast_b200 import ops, templates

    for name in ("PointingDetectorSimple", "PixelsHealpix", "StokesWeights", "NoiseWeight",
                 "BuildNoiseWeighted", "ScanMap", "BinMap", "MapMaker", "TemplateMatrix",
                 "Pipeline", "BuildHitMap", "BuildInverseCovariance", "CovarianceAndHits"):
        assert hasattr(ops, name)
    assert hasattr(templates, "Offset")
    dp = ops.PointingDetectorSimple(boresight="boresight_radec", shared_flag_mask=3)
    pix = ops.PixelsHealpix(detector_pointing=dp, nside=512, nside_submap=16, nest=False,
                            create_dist="dist")
    assert (pix.nside, pix.nest, dp.shared_flag_mask) == (512, False, 3)
    with pytest.raises(AttributeError):
        ops.PixelsHealpix(no_such_trait=1)
    obs = S.make_observation("c1", n_det=4, n_samp=600)
    data = Data()
    data.obs.append(observation_from_synthetic(obs))
    ob = data.obs[0]
    assert ob.detdata["signal"].data.shape == (4, 600)
    assert ob.select_local_detectors(["D00001"]) == ["D00001"]
    t = templates.Offset(name="b", step_time=10.0, noise_model="noise_model")
    assert t._step_length(10.0, 10.0) == 100
    with pytest.raises(RuntimeError):
        ops.MapMaker(name="mm").apply(data)      # binning / template_matrix traits missing


def test_pointing_detector_fp():
    """ops/pointing_detector_fp.py:82-121 (SURVEY 8f rank 4): every sample of a detector gets its
    focalplane quaternion; existing quats are left alone; ignored traits only warn; the operator
    is host-only (no accelerator support), as in the reference."""
    import warnings

    from toast_b200 import ops

    obs = S.make_observation("c1", n_det=4, n_samp=500, nside=64)
    data = Data()
    ob = observation_from_synthetic(obs)
    data.obs.append(ob)
    op = ops.PointingDetectorFP(quats="quats_fp")
    assert not op.supports_accel()
    assert op.provides() == {"meta": [], "shared": [], "detdata": ["quats_fp"]}
    assert op.requires() == {"meta": [], "shared": [], "detdata": [], "intervals": []}
    dets = ob.local_detectors[1:3]
    op.apply(data, detectors=dets)
    q = ob.detdata["quats_fp"]
    assert q.detectors == dets and q.data.shape == (2, 500, 4)
    for i, d in enumerate(dets):
        np.testing.assert_array_equal(q.data[i], np.tile(obs["focalplane"][i + 1], (500, 1)))
    q.data[:] = 7.0
    op.apply(data, detectors=dets)        # exists for these detectors: skipped
    assert np.all(q.data == 7.0)
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        ops.PointingDetectorFP(quats="q2", boresight="boresight_radec", coord_in="C").apply(data)
    assert len(w) == 2 and "will not use" in str(w[0].message)
    assert ob.detdata["q2"].data.shape == (4, 500, 4)
    with pytest.raises(AttributeError):
        ops.PointingDetectorFP(nside=64)


def test_pipeline_chunk_bounds():
    """The pixel chunks of the multi-GPU pipeline: cover [0, n_pix) without gaps, every inner
    bound aligned to 256 x world pixels (reduction tile x one slice per rank), None when two
    chunks are not possible."""
    import torch  # noqa: F401  (toast_b200.solver imports it)
    from toast_b200.solver import pipeline_chunk_bounds

    for n_sub, world, want in ((4438, 8, 4), (4438, 2, 4), (25, 4, 8), (3, 8, 4), (78, 2, 16)):
        n_pix = n_sub * 3072
        b = pipeline_chunk_bounds(n_pix, world, want)
        assert b is not None and b[0] == 0 and b[-1] == n_pix
        assert np.all(np.diff(b) > 0) and len(b) - 1 <= want
        assert np.all(b[:-1] % (256 * world) == 0)
        assert n_pix % 256 == 0   # so the last chunk is whole reduction tiles too
    assert pipeline_chunk_bounds(3072, 8, 4) is None        # 12 tiles: one unit only
    assert pipeline_chunk_bounds(10 * 3072, 2, 1) is None   # a single chunk requested
    b = pipeline_chunk_bounds(2 * 3072, 4, 100)             # more chunks wanted than units
    assert len(b) - 1 == (2 * 3072) // 1024


def _pcg_on_amplitude_maps(rhs, lhs, precond, convergence, n_iter_max, n_iter_min):
    """The oracle's PCG loop (oracle.toast_oracle._solve, the restatement of the reference's
    solve(), ops/mapmaker_solve.py:524-755) written with nothing but the AmplitudesMap operations
    that solve() uses: duplicate, reset, +=, -=, *= and the masked dot."""
    result = rhs.duplicate()
    result.reset()
    residual = rhs.duplicate()
    residual -= lhs(result)
    precond_residual = residual.duplicate()
    precond_residual.reset()
    precond(residual, precond_residual)
    proposal = precond_residual.duplicate()
    sqsum = rhs.dot(rhs)
    sqsum_init = sqsum_best = last_best = sqsum
    delta = proposal.dot(residual)
    history = []
    for it in range(n_iter_max):
        q = lhs(proposal)
        alpha = delta / proposal.dot(q)
        step = proposal.duplicate()
        step *= alpha
        result += step
        q *= alpha
        residual -= q
        sqsum = residual.dot(residual)
        history.append(sqsum / sqsum_init)
        if history[-1] < convergence or sqsum < 1e-30:
            break
        sqsum_best = min(sqsum, sqsum_best)
        if it % 10 == 0 and it >= n_iter_min:
            if last_best < sqsum_best * 2:
                break
            last_best = sqsum_best
        precond(residual, precond_residual)
        delta_last = delta
        delta = precond_residual.dot(residual)
        proposal *= delta / delta_last
        proposal += precond_residual
    return result, history


def test_product_amplitudes_drive_the_reference_solve():
    """templates.Amplitudes / AmplitudesMap as the amplitude objects of the PCG driver
    (duplicate, reset, +=, -=, *=, masked dot) with the oracle as the LHS operator: amplitudes
    and residual history must be, bit for bit, what the reference's own solve() computed on the
    same problem (tests/golden/solve_reference.npz, make_golden_solve.py) and what the oracle's
    restatement computes.  The c1 problem stops on the convergence test."""
    g = np.load(f"{H.GOLDEN}/solve_reference.npz")
    n_det, n_samp, nside, n_iter = [int(x) for x in g["c1_args"]]
    obs = S.make_observation("c1", n_det=n_det, n_samp=n_samp, nside=nside, eps_max=0.03)
    pb = O.build_problem(obs, O)
    rhs = O.solver_rhs(pb, O, obs["signal"])

    def as_map(values):
        a = Amplitudes(None, pb.n_amp, pb.n_amp)
        a.local[:] = values
        a.local_flags[:] = pb.amp_flags
        return AmplitudesMap(baselines=a)

    def lhs(a_in):
        return as_map(O.solver_lhs(pb, O, a_in["baselines"].local))

    def precond(a_in, a_out):
        O.template_offset_apply_diag_precond(pb.offset_var, a_in["baselines"].local,
                                             a_in["baselines"].local_flags,
                                             a_out["baselines"].local, False)

    result, hist = _pcg_on_amplitude_maps(as_map(rhs), lhs, precond, convergence=1e-12,
                                          n_iter_max=n_iter, n_iter_min=3)
    assert len(hist) < n_iter
    np.testing.assert_array_equal(np.array(hist), g["c1_history"])
    np.testing.assert_array_equal(result["baselines"].local, g["c1_amplitudes"])
    amps_ref, hist_ref = O.solve(pb, O, rhs, convergence=1e-12, n_iter_max=n_iter, n_iter_min=3)
    assert hist == hist_ref
    np.testing.assert_array_equal(result["baselines"].local, amps_ref)
