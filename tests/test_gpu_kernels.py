"""GPU parity tests: every CUDA operator kernel, called through the C ABI, against the oracle
(the compiled reference when oracle/_ref is present, else its C restatement) on identical
seeded inputs.  Bars (north_star): pixel indices / hit maps / integer work bit-exact; fp64
results within 1e-10 norm-wise (helpers.RTOL)."""

import numpy as np
import pytest

import helpers as H
from helpers import O, S, assert_close_norm
from toast_b200 import kernels as KC
from toast_b200 import lib as L

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ck():
    return H.checker()


class _PybindFirst:
    """The pybind11 `_libtoast` module (the reference-facing binding) for every function it
    exports; the ctypes twin for the extras (batched / fused entry points)."""

    def __init__(self):
        from toast_b200 import _libtoast

        self._m = _libtoast

    def __getattr__(self, name):
        if hasattr(self._m, name):
            return getattr(self._m, name)
        return getattr(KC, name)


@pytest.fixture(scope="module", params=["ctypes", "pybind"])
def K(request):
    """Both routes into the C ABI: toast_b200.kernels (ctypes) and toast_b200._libtoast
    (pybind11, the module TOAST's kernels.py files import)."""
    return KC if request.param == "ctypes" else _PybindFirst()


def _obs(name, n_det, n_samp, **kw):
    return S.make_observation(name, n_det=n_det, n_samp=n_samp, **kw)


def _quats(obs, ck, use_flags=True):
    n_det, n_samp = obs["n_det"], obs["n_samp"]
    idx = np.arange(n_det, dtype=np.int32)
    q = np.zeros((n_det, n_samp, 4))
    fl = obs["shared_flags"] if use_flags else np.zeros(1, dtype=np.uint8)
    ck.pointing_detector(obs["focalplane"], obs["boresight"], idx, q, obs["intervals"], fl, 1,
                         False)
    return idx, q


CASES = [("c1", 4, 6000), ("c2", 5, 20000), ("c5", 3, 20000), ("c4", 2, 30000)]


@pytest.mark.parametrize("name,n_det,n_samp", CASES)
def test_pointing_detector_bit_exact(K, ck, name, n_det, n_samp):
    obs = _obs(name, n_det, n_samp)
    idx, q_ref = _quats(obs, ck)
    q = np.zeros_like(q_ref)
    K.pointing_detector(obs["focalplane"], obs["boresight"], idx, q, obs["intervals"],
                        obs["shared_flags"], 1, False)
    np.testing.assert_array_equal(q, q_ref)
    # quat_index indirection into a larger buffer, no flags
    big = np.zeros((n_det + 2, n_samp, 4))
    big_ref = np.zeros_like(big)
    ridx = (idx[::-1] + 2).astype(np.int32)
    nofl = np.zeros(1, dtype=np.uint8)
    ck.pointing_detector(obs["focalplane"], obs["boresight"], ridx, big_ref, obs["intervals"],
                         nofl, 0, False)
    K.pointing_detector(obs["focalplane"], obs["boresight"], ridx, big, obs["intervals"], nofl,
                        0, False)
    np.testing.assert_array_equal(big, big_ref)


@pytest.mark.parametrize("name,n_det,n_samp", CASES)
@pytest.mark.parametrize("nest", [True, False])
@pytest.mark.parametrize("nside", [1, 64, 512, 2048, 16384])
def test_pixels_healpix_bit_exact(K, ck, name, n_det, n_samp, nest, nside):
    obs = _obs(name, n_det, n_samp)
    idx, quats = _quats(obs, ck)
    n_submap, nps = S.n_submap_for(nside, 16)
    pix_ref = np.full((n_det, n_samp), -7, dtype=np.int64)
    pix = pix_ref.copy()
    h_ref = np.zeros(n_submap, dtype=np.uint8)
    h = np.zeros(n_submap, dtype=np.uint8)
    ck.pixels_healpix(idx, quats, obs["shared_flags"], 1, idx, pix_ref, obs["intervals"], h_ref,
                      nps, nside, nest, False)
    K.pixels_healpix(idx, quats, obs["shared_flags"], 1, idx, pix, obs["intervals"], h, nps,
                     nside, nest, False)
    np.testing.assert_array_equal(pix, pix_ref)  # includes the untouched -7 outside intervals
    np.testing.assert_array_equal(h, h_ref)
    assert (pix_ref == -1).any()


@pytest.mark.parametrize("nest", [True, False])
def test_pixels_exact_path_agrees(K, ck, nest):
    """Force every sample through the double-double atan2 path: pixels must not change."""
    obs = _obs("c4", 2, 20000)
    idx, quats = _quats(obs, ck)
    nside = 2048
    n_submap, nps = S.n_submap_for(nside, 16)
    pix_ref = np.zeros((2, 20000), dtype=np.int64)
    h_ref = np.zeros(n_submap, dtype=np.uint8)
    ck.pixels_healpix(idx, quats, obs["shared_flags"], 1, idx, pix_ref, obs["intervals"], h_ref,
                      nps, nside, nest, False)
    lib = L.load()
    try:
        for scale, expect_all in ((1.0e20, True), (0.0, False), (1.0, False)):
            lib.tb_set_pixel_guard_scale(scale)
            lib.tb_pixel_exact_count(1)
            pix = np.zeros_like(pix_ref)
            h = np.zeros_like(h_ref)
            K.pixels_healpix(idx, quats, obs["shared_flags"], 1, idx, pix, obs["intervals"], h,
                             nps, nside, nest, False)
            np.testing.assert_array_equal(pix, pix_ref)
            n_exact = lib.tb_pixel_exact_count(1)
            if expect_all:
                assert n_exact == pix.size
            else:
                assert n_exact < 100
    finally:
        lib.tb_set_pixel_guard_scale(1.0)


def test_healpix_reference_angle_sets(K, ck):
    """tests/healpix.py:95-184: eps-perturbed poles / meridians and a regular grid, at nside
    1 / 256 / 16384, NEST and RING -- against the committed reference outputs."""
    gold = np.load(H.GOLDEN + "/healpix_angles.npz")
    theta, phi = H.healpix_angle_sets()
    quats = H.ang_to_quat(theta, phi).reshape(1, -1, 4)
    n = quats.shape[1]
    idx = np.zeros(1, dtype=np.int32)
    iv = S.make_intervals([(0, n)])
    nofl = np.zeros(1, dtype=np.uint8)
    for nside in (1, 256, 16384):
        for nest in (True, False):
            n_submap, nps = S.n_submap_for(nside, 16)
            pix = np.zeros((1, n), dtype=np.int64)
            pix_ref = np.zeros((1, n), dtype=np.int64)
            h = np.zeros(n_submap, dtype=np.uint8)
            K.pixels_healpix(idx, quats, nofl, 0, idx, pix, iv, h, nps, nside, nest, False)
            ck.pixels_healpix(idx, quats, nofl, 0, idx, pix_ref, iv, np.zeros_like(h), nps, nside,
                              nest, False)
            np.testing.assert_array_equal(pix, pix_ref)
            assert pix.min() >= 0 and pix.max() < 12 * nside * nside
            # the quaternion route agrees with the reference's angle route wherever the
            # direction is not within rounding of a pixel edge
            g = gold[("nest_" if nest else "ring_") + str(nside)]
            assert np.mean(pix[0] == g) > 0.97


def test_pointing_matrix_bounds(K, ck):
    """tests/ops_pointing_healpix.py:25-96: phi in {-360..360} deg stays inside the map."""
    nside = 64
    npix = 12 * nside**2
    phivec = np.radians([-360, -270, -180, -135, -90, -45, 0, 45, 90, 135, 180, 270, 360])
    n = len(phivec)
    quats = np.ascontiguousarray(
        H.iso_quat(np.full(n, np.radians(135)), phivec, np.full(n, np.radians(135)))
    ).reshape(1, n, 4)
    idx = np.zeros(1, dtype=np.int32)
    iv = S.make_intervals([(0, n)])
    pix = np.zeros((1, n), dtype=np.int64)
    pix_ref = np.zeros((1, n), dtype=np.int64)
    h = np.zeros(1, dtype=np.uint8)
    K.pixels_healpix(idx, quats, np.zeros(n, dtype=np.uint8), 0, idx, pix, iv, h, npix, nside,
                     True, False)
    ck.pixels_healpix(idx, quats, np.zeros(n, dtype=np.uint8), 0, idx, pix_ref, iv,
                      np.zeros(1, dtype=np.uint8), npix, nside, True, False)
    assert np.all((pix >= 0) & (pix < npix))
    np.testing.assert_array_equal(pix, pix_ref)
    assert h[0] == 1


@pytest.mark.parametrize("hwp", [False, True])
def test_pointing_matrix_weights_analytic(K, hwp):
    """tests/ops_pointing_healpix.py:98-227: Q/U = (+-1, 0) at psi multiples of 45 deg."""
    psivec = np.radians([-180, -135, -90, -45, 0, 45, 90, 135, 180])
    expected_Q = np.array([1.0, 0.0, -1.0, 0.0, 1.0, 0.0, -1.0, 0.0, 1.0])
    expected_U = np.array([0.0, 1.0, 0.0, -1.0, 0.0, 1.0, 0.0, -1.0, 0.0])
    n = len(psivec)
    theta, phi = 1.2345, 0.9876
    quats = np.ascontiguousarray(H.iso_quat(np.full(n, theta), np.full(n, phi), psivec))
    idx = np.zeros(1, dtype=np.int32)
    iv = S.make_intervals([(0, n)])
    w = np.zeros((1, n, 3))
    hwpang = np.zeros(n) if hwp else np.zeros(1)
    K.stokes_weights_IQU(idx, quats.reshape(1, n, 4), idx, w, hwpang, iv, np.zeros(1),
                         np.zeros(1), np.ones(1), False, False)
    assert np.allclose(w[0, :, 0], 1.0)
    assert np.allclose(w[0, :, 1], expected_Q, atol=1e-12)
    assert np.allclose(w[0, :, 2], expected_U, atol=1e-12)


@pytest.mark.parametrize("name,n_det,n_samp", CASES)
@pytest.mark.parametrize("hwp,IAU", [(False, False), (True, False), (False, True), (True, True)])
def test_stokes_weights_IQU(K, ck, name, n_det, n_samp, hwp, IAU):
    obs = _obs(name, n_det, n_samp, eps_max=0.05)
    idx, quats = _quats(obs, ck)
    rng = np.random.default_rng(3)
    hwpang = (np.arange(n_samp) * 0.0123) % (2 * np.pi) if hwp else np.zeros(1)
    gamma = rng.random(n_det) * 0.3
    cal = 1.0 + 0.1 * rng.random(n_det)
    w_ref = np.full((n_det, n_samp, 3), 9.0)
    w = w_ref.copy()
    ck.stokes_weights_IQU(idx, quats, idx, w_ref, hwpang, obs["intervals"], obs["epsilon"],
                          gamma, cal, IAU, False)
    K.stokes_weights_IQU(idx, quats, idx, w, hwpang, obs["intervals"], obs["epsilon"], gamma, cal,
                         IAU, False)
    np.testing.assert_array_equal(w[..., 0], w_ref[..., 0])
    assert_close_norm(w, w_ref, what="stokes IQU")
    # the trig-free evaluation is far inside the bar
    assert np.max(np.abs(w - w_ref)) < 1e-13


def test_stokes_weights_I(K, ck):
    obs = _obs("c2", 4, 9000)
    idx = np.array([3, 1, 0, 2], dtype=np.int32)
    cal = np.array([1.0, 1.5, 0.5, 2.0])
    w_ref = np.zeros((4, 9000))
    w = np.zeros_like(w_ref)
    ck.stokes_weights_I(idx, w_ref, obs["intervals"], cal, False)
    K.stokes_weights_I(idx, w, obs["intervals"], cal, False)
    np.testing.assert_array_equal(w, w_ref)


@pytest.mark.parametrize("name,n_det,n_samp", CASES)
@pytest.mark.parametrize("hwp,IAU", [(False, False), (True, False), (False, True), (True, True)])
def test_pointing_fused_equals_chain(K, ck, name, n_det, n_samp, hwp, IAU):
    obs = _obs(name, n_det, n_samp, eps_max=0.05)
    idx, q_ref = _quats(obs, ck)
    nside, nest = obs["nside"], obs["nest"]
    n_submap, nps = S.n_submap_for(nside, 16)
    # a half-wave plate turning a few times a minute and a per-detector gamma
    hwpang = (2.0 * np.pi * 3.0 / 60.0 / obs["rate"] * np.arange(n_samp)) % (2.0 * np.pi) \
        if hwp else None
    gamma = 0.3 * np.random.default_rng(4).random(n_det) if hwp else obs["gamma"]
    pix_ref = np.zeros((n_det, n_samp), dtype=np.int64)
    h_ref = np.zeros(n_submap, dtype=np.uint8)
    ck.pixels_healpix(idx, q_ref, obs["shared_flags"], 1, idx, pix_ref, obs["intervals"], h_ref,
                      nps, nside, nest, False)
    w_ref = np.zeros((n_det, n_samp, 3))
    ck.stokes_weights_IQU(idx, q_ref, idx, w_ref, np.zeros(1) if hwpang is None else hwpang,
                          obs["intervals"], obs["epsilon"], gamma, obs["cal"], IAU, False)
    q = np.zeros_like(q_ref)
    pix = np.zeros_like(pix_ref)
    w = np.zeros_like(w_ref)
    h = np.zeros_like(h_ref)
    K.pointing_fused(obs["focalplane"], obs["boresight"], obs["shared_flags"], 1, idx, q, idx,
                     pix, idx, w, hwpang, obs["intervals"], h, nps, nside, nest, obs["epsilon"],
                     gamma, obs["cal"], IAU, False)
    np.testing.assert_array_equal(q, q_ref)
    np.testing.assert_array_equal(pix, pix_ref)
    np.testing.assert_array_equal(h, h_ref)
    assert_close_norm(w, w_ref, what="fused weights")


def test_noise_weight_bit_exact(K, ck):
    obs = _obs("c2", 4, 9000)
    idx = np.array([2, 0, 3, 1], dtype=np.int32)
    d_ref = obs["signal"].copy()
    d = obs["signal"].copy()
    ck.noise_weight(d_ref, idx, obs["intervals"], obs["detweight"], False)
    K.noise_weight(d, idx, obs["intervals"], obs["detweight"], False)
    np.testing.assert_array_equal(d, d_ref)


def _pointing(obs, ck):
    pb = O.Problem()
    pb.n_det, pb.n_samp = obs["n_det"], obs["n_samp"]
    pb.nside, pb.nest = obs["nside"], obs["nest"]
    pb.n_submap, pb.n_pix_submap = S.n_submap_for(pb.nside, 16)
    pb.focalplane, pb.boresight, pb.intervals = obs["focalplane"], obs["boresight"], obs["intervals"]
    pb.epsilon, pb.gamma, pb.cal, pb.IAU = obs["epsilon"], obs["gamma"], obs["cal"], False
    pb.hwp = np.zeros(1)
    pb.shared_flags, pb.shared_flag_mask = obs["shared_flags"], 1
    pixels, weights, hits = O.expand_pointing(pb, ck)
    local, g2l = O.pixel_distribution(hits)
    return pixels, weights, hits, local, g2l, pb.n_pix_submap


@pytest.mark.parametrize("name,n_det,n_samp", CASES)
@pytest.mark.parametrize("use_det_flags,use_shared", [(True, True), (False, False), (True, False)])
def test_build_noise_weighted(K, ck, name, n_det, n_samp, use_det_flags, use_shared):
    obs = _obs(name, n_det, n_samp, eps_max=0.03)
    pixels, weights, hits, local, g2l, nps = _pointing(obs, ck)
    idx = np.arange(n_det, dtype=np.int32)
    z_ref = np.zeros((len(local), nps, 3))
    z = np.zeros_like(z_ref)
    df = obs["det_flags"] if use_det_flags else np.zeros((1, 1), dtype=np.uint8)
    sf = obs["shared_flags"] if use_shared else np.zeros(1, dtype=np.uint8)
    args = (idx, pixels, idx, weights, idx, obs["signal"], idx, df, obs["detweight"], 1,
            obs["intervals"], sf, 1, False)
    ck.build_noise_weighted(g2l, z_ref, *args)
    K.build_noise_weighted(g2l, z, *args)
    assert np.count_nonzero(z_ref) > 0
    assert_close_norm(z, z_ref, what="zmap")
    # accumulation: a second call doubles the map
    K.build_noise_weighted(g2l, z, *args)
    assert_close_norm(z, 2 * z_ref, what="zmap accumulate")


@pytest.mark.parametrize("nnz", [1, 2])
def test_build_noise_weighted_other_nnz(K, ck, nnz):
    obs = _obs("c2", 4, 12000)
    pixels, weights3, hits, local, g2l, nps = _pointing(obs, ck)
    idx = np.arange(4, dtype=np.int32)
    weights = np.ascontiguousarray(weights3[..., 0]) if nnz == 1 else np.ascontiguousarray(
        weights3[..., :2])
    z_ref = np.zeros((len(local), nps, nnz))
    z = np.zeros_like(z_ref)
    args = (idx, pixels, idx, weights, idx, obs["signal"], idx, obs["det_flags"],
            obs["detweight"], 1, obs["intervals"], obs["shared_flags"], 1, False)
    ck.build_noise_weighted(g2l, z_ref, *args)
    K.build_noise_weighted(g2l, z, *args)
    assert_close_norm(z, z_ref, what=f"zmap nnz={nnz}")


@pytest.mark.parametrize("dtype", ["float64", "float32", "int64", "int32"])
@pytest.mark.parametrize("mode", ["add", "subtract", "scale", "zero_add"])
def test_scan_map(K, ck, dtype, mode):
    obs = _obs("c2", 4, 12000)
    pixels, weights, hits, local, g2l, nps = _pointing(obs, ck)
    idx = np.arange(4, dtype=np.int32)
    rng = np.random.default_rng(11)
    m = rng.standard_normal((len(local), nps, 3)) * 100.0
    m = m.astype(dtype)
    d_ref = obs["signal"].copy()
    d = obs["signal"].copy()
    flags = dict(add=(False, False, False), subtract=(False, True, False),
                 scale=(False, False, True), zero_add=(True, False, False))[mode]
    args = (idx, pixels, idx, weights, idx, obs["intervals"], 0.75) + flags + (False,)
    H.scan_fn(ck, dtype)(g2l, nps, m, d_ref, *args)
    H.scan_fn(K, dtype)(g2l, nps, m, d, *args)
    np.testing.assert_array_equal(d, d_ref)  # same operations in the same order: bit-exact


def test_scan_map_add_then_subtract_is_zero(K, ck):
    """tests/ops_scan_map.py:99-172."""
    obs = _obs("c1", 4, 6000)
    pixels, weights, hits, local, g2l, nps = _pointing(obs, ck)
    idx = np.arange(4, dtype=np.int32)
    m = np.random.default_rng(2).standard_normal((len(local), nps, 3))
    d = np.zeros((4, 6000))
    K.ops_scan_map_float64(g2l, nps, m, d, idx, pixels, idx, weights, idx, obs["intervals"], 1.0,
                           False, False, False, False)
    assert np.count_nonzero(d) > 0
    K.ops_scan_map_float64(g2l, nps, m, d, idx, pixels, idx, weights, idx, obs["intervals"], 1.0,
                           False, True, False, False)
    assert np.count_nonzero(d) == 0


@pytest.mark.parametrize("name,n_det,n_samp", CASES)
def test_offset_kernels(K, ck, name, n_det, n_samp):
    obs = _obs(name, n_det, n_samp)
    iv = obs["intervals"]
    step = obs["step_length"]
    nav, det_start, n_amp = O.offset_layout(n_det, iv, step)
    rng = np.random.default_rng(5)
    amps = rng.standard_normal(n_amp)
    aflags = (rng.random(n_amp) < 0.1).astype(np.uint8)
    d_ref = obs["signal"].copy()
    d = obs["signal"].copy()
    for det in range(n_det):
        ck.template_offset_add_to_signal(step, int(det_start[det]), nav, amps, aflags, det, d_ref,
                                         iv, False)
        K.template_offset_add_to_signal(step, int(det_start[det]), nav, amps, aflags, det, d, iv,
                                        False)
    np.testing.assert_array_equal(d, d_ref)
    # batched form == per-detector calls
    d2 = obs["signal"].copy()
    K.template_offset_add_to_signal_batch(step, det_start, nav, amps, aflags,
                                          np.arange(n_det, dtype=np.int32), d2, iv, False)
    np.testing.assert_array_equal(d2, d_ref)

    out_ref = np.zeros(n_amp)
    out = np.zeros(n_amp)
    out_nf = np.zeros(n_amp)
    out_nf_ref = np.zeros(n_amp)
    for det in range(n_det):
        ck.template_offset_project_signal(det, d_ref, det, obs["det_flags"], 1, step,
                                          int(det_start[det]), nav, out_ref, aflags, iv, False)
        K.template_offset_project_signal(det, d, det, obs["det_flags"], 1, step,
                                         int(det_start[det]), nav, out, aflags, iv, False)
        ck.template_offset_project_signal(det, d_ref, -1, np.zeros(1, dtype=np.uint8), 1, step,
                                          int(det_start[det]), nav, out_nf_ref, aflags, iv, False)
        K.template_offset_project_signal(det, d, -1, np.zeros(1, dtype=np.uint8), 1, step,
                                         int(det_start[det]), nav, out_nf, aflags, iv, False)
    assert_close_norm(out, out_ref, what="project")
    assert_close_norm(out_nf, out_nf_ref, what="project (no flags)")
    outb = np.zeros(n_amp)
    K.template_offset_project_signal_batch(np.arange(n_det, dtype=np.int32), d,
                                           np.arange(n_det, dtype=np.int32), obs["det_flags"], 1,
                                           step, det_start, nav, outb, aflags, iv, False)
    assert_close_norm(outb, out_ref, what="project batch")

    var = rng.random(n_amp)
    p_ref = np.zeros(n_amp)
    p = np.zeros(n_amp)
    ck.template_offset_apply_diag_precond(var, amps, aflags, p_ref, False)
    K.template_offset_apply_diag_precond(var, amps, aflags, p, False)
    np.testing.assert_array_equal(p, p_ref)


def test_offset_project_of_add_one_is_step_size(K):
    """tests/template_offset.py:26-92: project(add(1)) == number of samples per step."""
    n_samp, step = 1000, 37
    iv = S.make_intervals([(0, 400), (450, 1000)])
    nav, det_start, n_amp = O.offset_layout(1, iv, step)
    amps = np.ones(n_amp)
    aflags = np.zeros(n_amp, dtype=np.uint8)
    d = np.zeros((1, n_samp))
    K.template_offset_add_to_signal(step, 0, nav, amps, aflags, 0, d, iv, False)
    out = np.zeros(n_amp)
    K.template_offset_project_signal(0, d, -1, np.zeros(1, dtype=np.uint8), 0, step, 0, nav, out,
                                     aflags, iv, False)
    expect = []
    for v in iv:
        ln = int(v["last"] - v["first"])
        expect += [step] * (ln // step) + ([ln % step] if ln % step else [])
    np.testing.assert_array_equal(out, np.array(expect, dtype=np.float64))
    assert d[0, 400:450].sum() == 0.0


def test_covariance_kernels(K, ck):
    obs = _obs("c2", 6, 20000, eps_max=0.03)
    pixels, weights, hits, local, g2l, nps = _pointing(obs, ck)
    n_det, n_loc = 6, len(local)
    idx = np.arange(n_det, dtype=np.int32)
    hits_ref = np.zeros(n_loc * nps, dtype=np.int64)
    inv_ref = np.zeros(n_loc * nps * 6)
    for d in range(n_det):
        for iv in obs["intervals"]:
            a, b = int(iv["first"]), int(iv["last"])
            sm, lp = O.global_to_local(pixels[d, a:b], nps, g2l)
            bad = ((obs["det_flags"][d, a:b] & 1) != 0) | ((obs["shared_flags"][a:b] & 1) != 0)
            lp[bad] = -1
            O.cov_accum_diag_hits(n_loc, nps, 3, sm, lp, hits_ref)
            O.cov_accum_diag_invnpp(n_loc, nps, 3, sm, lp,
                                    np.ascontiguousarray(weights[d, a:b]).reshape(-1),
                                    float(obs["detweight"][d]), inv_ref)
    hits_gpu = np.zeros(n_loc * nps, dtype=np.int64)
    inv = np.zeros(n_loc * nps * 6)
    K.cov_accum(g2l, n_loc, nps, 3, hits_gpu, inv, idx, pixels, idx, weights, idx,
                obs["det_flags"], obs["detweight"], 1, obs["intervals"], obs["shared_flags"], 1)
    np.testing.assert_array_equal(hits_gpu, hits_ref)  # hit map: bit-exact
    assert_close_norm(inv, inv_ref, what="inverse covariance")

    # inversion with rcond threshold vs the eigh restatement
    cov_ref = inv_ref.copy()
    rc_ref = np.zeros(n_loc * nps)
    O.cov_eigendecompose_diag(n_loc, nps, 3, cov_ref, rc_ref, 1e-3, True)
    cov = inv_ref.copy()
    rc = np.zeros(n_loc * nps)
    K.cov_invert(n_loc * nps, 3, cov, rc, 1e-3)
    assert (rc_ref > 0).sum() > 100
    np.testing.assert_array_equal(rc > 0, rc_ref > 0)
    # (the kernel's per-pixel code agrees with this restatement to 1e-13 at this threshold when
    # it runs on the host: tests/test_host_math.py)
    assert np.allclose(rc, rc_ref, rtol=1e-10, atol=1e-14)
    assert_close_norm(cov, cov_ref, what="inverse of the pixel covariance")

    # cov_apply
    v_ref = np.random.default_rng(4).standard_normal(n_loc * nps * 3)
    v = v_ref.copy()
    ck_apply = getattr(ck, "cov_apply_diag")
    ck_apply(n_loc, nps, 3, cov_ref, v_ref)
    K.cov_apply_diag(n_loc, nps, 3, cov_ref, v)
    np.testing.assert_array_equal(v, v_ref)


def test_accel_table_round_trip(K, ck):
    """tests/accelerator.py:106-389 (test_memory): create / update / reset / delete, and a kernel
    running on table-resident buffers (`use_accel=True`)."""
    obs = _obs("c1", 4, 6000)
    idx = np.arange(4, dtype=np.int32)
    bore = obs["boresight"]
    quats = np.zeros((4, 6000, 4))
    flags = obs["shared_flags"]
    for buf, nm in ((bore, "boresight"), (quats, "quats"), (flags, "flags")):
        assert not K.accel_present(buf, nm)
        K.accel_create(buf, nm)
        assert K.accel_present(buf, nm)
        K.accel_update_device(buf, nm)
    with pytest.raises(RuntimeError):
        K.accel_create(quats, "quats")  # accelerator.cpp:339-347
    K.pointing_detector(obs["focalplane"], bore, idx, quats, obs["intervals"], flags, 1, True)
    assert np.count_nonzero(quats) == 0  # host copy untouched until update_host
    K.accel_update_host(quats, "quats")
    _, q_ref = _quats(obs, ck)
    np.testing.assert_array_equal(quats, q_ref)
    K.accel_reset(quats, "quats")
    K.accel_update_host(quats, "quats")
    assert np.count_nonzero(quats) == 0
    other = np.zeros((4, 6000, 4))
    with pytest.raises(RuntimeError):  # accelerator.hpp:127-133: not present
        K.pointing_detector(obs["focalplane"], bore, idx, other, obs["intervals"], flags, 1, True)
    for buf, nm in ((bore, "boresight"), (quats, "quats"), (flags, "flags")):
        K.accel_delete(buf, nm)
        assert not K.accel_present(buf, nm)
    with pytest.raises(RuntimeError):
        K.accel_delete(quats, "quats")


def test_argument_validation_raises(K):
    """common.hpp:50-122: wrong dtype / shape raise RuntimeError."""
    obs = _obs("c1", 4, 600)
    idx = np.arange(4, dtype=np.int32)
    with pytest.raises(RuntimeError):
        K.pointing_detector(obs["focalplane"], obs["boresight"].astype(np.float32), idx,
                            np.zeros((4, 600, 4)), obs["intervals"], obs["shared_flags"], 1, False)
    with pytest.raises(RuntimeError):
        K.pointing_detector(obs["focalplane"], obs["boresight"], idx, np.zeros((4, 599, 4)),
                            obs["intervals"], obs["shared_flags"], 1, False)
    with pytest.raises(RuntimeError):  # quat index outside the buffer
        K.pointing_detector(obs["focalplane"], obs["boresight"], idx + 1, np.zeros((4, 600, 4)),
                            obs["intervals"], obs["shared_flags"], 1, False)
    bad_iv = S.make_intervals([(0, 601)])
    with pytest.raises(RuntimeError):
        K.pointing_detector(obs["focalplane"], obs["boresight"], idx, np.zeros((4, 600, 4)),
                            bad_iv, obs["shared_flags"], 1, False)


def test_empty_and_ragged_inputs(K, ck):
    """No intervals => nothing is touched; ragged intervals incl. empty and 1-sample ones."""
    obs = _obs("c1", 4, 600)
    idx = np.arange(4, dtype=np.int32)
    q = np.full((4, 600, 4), 5.0)
    K.pointing_detector(obs["focalplane"], obs["boresight"], idx, q,
                        np.zeros(0, dtype=S.interval_dtype), obs["shared_flags"], 1, False)
    assert np.all(q == 5.0)
    iv = S.make_intervals([(0, 1), (5, 5), (7, 300), (300, 310), (599, 600)])
    q_ref = np.full((4, 600, 4), 5.0)
    ck.pointing_detector(obs["focalplane"], obs["boresight"], idx, q_ref, iv, obs["shared_flags"],
                         1, False)
    K.pointing_detector(obs["focalplane"], obs["boresight"], idx, q, iv, obs["shared_flags"], 1,
                        False)
    np.testing.assert_array_equal(q, q_ref)
    d_ref = obs["signal"].copy()
    d = obs["signal"].copy()
    ck.noise_weight(d_ref, idx, iv, obs["detweight"], False)
    K.noise_weight(d, idx, iv, obs["detweight"], False)
    np.testing.assert_array_equal(d, d_ref)
