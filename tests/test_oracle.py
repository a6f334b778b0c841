"""CPU tests of the oracle itself: the C restatement (oracle/toast_oracle.c) against the
reference's compiled kernels (oracle/_ref, when built) and against the committed golden vectors
and known-answer tests of the reference's own test-suite."""

import os

import numpy as np
import pytest

import helpers as H
from helpers import O, S

REF = O.load_ref()

# What the comparisons with the compiled reference below are held to on every machine: their
# outputs as stored by tests/golden/make_golden_oracle_checks.py.  Where oracle/_ref is built, the
# tests compare with it live as well.
CHECKS = os.path.join(H.GOLDEN, "oracle_checks.npz")


def _case(name, n_det, n_samp, **kw):
    return S.make_observation(name, n_det=n_det, n_samp=n_samp, eps_max=0.04, **kw)


def _assert_golden(prefix, arrays):
    g = np.load(CHECKS)
    for key, a in arrays.items():
        H.assert_packed(g, f"{prefix}/{key}", a)


POINTING_CASES = [("c1", 4, 6000), ("c2", 5, 15000), ("c5", 4, 15000), ("c4", 3, 20000)]


def pointing_outputs(K, name, n_det, n_samp):
    obs = _case(name, n_det, n_samp)
    idx = np.arange(n_det, dtype=np.int32)
    iv = obs["intervals"]
    q = np.zeros((n_det, n_samp, 4))
    K.pointing_detector(obs["focalplane"], obs["boresight"], idx, q, iv, obs["shared_flags"],
                        1, False)
    res = {"quats": q}
    for nside, nest in ((obs["nside"], obs["nest"]), (64, not obs["nest"]), (8192, True)):
        n_submap, nps = S.n_submap_for(nside, 16)
        p = np.zeros((n_det, n_samp), dtype=np.int64)
        h = np.zeros(n_submap, dtype=np.uint8)
        K.pixels_healpix(idx, q, obs["shared_flags"], 1, idx, p, iv, h, nps, nside, nest, False)
        res[f"pix_{nside}_{nest}"] = p
        res[f"hit_{nside}_{nest}"] = h
    for hwp in (False, True):
        w = np.zeros((n_det, n_samp, 3))
        ang = (np.arange(n_samp) * 0.01) % 6.0 if hwp else np.zeros(1)
        K.stokes_weights_IQU(idx, q, idx, w, ang, iv, obs["epsilon"], obs["gamma"] + 0.1,
                             obs["cal"], hwp, False)
        res[f"w_{hwp}"] = w
    wi = np.zeros((n_det, n_samp))
    K.stokes_weights_I(idx, wi, iv, obs["cal"], False)
    res["wI"] = wi
    return res


def solver_chain_outputs(K):
    """Problem assembly, RHS, ten PCG iterations and scan_map in all four map dtypes with the
    kernels of ``K`` (the C restatement or the compiled reference)."""
    obs = _case("c2", 6, 20000, nside=64)
    pb = O.build_problem(obs, K)
    covapply = None if K is O else K.cov_apply_diag
    rhs = O.solver_rhs(pb, K, obs["signal"], covapply=covapply)
    a, h = O.solve(pb, K, rhs, n_iter_max=10, covapply=covapply)
    res = dict(pixels=pb.pixels, weights=pb.weights, cov=pb.cov, rhs=rhs, history=np.array(h),
               amplitudes=a)
    idx = np.arange(6, dtype=np.int32)
    for dt in ("float64", "float32", "int64", "int32"):
        m = (np.random.default_rng(1).standard_normal(pb.cov.shape[:2] + (3,)) * 50).astype(dt)
        d = obs["signal"].copy()
        if K is O:
            O.scan_map(pb.global2local, pb.n_pix_submap, m, d, idx, pb.pixels, idx, pb.weights,
                       idx, pb.intervals, 0.5, False, False, True)
        else:
            getattr(K, f"ops_scan_map_{dt}")(pb.global2local, pb.n_pix_submap, m, d, idx,
                                             pb.pixels, idx, pb.weights, idx, pb.intervals, 0.5,
                                             False, False, True, False)
        res[f"scan_{dt}"] = d
    return res


def covariance_outputs(K):
    rng = np.random.default_rng(3)
    nsub, subsize, nnz, n = 3, 50, 3, 4000
    sm = rng.integers(-1, nsub, n).astype(np.int64)
    px = rng.integers(-1, subsize, n).astype(np.int64)
    w = rng.standard_normal(n * nnz)
    accel = () if K is O else (False,)
    h = np.zeros(nsub * subsize, dtype=np.int64)
    K.cov_accum_diag_hits(nsub, subsize, nnz, sm, px, h, *accel)
    c = np.zeros(nsub * subsize * 6)
    K.cov_accum_diag_invnpp(nsub, subsize, nnz, sm, px, w, 1.7, c, *accel)
    v = rng.standard_normal(nsub * subsize * nnz)
    K.cov_apply_diag(nsub, subsize, nnz, c, v)
    return dict(hits=h, invnpp=c, applied=v)


@pytest.mark.parametrize("name,n_det,n_samp", POINTING_CASES)
def test_c_port_is_bit_identical_to_compiled_reference(name, n_det, n_samp):
    out = pointing_outputs(O, name, n_det, n_samp)
    _assert_golden(f"pointing_{name}", out)
    if REF is not None:
        ref = pointing_outputs(REF, name, n_det, n_samp)
        for key in out:
            np.testing.assert_array_equal(out[key], ref[key], err_msg=key)


def test_c_port_solver_chain_matches_reference():
    out = solver_chain_outputs(O)
    _assert_golden("solver_chain", out)
    if REF is not None:
        ref = solver_chain_outputs(REF)
        for key in out:
            np.testing.assert_array_equal(out[key], ref[key], err_msg=key)


def test_c_port_covariance_matches_reference():
    out = covariance_outputs(O)
    _assert_golden("covariance", out)
    if REF is not None:
        ref = covariance_outputs(REF)
        for key in out:
            np.testing.assert_array_equal(out[key], ref[key], err_msg=key)


def _check_cov_inverse(inv, rc, inv_ref, rc_ref, threshold, what):
    """rcond to 1e-12; the same pixels kept (except where rcond sits on the threshold); the
    inverse of a kept pixel within 1e-13 / rcond of the reference's (its conditioning)."""
    near = np.abs(rc_ref - threshold) < 1e-6 * threshold
    np.testing.assert_array_equal((rc > 0)[~near], (rc_ref > 0)[~near], err_msg=what)
    kept = (rc > 0) & (rc_ref > 0)
    assert kept.sum() > 100
    np.testing.assert_allclose(rc[kept], rc_ref[kept], rtol=1e-12, err_msg=what)
    scale = np.max(np.abs(inv_ref), axis=1)
    err = np.max(np.abs(inv - inv_ref), axis=1)
    assert np.all(err[kept] <= 1e-13 / rc_ref[kept] * scale[kept]), what
    dropped = (rc == 0) & (rc_ref == 0)
    assert np.all(inv[dropped] == 0.0) and np.all(inv_ref[dropped] == 0.0)


@pytest.mark.parametrize("thr", ["1e-3", "1e-8"])
def test_cov_eigendecompose_matches_reference_golden(thr):
    """The numpy restatement of cov_eigendecompose_diag against the outputs of the reference's
    own LAPACK-based implementation (tests/golden/make_golden_cov.py)."""
    g = np.load(f"{H.GOLDEN}/cov_invert.npz")
    blocks = g["blocks"]
    d = blocks.reshape(-1).copy()
    rc = np.zeros(len(blocks))
    O.cov_eigendecompose_diag(1, len(blocks), 3, d, rc, float(thr), True)
    _check_cov_inverse(d.reshape(-1, 6), rc, g[f"inverse_{thr}"], g[f"rcond_{thr}"], float(thr),
                       f"golden {thr}")
    d2 = blocks.reshape(-1).copy()
    rc2 = np.zeros(len(blocks))
    O.cov_eigendecompose_diag(1, len(blocks), 3, d2, rc2, 1e-3, False)
    np.testing.assert_array_equal(d2.reshape(-1, 6), blocks)
    np.testing.assert_allclose(rc2, g["rcond_noinvert"], rtol=1e-12, atol=0)


def eigendecompose_outputs(K):
    """cov_eigendecompose_diag of ``K`` on other matrices than the cov_invert.npz fixture's."""
    rng = np.random.default_rng(11)
    npix = 3000
    w = rng.standard_normal((npix, 6, 3))
    w[:, :, 0] = 1.0
    m = np.einsum("pki,pkj->pij", w, w)
    iu = np.triu_indices(3)
    d = np.ascontiguousarray(m[:, iu[0], iu[1]]).reshape(-1)
    r = np.zeros(npix)
    K.cov_eigendecompose_diag(1, npix, 3, d, r, 1e-4, True)
    return d.reshape(-1, 6), r


def test_cov_eigendecompose_matches_compiled_reference():
    """Against the outputs stored in oracle_checks.npz, and live against the reference's
    LAPACK-based inversion when oracle/_ref is built with it (scipy's OpenBLAS through
    oracle/ref_shim/lapack_shim.cpp)."""
    d1, r1 = eigendecompose_outputs(O)
    g = np.load(CHECKS)
    _check_cov_inverse(d1, r1, g["eigendecompose/inverse"], g["eigendecompose/rcond"], 1e-4,
                       "golden")
    if REF is not None:
        try:
            d2, r2 = eigendecompose_outputs(REF)
        except RuntimeError:  # reference built without LAPACK: the stored outputs stand alone
            return
        _check_cov_inverse(d1, r1, d2, r2, 1e-4, "live")


@pytest.mark.parametrize("fixture", ["c1_tiny", "c2_slice", "c5_slice"])
def test_c_port_reproduces_golden_reference_outputs(fixture):
    """Pins the C restatement on machines where /root/reference does not exist."""
    g = np.load(os.path.join(H.GOLDEN, fixture + ".npz"))
    obs = S.make_observation(str(g["workload"]), n_det=int(g["n_det"]), n_samp=int(g["n_samp"]),
                             eps_max=0.05, nside=int(g["nside"]))
    pb = O.build_problem(obs, O)
    np.testing.assert_array_equal(pb.pixels, g["pixels"])
    np.testing.assert_array_equal(pb.weights, g["weights"])
    np.testing.assert_array_equal(pb.hit_submaps, g["hit_submaps"])
    idx = np.arange(pb.n_det, dtype=np.int32)
    zmap = np.zeros((pb.n_local_submap, pb.n_pix_submap, 3))
    O.build_noise_weighted(pb.global2local, zmap, idx, pb.pixels, idx, pb.weights, idx,
                           obs["signal"], idx, pb.solver_flags, pb.det_scale, 1, pb.intervals,
                           pb.shared_flags, 1)
    zg = np.zeros((pb.n_local_submap * pb.n_pix_submap, 3))
    zg[g["zmap_index"]] = g["zmap_values"]
    np.testing.assert_array_equal(zmap.reshape(-1, 3), zg)
    rhs = O.solver_rhs(pb, O, obs["signal"])
    np.testing.assert_array_equal(rhs, g["rhs"])
    ones = np.where(pb.amp_flags == 0, 1.0, 0.0)
    np.testing.assert_array_equal(O.solver_lhs(pb, O, ones), g["lhs_of_ones"])
    amps, hist = O.solve(pb, O, rhs, n_iter_max=12)
    np.testing.assert_array_equal(np.array(hist), g["history"])
    np.testing.assert_array_equal(amps, g["amplitudes"])


@pytest.mark.parametrize("fixture", ["c1_wide", "c2_wide", "c4_wide", "c5_wide"])
def test_c_port_reproduces_wide_golden_reference_outputs(fixture):
    """The fixtures with thousands of hit pixels (tests/golden/make_golden_wide.py)."""
    g = np.load(os.path.join(H.GOLDEN, fixture + ".npz"))
    obs = S.make_observation(str(g["workload"]), n_det=int(g["n_det"]), n_samp=int(g["n_samp"]),
                             eps_max=0.05, nside=int(g["nside"]))
    pb = O.build_problem(obs, O)
    assert len(g["zmap_index"]) >= 1000
    np.testing.assert_array_equal(pb.pixels, g["pixels"].astype(np.int64))
    ws = int(g["weight_stride"])
    H.assert_packed(g, "weights_strided", pb.weights[:, ::ws, :])
    np.testing.assert_array_equal(pb.weights.sum(axis=1), g["weights_colsum"])
    np.testing.assert_array_equal(pb.hit_submaps, g["hit_submaps"])
    idx = np.arange(pb.n_det, dtype=np.int32)
    zmap = np.zeros((pb.n_local_submap, pb.n_pix_submap, 3))
    O.build_noise_weighted(pb.global2local, zmap, idx, pb.pixels, idx, pb.weights, idx,
                           obs["signal"], idx, pb.solver_flags, pb.det_scale, 1, pb.intervals,
                           pb.shared_flags, 1)
    zg = np.zeros((pb.n_local_submap * pb.n_pix_submap, 3))
    zg[g["zmap_index"]] = g["zmap_values"]
    np.testing.assert_array_equal(zmap.reshape(-1, 3), zg)
    rhs = O.solver_rhs(pb, O, obs["signal"])
    np.testing.assert_array_equal(rhs, g["rhs"])
    ones = np.where(pb.amp_flags == 0, 1.0, 0.0)
    np.testing.assert_array_equal(O.solver_lhs(pb, O, ones), g["lhs_of_ones"])
    amps2, _ = O.solve(pb, O, rhs, n_iter_max=2)
    np.testing.assert_array_equal(amps2, g["amplitudes_iter2"])
    _, hist = O.solve(pb, O, rhs, n_iter_max=12)
    np.testing.assert_array_equal(np.array(hist), g["history"])


def test_healpix_primitives_against_golden():
    """tests/healpix.py:95-184 with the compiled reference's outputs as the authority."""
    g = np.load(os.path.join(H.GOLDEN, "healpix_angles.npz"))
    theta, phi = H.healpix_angle_sets()
    for nside in (1, 256, 16384):
        nest = O.healpix_ang2pix(nside, True, theta, phi)
        ring = O.healpix_ang2pix(nside, False, theta, phi)
        np.testing.assert_array_equal(nest, g[f"nest_{nside}"])
        np.testing.assert_array_equal(ring, g[f"ring_{nside}"])
        np.testing.assert_array_equal(O.healpix_ring2nest(nside, ring), g[f"ring2nest_{nside}"])
        np.testing.assert_array_equal(O.healpix_ring2nest(nside, ring), nest)
        np.testing.assert_array_equal(O.healpix_nest2ring(nside, nest), ring)
        assert nest.min() >= 0 and nest.max() < 12 * nside * nside


def test_stokes_weight_known_answers():
    """tests/ops_pointing_healpix.py:98-227: Q/U at psi multiples of 45 deg, with / without HWP."""
    psivec = np.radians([-180, -135, -90, -45, 0, 45, 90, 135, 180])
    expected_Q = np.array([1.0, 0.0, -1.0, 0.0, 1.0, 0.0, -1.0, 0.0, 1.0])
    expected_U = np.array([0.0, 1.0, 0.0, -1.0, 0.0, 1.0, 0.0, -1.0, 0.0])
    n = len(psivec)
    q = np.ascontiguousarray(H.iso_quat(np.full(n, 1.1), np.full(n, 0.7), psivec)).reshape(1, n, 4)
    idx = np.zeros(1, dtype=np.int32)
    iv = S.make_intervals([(0, n)])
    for hwp in (np.zeros(1), np.zeros(n)):
        w = np.zeros((1, n, 3))
        O.stokes_weights_IQU(idx, q, idx, w, hwp, iv, np.zeros(1), np.zeros(1), np.ones(1), False)
        assert np.allclose(w[0, :, 1], expected_Q, atol=1e-12)
        assert np.allclose(w[0, :, 2], expected_U, atol=1e-12)


def test_offset_project_of_add_one():
    """tests/template_offset.py:62-90."""
    iv = S.make_intervals([(0, 400), (450, 1000)])
    nav, det_start, n_amp = O.offset_layout(2, iv, 37)
    amps = np.ones(n_amp)
    fl = np.zeros(n_amp, dtype=np.uint8)
    d = np.zeros((2, 1000))
    out = np.zeros(n_amp)
    for det in range(2):
        O.template_offset_add_to_signal(37, int(det_start[det]), nav, amps, fl, det, d, iv)
        O.template_offset_project_signal(det, d, -1, np.zeros(1, dtype=np.uint8), 0, 37,
                                         int(det_start[det]), nav, out, fl, iv)
    lens = []
    for v in iv:
        ln = int(v["last"] - v["first"])
        lens += [37] * (ln // 37) + ([ln % 37] if ln % 37 else [])
    np.testing.assert_array_equal(out, np.tile(np.array(lens, dtype=np.float64), 2))


def test_lhs_equals_rhs_of_template_signal():
    """tests/ops_mapmaker_solve.py:150-265."""
    obs = _case("c1", 4, 6000)
    pb = O.build_problem(obs, O)
    a = np.where(pb.amp_flags == 0, np.random.default_rng(1).standard_normal(pb.n_amp), 0.0)
    sig = np.zeros((pb.n_det, pb.n_samp))
    O.template_add(pb, O, a, sig)
    np.testing.assert_allclose(O.solver_lhs(pb, O, a), O.solver_rhs(pb, O, sig), rtol=0,
                               atol=1e-12 * np.abs(a).max() * pb.det_scale.max() * 100)


@pytest.mark.parametrize("tag,name", [("c1", "c1"), ("c2", "c2")])
def test_solve_restatement_is_bit_identical_to_reference_solve(tag, name):
    """The oracle's PCG loop against the reference's OWN ``solve()``
    (ops/mapmaker_solve.py:524-755), which tests/golden/make_golden_solve.py executes from the
    reference source with the compiled reference kernels behind its LHS operator: residual
    history (every iteration, including the convergence break of c1) and amplitudes, bit for
    bit."""
    g = np.load(f"{H.GOLDEN}/solve_reference.npz")
    n_det, n_samp, nside, n_iter = [int(x) for x in g[f"{tag}_args"]]
    obs = S.make_observation(name, n_det=n_det, n_samp=n_samp, nside=nside, eps_max=0.03)
    pb = O.build_problem(obs, O)
    rhs = O.solver_rhs(pb, O, obs["signal"])
    np.testing.assert_array_equal(rhs, g[f"{tag}_rhs"])
    amps, hist = O.solve(pb, O, rhs, n_iter_max=n_iter)
    np.testing.assert_array_equal(np.array(hist), g[f"{tag}_history"])
    np.testing.assert_array_equal(amps, g[f"{tag}_amplitudes"])
    if tag == "c1":
        assert len(hist) < n_iter and hist[-1] < 1e-12   # the convergence test fired
