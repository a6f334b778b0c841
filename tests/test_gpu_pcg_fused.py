"""The PCG's next direction fused with the prescale of the fused LHS (tb_bx_direction_prescale):
d = s + beta d, the prescaled copy of the new d that tb_bx_fused(amplitudes = NULL) reads, q = 0
and delta_old <- delta_new in one pass must leave exactly what the separate sequence leaves
(tb_pcg_direction, the delta copy, the zero-fill of q and tb_bx_fused with the amplitudes).

The problems are the dyadic ones of test_gpu_blocked.py (paired rows, split blocks, partial last
blocks, an odd detector count) and their intensity forms of test_gpu_intensity.py, plus "apart"
(the partners point apart: one row per detector).  With beta = 1/2 and integer d and s the new d
stays dyadic, so the LHS is exact in any summation order: q identical after both sequences also
proves that the prescaled copies are identical."""

import numpy as np
import pytest
import torch

import test_gpu_blocked as GB
import test_gpu_intensity as GI
from helpers import O
from toast_b200 import lib as L
from toast_b200.solver import Destriper, _PCGState

pytestmark = pytest.mark.gpu

CASES = list(GB.PROBLEMS) + ["apart", "I:split", "I:odd", "I:apart"]


def _device_problem(case, relayout=None):
    nnz1 = case.startswith("I:")
    name = case[2:] if nnz1 else case
    obs = GI._observation(name)
    pb = O.build_problem(obs, O, rcond_threshold=1e-3)
    cov = GB._dyadic_cov(pb)
    if nnz1:
        cov = GI._cov1(cov[..., 0].reshape(-1), pb.n_local_submap, pb.n_pix_submap)
        dobs = GI._device_observation(obs, pb)
    else:
        dobs = GB._device_observation(obs, pb)
    if relayout is not None:
        dobs.amp_offsets = relayout(dobs.amp_offsets)
        dobs.invalidate()
    _, aflags = GB._dyadic_amplitudes(pb)
    ds = Destriper([dobs], pb.n_local_submap, pb.n_pix_submap, cov, pb.offset_var, aflags)
    assert ds._blocked()
    return pb, dobs, ds


@pytest.fixture(scope="module", params=CASES)
def problem(request):
    return _device_problem(request.param)


def _bits(t):
    return t.detach().cpu().numpy().view(np.int64)


def _inputs(pb, seed):
    """Integer d and s in [-8, 8]; flagged entries of both also carry NaN and +-Inf."""
    rng = np.random.default_rng(seed)
    n = pb.n_amp
    d = rng.integers(-8, 9, n).astype(np.float64)
    s = rng.integers(-8, 9, n).astype(np.float64)
    flagged = np.flatnonzero(GB._dyadic_amplitudes(pb)[1])
    d[flagged[0::5]] = np.nan
    d[flagged[1::5]] = np.inf
    s[flagged[2::5]] = -np.inf
    s[flagged[3::5]] = np.nan
    return torch.from_numpy(d).cuda(), torch.from_numpy(s).cuda()


def test_direction_prescale_matches_the_separate_sequence(problem):
    pb, dobs, ds = problem
    lib, h, st = L.load(), dobs.handle().h, torch.cuda.current_stream().cuda_stream
    assert ds._direction_prescale()
    n = pb.n_amp
    d0, s = _inputs(pb, 3)
    fl = ds.amp_flags
    # sums[1] = delta_new; beta = 1/2, then 1 in the second round (delta_old = delta_new)
    sums = torch.tensor([0.0, 3.0], dtype=torch.float64, device="cuda")
    da, delta_a, qa = d0.clone(), torch.tensor([6.0], dtype=torch.float64, device="cuda"), \
        torch.full_like(d0, float("nan"))
    db, delta_b, qb = d0.clone(), delta_a.clone(), torch.full_like(d0, float("nan"))
    for rnd in range(2):
        # the separate sequence
        L.check(lib.tb_pcg_direction(L.ptr(sums[1:]), L.ptr(delta_a), L.ptr(da), L.ptr(s), n, st))
        delta_a.copy_(sums[1:2])
        qa.zero_()
        L.check(lib.tb_bx_fused(h, L.ptr(da), L.ptr(fl), L.ptr(ds.cov), L.ptr(ds.zmap),
                                L.ptr(qa), st))
        # the fused one
        qb.fill_(float("nan"))
        L.check(lib.tb_bx_direction_prescale(h, L.ptr(sums[1:]), L.ptr(delta_b), L.ptr(db),
                                             L.ptr(s), L.ptr(fl), L.ptr(qb), n, st))
        assert int(torch.count_nonzero(qb).item()) == 0 and not bool(torch.signbit(qb).any())
        np.testing.assert_array_equal(_bits(db), _bits(da), err_msg=f"d, round {rnd}")
        np.testing.assert_array_equal(_bits(delta_b), _bits(delta_a), err_msg=f"delta, round {rnd}")
        L.check(lib.tb_bx_fused(h, None, None, L.ptr(ds.cov), L.ptr(ds.zmap), L.ptr(qb), st))
        np.testing.assert_array_equal(_bits(qb), _bits(qa), err_msg=f"q = A d, round {rnd}")
        assert np.all(np.isfinite(qa.cpu().numpy()))


def test_solver_steps_use_the_fused_direction(problem):
    """Destriper.advance_direction takes the fused kernel (one launch fewer per PCG step) and the
    next lhs_and_dot reuses its prescaled d; the solver's vectors are those of the separate
    sequence, which runs when the layout check is switched off."""
    pb, dobs, ds = problem
    lib = L.load()

    def run(fused):
        ds._amps_tiled = fused
        st = _PCGState(pb.n_amp, ds.device)
        d, s = _inputs(pb, 5)
        st.d.copy_(torch.nan_to_num(d, nan=0.0, posinf=0.0, neginf=0.0))
        st.r.copy_(torch.nan_to_num(s, nan=0.0, posinf=0.0, neginf=0.0))
        st.delta.fill_(float(pb.n_amp))
        ds.lhs_and_dot(st)
        torch.cuda.synchronize()
        n0 = lib.tb_launch_count()
        for _ in range(3):
            ds.update(st)
            ds.advance_direction(st)
            ds.lhs_and_dot(st)
        torch.cuda.synchronize()
        return st, lib.tb_launch_count() - n0

    try:
        new, n_new = run(True)
        old, n_old = run(False)
    finally:
        ds._amps_tiled = True
    assert n_old - n_new == 3
    for name in ("x", "r", "s", "d", "q", "dq", "delta", "sums"):
        a, b = getattr(new, name).cpu().numpy(), getattr(old, name).cpu().numpy()
        # (the REDs of the LHS make q differ in the last bits from run to run)
        np.testing.assert_allclose(a, b, rtol=1e-12, atol=1e-12 * np.max(np.abs(b)),
                                   err_msg=name)


def test_a_direction_changed_after_advance_direction_is_not_reused(problem):
    """restart_parity loads d between advance_direction and lhs_and_dot: the LHS must then be
    that of the loaded d, not of the prescaled copy."""
    pb, dobs, ds = problem
    st = _PCGState(pb.n_amp, ds.device)
    d, s = _inputs(pb, 7)
    st.d.copy_(d)
    st.s.copy_(s)
    st.sums[1] = 3.0
    st.delta.fill_(6.0)
    ds.advance_direction(st)
    assert ds._prescaled is not None
    other = torch.from_numpy(np.random.default_rng(8).integers(-8, 9, pb.n_amp).astype(
        np.float64)).cuda()
    st.d.copy_(other)
    ds.lhs_and_dot(st)
    want = torch.full_like(other, float("nan"))
    ds.lhs(other, want)
    np.testing.assert_array_equal(_bits(st.q), _bits(want))


def test_rows_that_do_not_cover_the_amplitudes_are_refused():
    pb, dobs, ds = _device_problem("odd", relayout=lambda off: np.ascontiguousarray(off[::-1]))
    assert not ds._direction_prescale()
    lib, st = L.load(), torch.cuda.current_stream().cuda_stream
    v = lambda: torch.zeros(pb.n_amp, dtype=torch.float64, device="cuda")
    d, s, q, sc = v(), v(), v(), torch.ones(2, dtype=torch.float64, device="cuda")
    args = lambda h, n: (h, L.ptr(sc[1:]), L.ptr(sc[:1]), L.ptr(d), L.ptr(s), L.ptr(ds.amp_flags),
                         L.ptr(q), n, st)
    assert lib.tb_bx_direction_prescale(*args(dobs.handle().h, pb.n_amp)) != 0
    _, dense, _ = _device_problem("odd")
    assert lib.tb_bx_direction_prescale(*args(dense.handle().h, pb.n_amp - 1)) != 0
    assert lib.tb_bx_direction_prescale(*args(dense.handle().h, pb.n_amp)) == 0
