"""Detector pairs whose weight rotation is not a sign flip.

tb_obs_pack_pointing fits one rotation (A, B) per detector pair, (q1, u1) = (A q0 - B u0,
B q0 + A u0), and from then on streams detector 0's (sum Q, sum U) only: every LHS kernel that
runs on pairs (k_bx, k_lhs_x, k_lhs_pairw) rebuilds detector 1's weights from (A, B).  The
synthetic focal planes are orthogonal pairs, (A, B) = (-1, 0), so the B terms are multiplied by
zero everywhere else in the suite.  Here:

  * part A: stored pointing built by hand, with no trigonometry: rotations (0, +-1), (0.5, 0.5),
    (-0.5, 0.25) and the control (-1, 0), a full symmetric covariance with non-zero off-diagonals,
    power-of-two weights and calibrations, integer amplitudes and timestreams.  Every term is a
    dyadic rational and every partial sum stays below 2^53 grains (asserted on the reference's own
    values), so every LHS path, the RHS and the binned map must equal a plain numpy reference bit
    for bit;
  * part B: real pointing with a half-wave plate, the IAU convention, gamma != 0, epsilon > 0 and
    pairs whose partner is turned by pi/8, pi/4, pi/3 or pi/2 about its line of sight, against the
    oracle at the 1e-10 bar, with stored and regenerated pointing and through ops.MapMaker."""

import ctypes as ct
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import helpers as H
from helpers import O, S, assert_close_norm
from test_gpu_blocked import (BLOCK_PIX, DEFAULT_OPTIONS, VARIANTS, _block_entries, _exact_sum,
                              _flat_view_samples, _local_pixels, _units)
from toast_b200 import lib as L
from toast_b200 import ops
from toast_b200.data import Data, observation_from_synthetic
from toast_b200.solver import DeviceObservation, Destriper
from toast_b200.templates import Offset

pytestmark = pytest.mark.gpu

# ---- part A: hand-built dyadic problems ----------------------------------------------------------
NSIDE, NPS, N_SUBMAP = 16, 192, 16
LOCAL_SUBMAPS = np.array([1, 4, 6, 11, 13])   # 960 local pixels: 7 full blocks and a partial one
N_PIX = len(LOCAL_SUBMAPS) * NPS
STEP = 50
ROTATIONS = ((0.0, 1.0), (0.0, -1.0), (0.5, 0.5), (-0.5, 0.25), (-1.0, 0.0))
# grains: q, u of detector 0 are multiples of 2^-3, the rotations of 2^-2, weights and
# calibrations are at least 2^-1 and the covariance a multiple of 2^-12
GRAIN_Z = 2.0 ** -6      # noise-weighted map: a w (cal, q, u)
GRAIN_M = 2.0 ** -18     # m = C z
GRAIN_OUT = 2.0 ** -24   # amplitudes: w (a - (cal, q, u) . m)

# id: detectors, samples, pair rotation (None: ROTATIONS in turn), share of samples whose partner
# is in another pixel, share of runs in pixel block 0, pair relation broken on one sample
PROBLEMS = {
    # every row has the same {cal0, cal1, A, B}: the kernel-constants form of k_bx
    "uniform": dict(n_det=7, n_samp=20000, rot=(-0.5, 0.25)),
    # rotations and calibrations differ between pairs: the per-row table
    "table": dict(n_det=10, n_samp=20000),
    # partners in other pixels, across the 127 / 128 block boundary too: two-slot records
    "split": dict(n_det=10, n_samp=20000, split=0.05),
    # block 0 holds several work units of kBxUnitMax records
    "contention": dict(n_det=6, n_samp=80000, hot=0.6),
    # one sample of pair 0 off its rotation by one grain: no pair weights, per-detector rows
    "broken": dict(n_det=10, n_samp=20000, broken=True),
}


def _runs(rng, n, hot):
    """Local pixels of n samples in runs of 2..6 samples; a share `hot` of the runs in block 0."""
    lens = rng.integers(2, 7, n // 2 + 1)
    k = len(lens)
    pix = np.where(rng.random(k) < hot, rng.integers(0, BLOCK_PIX, k), rng.integers(0, N_PIX, k))
    return np.repeat(pix, lens)[:n]


def _dyadic_problem(pid):
    cfg = dict(dict(rot=None, split=0.0, hot=0.0, broken=False), **PROBLEMS[pid])
    n_det, n_samp = cfg["n_det"], cfg["n_samp"]
    rng = np.random.default_rng([23, n_det, n_samp])
    a, b = int(0.4 * n_samp), int(0.8 * n_samp)
    intervals = S.make_intervals([(37, a), (a + 113, b), (b + 91, n_samp - 17)])
    in_view = np.zeros(n_samp, dtype=bool)
    for iv in intervals:
        in_view[iv["first"]:iv["last"]] = True
    view_samples = np.flatnonzero(in_view)

    det_scale = rng.choice([0.5, 1.0, 2.0, 4.0], n_det)
    if cfg["rot"] is not None:   # the constants of every row are the same
        cal = np.where(np.arange(n_det) % 2 == 0, 2.0, 0.5)
    else:
        cal = rng.choice([0.5, 1.0, 2.0], n_det)
    lpix = np.empty((n_det, n_samp), dtype=np.int64)
    weights = np.empty((n_det, n_samp, 3))
    rots = []
    for d0 in range(0, n_det, 2):
        p = d0 // 2
        lpix[d0] = _runs(rng, n_samp, cfg["hot"])
        q0 = rng.integers(-8, 9, n_samp).astype(np.float64)
        u0 = rng.integers(-8, 9, n_samp).astype(np.float64)
        q0[(q0 == 0) & (u0 == 0)] = 1.0   # (the rotation is fitted on one sample: never 0)
        q0 *= 0.125
        u0 *= 0.125
        weights[d0] = np.stack([np.full(n_samp, cal[d0]), q0, u0], axis=1)
        if d0 + 1 == n_det:
            continue
        A, B = cfg["rot"] if cfg["rot"] is not None else ROTATIONS[p % len(ROTATIONS)]
        rots.append((A, B))
        lpix[d0 + 1] = lpix[d0]
        if cfg["split"] > 0:
            moved = rng.random(n_samp) < cfg["split"]
            lpix[d0 + 1, moved] = rng.integers(0, N_PIX, int(moved.sum()))
            for k, s in enumerate(rng.choice(view_samples[:-3], 6, replace=False)):
                lpix[d0 + k % 2, s:s + 3] = BLOCK_PIX - 1
                lpix[d0 + 1 - k % 2, s:s + 3] = BLOCK_PIX
        weights[d0 + 1] = np.stack([np.full(n_samp, cal[d0 + 1]), A * q0 - B * u0,
                                    B * q0 + A * u0], axis=1)
    if cfg["broken"]:
        weights[1, view_samples[len(view_samples) // 2], 1] += 2.0 ** -5
    assert np.all(np.mod(weights[..., 1:] / 2.0 ** -5, 1.0) == 0.0)

    flags = S.burst_flags((n_det, n_samp), 0.03, 7, rng)
    flags[:, ~in_view] = 1
    g2l = np.full(N_SUBMAP, -1, dtype=np.int64)
    g2l[LOCAL_SUBMAPS] = np.arange(len(LOCAL_SUBMAPS))
    pixels = LOCAL_SUBMAPS[lpix // NPS] * NPS + lpix % NPS
    pixels[(flags != 0) & (rng.random((n_det, n_samp)) < 0.3)] = -1   # flagged: bad pointing

    n_amp_views = np.array([-(-int(iv["last"] - iv["first"]) // STEP) for iv in intervals])
    n_amp_det = int(n_amp_views.sum())
    n_amp = n_det * n_amp_det
    amps = rng.integers(-8, 9, n_amp).astype(np.float64)
    aflags = np.zeros(n_amp, dtype=np.uint8)
    aflags[::7] = 1
    signal = rng.integers(-16, 17, (n_det, n_samp)).astype(np.float64)

    cov = np.zeros((N_PIX, 6))
    cov[:, [0, 3, 5]] = rng.integers(16, 65, (N_PIX, 3))
    cov[:, [1, 2, 4]] = rng.integers(-8, 9, (N_PIX, 3))
    cov[rng.random(N_PIX) < 0.1] = 0.0   # rejected pixels
    cov *= 2.0 ** -12
    return SimpleNamespace(
        pid=pid, n_det=n_det, n_samp=n_samp, intervals=intervals, step_length=STEP,
        n_amp_views=n_amp_views, n_amp=n_amp, det_start=np.arange(n_det) * n_amp_det,
        det_scale=det_scale, cal=cal, rots=rots, pixels=pixels, weights=weights,
        solver_flags=flags, det_flag_mask=1, n_pix_submap=NPS, global2local=g2l, amps=amps,
        aflags=aflags, signal=signal, cov=cov.reshape(len(LOCAL_SUBMAPS), NPS, 6),
        broken=cfg["broken"])


class QUReference:
    """The LHS, RHS and binned map of problem `p` in plain numpy, sample by sample:
        bin      z[p]   = sum over unflagged samples on p of  t_s w_d (cal_d, q_s, u_s)
        cov      m[p]   = C[p] z[p]
        project  out[b] = sum over unflagged samples of b of  w_d (t_s - (cal_d, q_s, u_s) . m[p])
    with t the template (a_b, 0 on flagged baselines) or the timestream, out = 0 on flagged
    baselines.  Every sum goes through _exact_sum."""

    def __init__(self, p):
        self.p = p
        idx, rel = _flat_view_samples(p)
        lpix = _local_pixels(p, p.global2local)[:, idx]
        good = lpix >= 0
        det = np.broadcast_to(np.arange(p.n_det)[:, None], lpix.shape)[good]
        self.s = np.broadcast_to(idx[None, :], lpix.shape)[good]
        self.det, self.lp = det, lpix[good]
        self.amp = (p.det_start[:, None] + rel[None, :])[good]
        self.w = p.det_scale[det]
        self.wt = p.weights[det, self.s]
        c = p.cov.reshape(-1, 6)
        self.C = c[:, [0, 1, 2, 1, 3, 4, 2, 4, 5]].reshape(-1, 3, 3)

    def template(self, amps):
        return np.where(self.p.aflags[self.amp] == 0, amps[self.amp], 0.0)

    def timestream(self, signal):
        return signal[self.det, self.s]

    def bin(self, t):
        return np.stack([_exact_sum(self.lp, t * self.w * self.wt[:, k], N_PIX, GRAIN_Z)
                         for k in range(3)], axis=1)

    def cov(self, z):
        pix = np.repeat(np.arange(N_PIX), 3)
        return np.stack([_exact_sum(pix, (self.C[:, i, :] * z).reshape(-1), N_PIX, GRAIN_M)
                         for i in range(3)], axis=1)

    def project(self, t, m):
        mp = m[self.lp]
        parts = [self.w * t] + [-self.w * self.wt[:, k] * mp[:, k] for k in range(3)]
        n_amp = self.p.n_amp
        # what any record or run adds up is bounded by the sums of magnitudes of the products
        _exact_sum(np.tile(self.amp, 4), np.concatenate(parts), n_amp, GRAIN_OUT)
        out = _exact_sum(self.amp, parts[0] + parts[1] + parts[2] + parts[3], n_amp, GRAIN_OUT)
        out[self.p.aflags != 0] = 0.0
        return out

    def apply(self, t):
        """(binned map m, amplitudes)"""
        m = self.cov(self.bin(t))
        return m, self.project(t, m)


def _row_constants(p):
    """The per-row {cal0, cal1, A, B} of tb_build_row_table on paired rows (a missing partner takes
    the constants of row 0)."""
    tab = []
    for r in range((p.n_det + 1) // 2):
        if 2 * r + 1 < p.n_det:
            tab.append((p.cal[2 * r], p.cal[2 * r + 1]) + tuple(p.rots[r]))
        else:
            tab.append((p.cal[2 * r],) + tab[0][1:])
    return np.array(tab)


def _hand_built_observation(p):
    unit = np.tile([0.0, 0.0, 0.0, 1.0], (p.n_det, 1))
    return DeviceObservation(
        focalplane=unit, boresight=np.tile([0.0, 0.0, 0.0, 1.0], (p.n_samp, 1)),
        intervals=p.intervals, det_scale=p.det_scale, step_length=p.step_length, nside=NSIDE,
        nest=True, n_pix_submap=NPS, n_submap=N_SUBMAP, global2local=p.global2local, cal=p.cal,
        solver_flags=p.solver_flags, solver_flag_mask=1, pixels=p.pixels, weights=p.weights)


def _destriper(p, dobs):
    return Destriper([dobs], len(LOCAL_SUBMAPS), NPS, p.cov, np.ones(p.n_amp), p.aflags)


def _check_paths(p, dobs):
    """The observation runs on the pair kernels (or, broken, on per-detector rows) and on the
    block-ordered list this problem is built for: record and work-unit counts are the numpy
    model's."""
    lib = L.load()
    h = dobs.handle().h
    expect = 0 if p.broken else 1
    assert lib.tb_obs_has_pair_weights(h) == expect, p.pid
    n_rec, n_rows, paired = ct.c_int64(0), ct.c_int64(0), ct.c_int(0)
    L.check(lib.tb_obs_crossing_stats(h, ct.byref(n_rec), ct.byref(n_rows), ct.byref(paired)))
    assert paired.value == expect
    assert n_rows.value == ((p.n_det + 1) // 2 if expect else p.n_det)
    assert lib.tb_obs_blocked(h) == 1
    n_rec, n_units, n_multi, n_blocks = (ct.c_int64(0) for _ in range(4))
    L.check(lib.tb_obs_blocked_stats(h, ct.byref(n_rec), ct.byref(n_units), ct.byref(n_multi),
                                     ct.byref(n_blocks)))
    entries = _block_entries(p, expect)
    units = _units(entries)
    assert n_blocks.value == len(entries) and N_PIX % BLOCK_PIX != 0 and entries[-1] > 0
    assert (n_rec.value, n_units.value, n_multi.value) == \
        (int(entries.sum()), int(units.sum()), int(units[units > 1].sum())), p.pid
    assert (n_multi.value > 0) == (p.pid == "contention")
    # (no query reports the kernel-constants form: the rows' constants are the same exactly when
    # the problem is built so)
    if not p.broken:
        tab = _row_constants(p)
        assert np.all(tab == tab[0]) == (p.pid == "uniform")
        assert np.any(tab[:, 3] != 0.0)


@pytest.fixture(scope="module", params=list(PROBLEMS))
def dyadic_pair(request):
    p = _dyadic_problem(request.param)
    ref = QUReference(p)
    m, lhs = ref.apply(ref.template(p.amps))
    assert np.count_nonzero(lhs) > p.n_amp // 2
    if p.pid == "split":   # records across the block boundary
        assert np.any((p.pixels[0::2] % NPS == BLOCK_PIX - 1) & (p.pixels[1::2] % NPS == BLOCK_PIX))
    dobs = _hand_built_observation(p)
    _check_paths(p, dobs)
    ds = _destriper(p, dobs)
    assert ds._blocked()
    return SimpleNamespace(p=p, ref=ref, m=m, lhs=lhs, dobs=dobs, ds=ds, h=dobs.handle().h,
                           a_d=torch.from_numpy(p.amps).cuda())


def _lhs(ds, a_d):
    q = torch.full_like(a_d, float("nan"))
    ds.lhs(a_d, q)
    return q.cpu().numpy()


def test_blocked_lhs_is_exact(dyadic_pair):
    """tb_bx_fused, the three-launch form (which leaves m = C z in the map) and pixel-chunked
    pass 1 / pass 2, one chunk per block: bit for bit, twice in a row."""
    d, ds = dyadic_pair, dyadic_pair.ds
    lib = L.load()
    try:
        for fused in (True, False):
            ds.fuse_lhs = fused
            ds.zmap.fill_(float("nan"))
            for rep in range(2):
                np.testing.assert_array_equal(_lhs(ds, d.a_d), d.lhs,
                                              err_msg=f"fused={fused} call {rep}")
            if not fused:
                np.testing.assert_array_equal(ds.zmap.cpu().numpy().reshape(-1, 3), d.m)
    finally:
        ds.fuse_lhs = True
    b = np.array(list(range(0, N_PIX, BLOCK_PIX)) + [N_PIX], dtype=np.int64)
    try:
        L.check(lib.tb_obs_set_pixel_chunks(d.h, len(b) - 1, L.ptr(b)))
        ds.zmap.fill_(float("nan"))
        for c in range(len(b) - 1):
            L.check(lib.tb_bx_pass1(d.h, L.ptr(d.a_d), L.ptr(ds.amp_flags), L.ptr(ds.zmap), 0, c,
                                    None))
        ds.reduce_and_apply_cov()
        np.testing.assert_array_equal(ds.zmap.cpu().numpy().reshape(-1, 3), d.m)
        q = torch.zeros_like(d.a_d)
        for c in reversed(range(len(b) - 1)):
            L.check(lib.tb_bx_pass2(d.h, L.ptr(ds.zmap), L.ptr(q), c, None))
        np.testing.assert_array_equal(q.cpu().numpy(), d.lhs, err_msg="pixel chunks")
    finally:
        whole = np.array([0, N_PIX], dtype=np.int64)
        L.check(lib.tb_obs_set_pixel_chunks(d.h, 1, L.ptr(whole)))


def test_other_lhs_paths_are_exact(dyadic_pair):
    """The time-ordered crossing list (k_lhs_x), the pair kernels (k_lhs_pairw, k_lhs_pair) and
    the per-sample kernels on the same inputs."""
    lib = L.load()
    d = dyadic_pair
    try:
        for name, opts in VARIANTS:
            for k, v in opts.items():
                L.check(lib.tb_set_option(k.encode(), v))
            dobs = _hand_built_observation(d.p)
            ds = _destriper(d.p, dobs)
            assert not ds._blocked()
            if name == "crossings":
                paired = ct.c_int(0)
                L.check(lib.tb_obs_crossing_stats(dobs.handle().h, None, None, ct.byref(paired)))
                assert paired.value == (0 if d.p.broken else 1)
            np.testing.assert_array_equal(_lhs(ds, d.a_d), d.lhs, err_msg=name)
    finally:
        for k, v in DEFAULT_OPTIONS.items():
            lib.tb_set_option(k.encode(), v)


def test_rhs_and_binned_map_are_exact(dyadic_pair):
    d, ds = dyadic_pair, dyadic_pair.ds
    m, rhs = d.ref.apply(d.ref.timestream(d.p.signal))
    sig = torch.from_numpy(d.p.signal).cuda()
    np.testing.assert_array_equal(ds.bin_signal([sig]).cpu().numpy().reshape(-1, 3), m)
    np.testing.assert_array_equal(ds.rhs([sig]).cpu().numpy(), rhs)


# ---- part B: real pointing, HWP, IAU, gamma, rotated partners ------------------------------------
PSI = (np.pi / 8, np.pi / 4, np.pi / 3, np.pi / 2)


def _rotated_observation(n_samp):
    """Four co-pointed pairs: detector 2p + 1 is detector 2p turned by PSI[p] about its line of
    sight, so the pair's weight rotation is rigid; gamma != 0, epsilon > 0, and a half-wave plate
    turning three times a minute."""
    obs = S.make_observation("c2", n_det=2 * len(PSI), n_samp=n_samp, eps_max=0.03, nside=64)
    fp = obs["focalplane"]
    for p, psi in enumerate(PSI):
        fp[2 * p + 1] = S.q_mult(fp[2 * p], S.q_rotation(S.ZAXIS, psi))
    obs["gamma"] = 0.3 * np.random.default_rng(7).random(obs["n_det"])
    hwp = (2.0 * np.pi * (3.0 / 60.0) / obs["rate"] * np.arange(n_samp)) % (2.0 * np.pi)
    return obs, hwp


def _rotated_device_observation(obs, pb, hwp, IAU, expand):
    dobs = DeviceObservation(
        focalplane=obs["focalplane"], boresight=obs["boresight"], intervals=obs["intervals"],
        det_scale=pb.det_scale, step_length=pb.step_length, nside=pb.nside, nest=pb.nest,
        n_pix_submap=pb.n_pix_submap, n_submap=pb.n_submap, global2local=pb.global2local,
        epsilon=obs["epsilon"], gamma=obs["gamma"], cal=obs["cal"], IAU=IAU, hwp=hwp,
        shared_flags=pb.shared_flags, shared_flag_mask=pb.shared_flag_mask,
        solver_flags=pb.solver_flags, solver_flag_mask=pb.det_flag_mask)
    if expand:
        dobs.expand_pointing(np.zeros(pb.n_submap, dtype=np.uint8))
    return dobs


@pytest.fixture(scope="module", params=[False, True], ids=["COSMO", "IAU"])
def rotated(request):
    IAU = request.param
    ck = H.checker()
    obs, hwp = _rotated_observation(60000)
    pb = O.build_problem(obs, ck, rcond_threshold=1e-3, hwp=hwp, IAU=IAU)
    # every pair's rotation, from the oracle's weights on its first in-view sample: B != 0
    s = int(obs["intervals"][0]["first"])
    q0, u0 = pb.weights[0::2, s, 1], pb.weights[0::2, s, 2]
    q1, u1 = pb.weights[1::2, s, 1], pb.weights[1::2, s, 2]
    B = (u1 * q0 - q1 * u0) / (q0 * q0 + u0 * u0)
    assert np.all(np.abs(B[:3]) > 0.1), B
    return SimpleNamespace(ck=ck, obs=obs, hwp=hwp, IAU=IAU, pb=pb)


@pytest.mark.parametrize("regen", [False, True])
def test_rotated_pairs_match_the_oracle(rotated, regen):
    """Every LHS path, the RHS, the binned map and ten restarted PCG iterations, with stored
    pointing (from the fused pointing kernel, on the pair kernels) and regenerated pointing."""
    ck, obs, pb, hwp, IAU = rotated.ck, rotated.obs, rotated.pb, rotated.hwp, rotated.IAU
    lib = L.load()
    covapply = ck.cov_apply_diag
    dobs = _rotated_device_observation(obs, pb, hwp, IAU, expand=not regen)
    if not regen:
        np.testing.assert_array_equal(dobs.pixels.cpu().numpy(), pb.pixels)
        assert_close_norm(dobs.weights.cpu().numpy(), pb.weights, what="weights")
        h = dobs.handle().h
        assert lib.tb_obs_has_pair_weights(h) == 1
        paired = ct.c_int(0)
        L.check(lib.tb_obs_crossing_stats(h, None, None, ct.byref(paired)))
        assert paired.value == 1 and lib.tb_obs_blocked(h) == 1
    ds = Destriper([dobs], pb.n_local_submap, pb.n_pix_submap, pb.cov, pb.offset_var,
                   pb.amp_flags, regen=regen)
    assert ds._blocked() != regen
    rng = np.random.default_rng(3)
    a = np.where(pb.amp_flags == 0, rng.standard_normal(pb.n_amp), 0.0)
    ref = O.solver_lhs(pb, ck, a, covapply=covapply)
    a_d = torch.from_numpy(a).cuda()
    if regen:
        assert_close_norm(_lhs(ds, a_d), ref, what="LHS (regen)")
    else:
        for fused in (True, False):
            ds.fuse_lhs = fused
            assert_close_norm(_lhs(ds, a_d), ref, what=f"LHS (fused={fused})")
        ds.fuse_lhs = True
        try:
            for name, opts in VARIANTS:
                for k, v in opts.items():
                    L.check(lib.tb_set_option(k.encode(), v))
                dv = _rotated_device_observation(obs, pb, hwp, IAU, expand=True)
                if name in ("crossings", "pairw"):
                    assert lib.tb_obs_has_pair_weights(dv.handle().h) == 1
                dsv = Destriper([dv], pb.n_local_submap, pb.n_pix_submap, pb.cov, pb.offset_var,
                                pb.amp_flags)
                assert_close_norm(_lhs(dsv, a_d), ref, what=f"LHS ({name})")
        finally:
            for k, v in DEFAULT_OPTIONS.items():
                lib.tb_set_option(k.encode(), v)
    sig = torch.from_numpy(obs["signal"]).cuda()
    rhs_ref = O.solver_rhs(pb, ck, obs["signal"], covapply=covapply)
    assert_close_norm(ds.rhs([sig]).cpu().numpy(), rhs_ref, what="RHS")
    assert_close_norm(ds.bin_signal([sig]).cpu().numpy(), O.bin_map(pb, ck, obs["signal"],
                                                                     covapply), what="binned map")
    trace = []
    O.solve(pb, ck, rhs_ref, n_iter_max=10, covapply=covapply, trace=trace)
    assert len(trace) == 10
    H.restart_parity(ds, pb, trace, what=f"IAU={IAU} regen={regen}")


@pytest.mark.parametrize("IAU,regen", [(False, False), (True, True)])
def test_mapmaker_with_hwp_on_rotated_pairs(IAU, regen):
    """ops.MapMaker with StokesWeights(hwp_angle=..., IAU=...) on the rotated focal plane, against
    the oracle's restatement of the same stages (as tests/test_gpu_ops.py::
    test_mapmaker_end_to_end)."""
    ck = H.checker()
    covapply = ck.cov_apply_diag
    obs, hwp = _rotated_observation(24000)
    data = Data()
    data.obs.append(observation_from_synthetic(obs))
    data.obs[0].shared["hwp_angle"] = hwp
    pb = O.build_problem(obs, ck, rcond_threshold=1.0e-3, hwp=hwp, IAU=IAU)
    dp = ops.PointingDetectorSimple(view="scanning", shared_flags="flags", shared_flag_mask=1)
    pix = ops.PixelsHealpix(detector_pointing=dp, nside=obs["nside"], nest=obs["nest"],
                            create_dist="pixel_dist")
    wts = ops.StokesWeights(detector_pointing=dp, mode="IQU", hwp_angle="hwp_angle", IAU=IAU)
    binning = ops.BinMap(pixel_dist="pixel_dist", covariance="cov", pixel_pointing=pix,
                         stokes_weights=wts, noise_model="noise_model", full_pointing=True)
    tmpl = Offset(name="baselines", step_time=obs["step_time"], times="times",
                  noise_model="noise_model")
    tmat = ops.TemplateMatrix(templates=[tmpl], amplitudes="amplitudes")
    mapper = ops.MapMaker(name="mm", det_data="signal", binning=binning, template_matrix=tmat,
                          solve_rcond_threshold=1.0e-3, map_rcond_threshold=1.0e-3, iter_max=12,
                          convergence=1.0e-30, regenerate_pointing=regen)
    signal0 = obs["signal"].copy()
    mapper.apply(data)
    np.testing.assert_array_equal(data["pixel_dist"].global_submap_to_local, pb.global2local)
    assert_close_norm(data["mm_cov"].data, pb.cov, what="covariance")
    np.testing.assert_array_equal(data["mm_rcond"].raw > 0, pb.rcond > 0)
    assert_close_norm(data["mm_binmap"].data, O.bin_map(pb, ck, signal0, covapply),
                      what="binned map")
    rhs_ref = O.solver_rhs(pb, ck, signal0, covapply)
    _, hist_ref = O.solve(pb, ck, rhs_ref, convergence=1e-30, n_iter_max=12, covapply=covapply)
    H.assert_history_matches(mapper.history, hist_ref, H.pcg_envelope(pb, rhs_ref, 12),
                             what=f"IAU={IAU}")
    clean = signal0.copy()
    O.template_add(pb, O, -data["amplitudes"]["baselines"].local, clean)
    assert_close_norm(data["mm_map"].data, O.bin_map(pb, ck, clean, covapply),
                      what="destriped map")
