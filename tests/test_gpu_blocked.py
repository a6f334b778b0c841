"""The block-ordered LHS (toast_b200/csrc/tb_blocked.cu) on the shapes where it takes its rarer
paths: pixel blocks with more than kBxUnitMax records, which are cut into several work units
(zero-fill, fp64 REDs, a separate covariance launch and a separate projection), a partial last
block (a local map that is not a multiple of the 128-pixel block), an odd detector count, and
several observations accumulated into one map.

Every problem is checked two ways:
  * bit for bit against a plain numpy reference on DYADIC inputs: integer amplitudes, detector
    weights and calibrations that are powers of two and a covariance that is 2^-12 on the I-I
    entry only.  Every term is then a multiple of 2^-16 and every partial sum stays far below
    2^53 x 2^-16, so any summation order gives the same bits and the comparison needs no
    tolerance (the bound is asserted on the reference's values, not assumed);
  * against the oracle on the problem's own weights and covariance (the Q/U arithmetic), at the
    1e-10 bar of the other parity tests.

The numpy model of the crossing list (_block_entries) predicts the device's record and work-unit
counts exactly, so each problem also proves that it reaches the path it is meant to test."""

import ctypes as ct
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import helpers as H
from helpers import O, S, assert_close_norm
from toast_b200 import lib as L
from toast_b200.solver import DeviceObservation, Destriper

BLOCK_PIX = 128      # kBxPix: local pixels per block
UNIT_MAX = 16384     # kBxUnitMax: records per work unit
RUN_MAX = 32         # k_xbuild cuts its runs at 32 flat view samples
DYADIC_GRAIN = 2.0 ** -16
COV_II = 2.0 ** -12

# id: workload, detectors, samples, nside, nside_submap
PROBLEMS = {
    # one full submap (3072 pixels): two split blocks (one of three units) among single-unit ones
    "split": ("c2", 32, 120000, 64, 16),
    # 48-pixel submaps: 1200 local pixels (1200 % 128 = 48), blocks straddle submaps
    "split_tail": ("c2", 32, 120000, 64, 2),
    # 192 pixels: both blocks split, the partial one included
    "split_partial": ("c1", 16, 120000, 4, 4),
    # an odd detector count: the last pair row has no partner
    "odd": ("c2", 31, 120000, 64, 16),
}
TAILS = ("split_tail", "split_partial")


# ---- inputs --------------------------------------------------------------------------------------
def _observation(pid, det_first=0, dyadic=True):
    workload, n_det, n_samp, nside, nss = PROBLEMS[pid]
    obs = S.make_observation(workload, n_det=n_det, n_samp=n_samp, det_first=det_first,
                             eps_max=0.03, nside=nside)
    obs["nside_submap"] = nss
    if dyadic:
        _make_dyadic(obs, seed=det_first)
    return obs


def _make_dyadic(obs, seed):
    """Detector weights from {0.5, 1, 2, 4}, different within every pair, and calibrations from
    {0.5, 1, 2}: set before build_problem, so that the oracle, the device and the numpy reference
    all see them (the Stokes I weight is then `cal` bit for bit)."""
    rng = np.random.default_rng([11, seed])
    n_det = obs["n_det"]
    w = np.empty(n_det)
    for p in range(0, n_det, 2):
        k = min(2, n_det - p)
        w[p:p + k] = rng.choice([0.5, 1.0, 2.0, 4.0], k, replace=False)
    obs["detweight"] = w
    obs["cal"] = rng.choice([0.5, 1.0, 2.0], n_det)


def _dyadic_cov(pb):
    """2^-12 on the I-I entry of every pixel the rcond cut keeps, zero elsewhere."""
    cov = np.zeros((pb.n_local_submap * pb.n_pix_submap, 6))
    cov[pb.rcond > 0, 0] = COV_II
    return cov.reshape(pb.n_local_submap, pb.n_pix_submap, 6)


def _dyadic_amplitudes(pb, seed=0):
    """Integer amplitudes in [-8, 8] and the problem's flags with every 7th baseline flagged as
    well.  Flagged baselines keep a non-zero amplitude: the kernels must ignore it."""
    rng = np.random.default_rng(seed)
    aflags = pb.amp_flags.copy()
    aflags[::7] = 1
    return rng.integers(-8, 9, pb.n_amp).astype(np.float64), aflags


# ---- numpy reference -----------------------------------------------------------------------------
def _flat_view_samples(pb):
    """Sample index and detector-relative amplitude index of every flat view sample (the views
    concatenated, as the device lays them out)."""
    idx, rel, voff = [], [], 0
    for iv, n in zip(pb.intervals, pb.n_amp_views):
        first, last = int(iv["first"]), int(iv["last"])
        idx.append(np.arange(first, last))
        rel.append(voff + np.arange(last - first) // pb.step_length)
        voff += int(n)
    return np.concatenate(idx), np.concatenate(rel)


def _local_pixels(pb, g2l):
    """[n_det, n_samp] local pixel of every sample, -1 where the solver flags it."""
    sm, lp = O.global_to_local(pb.pixels, pb.n_pix_submap, g2l)
    lpix = np.where(sm >= 0, sm * pb.n_pix_submap + lp, -2)
    lpix[(pb.solver_flags & pb.det_flag_mask) != 0] = -1
    assert not np.any(lpix == -2), "unflagged samples off the local map"
    return lpix


def _good_samples(pb, g2l, amp_offset=0):
    """(detector, local pixel, amplitude index) of every unflagged view sample."""
    idx, rel = _flat_view_samples(pb)
    lpix = _local_pixels(pb, g2l)[:, idx]
    det = np.broadcast_to(np.arange(pb.n_det)[:, None], lpix.shape)
    amp = amp_offset + pb.det_start[:, None] + rel[None, :]
    good = lpix >= 0
    return det[good], lpix[good], amp[good]


def _exact_sum(index, terms, n, grain=DYADIC_GRAIN):
    """Per-index sums of `terms`, after checking that they cannot depend on summation order:
    every term a multiple of `grain`, and the sum of magnitudes of every index below
    2^53 x `grain`."""
    assert np.all(np.mod(terms / grain, 1.0) == 0.0), f"a term is finer than {grain}"
    mag = np.bincount(index, weights=np.abs(terms), minlength=n)
    assert np.max(mag, initial=0.0) / grain < 2.0 ** 53, "a sum could round"
    return np.bincount(index, weights=terms, minlength=n)


class DyadicReference:
    """The two passes of the LHS on dyadic inputs, in plain numpy, for the observations
    parts = [(pb, global2local, amp_offset)] sharing one map of n_pix local pixels:
        pass 1   zI[p]  = sum over unflagged samples on p of  a_b w_d cal_d
        pass 2   out[b] = sum over unflagged samples of b of  w_d (a_b - cal_d m[p])
    with a_b = 0 and out[b] = 0 on flagged baselines; the LHS takes m = cii zI (cii: the I-I
    covariance per pixel, the only non-zero entry)."""

    def __init__(self, parts, n_pix, amps, aflags):
        self.n_pix, self.aflags = n_pix, aflags
        self.a = np.where(aflags == 0, amps, 0.0)
        self.samples = []
        for pb, g2l, off in parts:
            det, lp, amp = _good_samples(pb, g2l, off)
            self.samples.append((lp, amp, pb.det_scale[det], pb.cal[det]))

    def pass1(self):
        a = self.a
        return sum(_exact_sum(lp, a[amp] * w * cal, self.n_pix) for lp, amp, w, cal in self.samples)

    def pass2(self, m):
        a = self.a
        out = np.zeros(len(a))
        for lp, amp, w, cal in self.samples:
            # what a record adds up, n a w and (n cal m) w, is bounded by the sums of magnitudes
            _exact_sum(amp, np.abs(a[amp] * w) + np.abs(w * cal * m[lp]), len(a))
            out += _exact_sum(amp, w * (a[amp] - cal * m[lp]), len(a))
        out[self.aflags != 0] = 0.0
        return out

    def lhs(self, cii):
        zI = self.pass1()
        return zI, self.pass2(cii * zI)


# ---- numpy model of the block-ordered list -------------------------------------------------------
def _block_entries(pb, paired, g2l=None):
    """Entries per pixel block of the block-ordered crossing list (k_xbuild, k_bx_keys):
      * a row is a detector pair when `paired` (the partner of an odd last detector is absent),
        a detector otherwise;
      * runs are cut at every 32 flat view samples and start anew when (pixel of detector 0,
        pixel of detector 1, baseline) changes; runs with both detectors flagged are dropped;
      * a record whose two detectors fall in different pixels is entered once per pixel.
    `g2l`: the submap distribution of the map (default: the problem's own)."""
    g2l = pb.global2local if g2l is None else g2l
    idx, rel = _flat_view_samples(pb)
    lpix = _local_pixels(pb, g2l)[:, idx]
    if paired:
        lp0 = lpix[0::2]
        lp1 = np.full_like(lp0, -1)
        lp1[:pb.n_det // 2] = lpix[1::2]
    else:
        lp0, lp1 = lpix, np.full_like(lpix, -1)
    t = np.arange(len(idx))
    head = np.broadcast_to(t % RUN_MAX == 0, lp0.shape).copy()
    amp = np.broadcast_to(rel, lp0.shape)
    head[:, 1:] |= ((lp0[:, 1:] != lp0[:, :-1]) | (lp1[:, 1:] != lp1[:, :-1]) |
                    (amp[:, 1:] != amp[:, :-1]))
    rec = head & ~((lp0 == -1) & (lp1 == -1))
    x, y = lp0[rec], lp1[rec]
    first = np.where(x >= 0, x, y)
    second = y[(x >= 0) & (y >= 0) & (x != y)]
    n_blocks = -(-int(np.sum(g2l >= 0)) * pb.n_pix_submap // BLOCK_PIX)
    return np.bincount(np.concatenate([first, second]) // BLOCK_PIX, minlength=n_blocks)


def _units(entries):
    return np.maximum(1, -(-entries // UNIT_MAX))


# ---- CPU: the reference itself -------------------------------------------------------------------
def test_dyadic_reference_matches_the_oracle_lhs():
    """The numpy reference is the oracle's SolverLHS, bit for bit, on the same dyadic inputs."""
    obs = S.make_observation("c2", n_det=8, n_samp=24000, eps_max=0.03, nside=16)
    _make_dyadic(obs, seed=0)
    pb = O.build_problem(obs, O, rcond_threshold=1e-3)
    assert np.mean((pb.solver_flags & pb.det_flag_mask) == 0) > 0.25
    amps, aflags = _dyadic_amplitudes(pb)
    pb.cov = _dyadic_cov(pb)
    pb.amp_flags = aflags
    n_pix = pb.n_local_submap * pb.n_pix_submap
    cii = pb.cov[..., 0].reshape(-1)
    zI, ref = DyadicReference([(pb, pb.global2local, 0)], n_pix, amps, aflags).lhs(cii)
    np.testing.assert_array_equal(ref, O.solver_lhs(pb, O, amps, covapply=O.cov_apply_diag))
    # pass 1 alone: the I component of the oracle's binned template
    tod = np.zeros((pb.n_det, pb.n_samp))
    O.template_add(pb, O, amps, tod)
    binned = O.bin_map(pb, O, tod, O.cov_apply_diag)
    np.testing.assert_array_equal(binned.reshape(-1, 3)[:, 0], cii * zI)
    assert np.count_nonzero(ref) > pb.n_amp // 2 and np.count_nonzero(zI) > 10


# ---- device problems -----------------------------------------------------------------------------
def _device_observation(obs, pb, g2l=None, amp_offset=0, expand=True):
    dobs = DeviceObservation(
        focalplane=obs["focalplane"], boresight=obs["boresight"], intervals=obs["intervals"],
        det_scale=pb.det_scale, step_length=pb.step_length, nside=pb.nside, nest=pb.nest,
        n_pix_submap=pb.n_pix_submap, n_submap=pb.n_submap,
        global2local=pb.global2local if g2l is None else g2l, amp_offset=amp_offset,
        epsilon=obs["epsilon"], gamma=obs["gamma"], cal=obs["cal"],
        shared_flags=pb.shared_flags, shared_flag_mask=pb.shared_flag_mask,
        solver_flags=pb.solver_flags, solver_flag_mask=pb.det_flag_mask)
    if expand:
        dobs.expand_pointing(np.zeros(pb.n_submap, dtype=np.uint8))
    return dobs


def _check_block_list(pid, dobs, pb, g2l=None):
    """The device built the block-ordered list this problem is meant to have: its record and
    work-unit counts are the numpy model's, it has split blocks and, for the tail problems, a
    partial last block that holds records.  Returns the model's entries per block."""
    lib = L.load()
    h = dobs.handle().h
    assert lib.tb_obs_blocked(h) == 1, f"{pid}: no block-ordered list"
    assert lib.tb_bx_block_pixels() == BLOCK_PIX
    n_rec, n_rows, paired = ct.c_int64(0), ct.c_int64(0), ct.c_int(0)
    L.check(lib.tb_obs_crossing_stats(h, ct.byref(n_rec), ct.byref(n_rows), ct.byref(paired)))
    # the synthetic focal planes are orthogonal pairs: the rows are detector pairs
    assert paired.value == 1 and n_rows.value == (pb.n_det + 1) // 2
    n_rec, n_units, n_multi, n_blocks = (ct.c_int64(0) for _ in range(4))
    L.check(lib.tb_obs_blocked_stats(h, ct.byref(n_rec), ct.byref(n_units), ct.byref(n_multi),
                                     ct.byref(n_blocks)))
    entries = _block_entries(pb, paired.value, g2l)
    units = _units(entries)
    print(f"BLOCKED_STATS {pid}: n_records {n_rec.value} n_units {n_units.value} "
          f"n_multi_units {n_multi.value} n_blocks {n_blocks.value} (split blocks "
          f"{np.flatnonzero(units > 1).tolist()} of {units[units > 1].tolist()} units; records in "
          f"the last block {int(entries[-1])})")
    assert n_blocks.value == len(entries)
    assert (n_rec.value, n_units.value, n_multi.value) == \
        (int(entries.sum()), int(units.sum()), int(units[units > 1].sum())), f"{pid}: model"
    assert n_multi.value > 0
    if pid in TAILS:
        g2l = pb.global2local if g2l is None else g2l
        assert int(np.sum(g2l >= 0)) * pb.n_pix_submap % BLOCK_PIX != 0 and entries[-1] > 0
    else:
        assert n_units.value > n_multi.value
    return entries


@pytest.fixture(scope="module", params=list(PROBLEMS))
def dyadic(request):
    """A problem of PROBLEMS on dyadic inputs, on the device, with its numpy reference."""
    pid = request.param
    obs = _observation(pid)
    pb = O.build_problem(obs, O, rcond_threshold=1e-3)
    cov = _dyadic_cov(pb)
    amps, aflags = _dyadic_amplitudes(pb)
    n_pix = pb.n_local_submap * pb.n_pix_submap
    ref = DyadicReference([(pb, pb.global2local, 0)], n_pix, amps, aflags)
    cii = cov[..., 0].reshape(-1)
    zI, lhs = ref.lhs(cii)
    dobs = _device_observation(obs, pb)
    entries = _check_block_list(pid, dobs, pb)
    if pid in TAILS:  # the exact comparisons cover the pixels of the partial block
        assert np.any(zI[(len(entries) - 1) * BLOCK_PIX:] != 0.0)
    ds = Destriper([dobs], pb.n_local_submap, pb.n_pix_submap, cov, pb.offset_var, aflags)
    assert ds._blocked()
    return SimpleNamespace(pid=pid, obs=obs, pb=pb, cov=cov, cii=cii, amps=amps, aflags=aflags,
                           n_pix=n_pix, ref=ref, zI=zI, lhs=lhs, dobs=dobs, ds=ds,
                           h=dobs.handle().h, entries=entries,
                           a_d=torch.from_numpy(amps).cuda())


def _lhs(ds, a_d):
    q = torch.full_like(a_d, float("nan"))
    ds.lhs(a_d, q)
    return q.cpu().numpy()


# ---- GPU: exact references on dyadic inputs ------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fused", [True, False])
def test_lhs_is_exact_and_repeatable(dyadic, fused):
    """The default LHS (one fused kernel, after the launches of the split blocks) and the
    three-launch form, twice in a row on the same Destriper: a split block's scratch that is not
    zeroed again would double on the second call.  The map scratch starts as NaN: nothing may
    read it before writing it."""
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
    if not fused:  # the three-launch form leaves m = C z in the map
        np.testing.assert_array_equal(ds.zmap.cpu().numpy().reshape(-1, 3)[:, 0],
                                      dyadic.cii * dyadic.zI)


@pytest.mark.gpu
def test_pass1_and_pass2_alone(dyadic):
    """tb_bx_pass1 writes every block of the map (from NaN), adds to a given map with
    accumulate = 1, and tb_bx_pass2 projects a given I-only map."""
    lib = L.load()
    d, z = dyadic, dyadic.ds.zmap
    aflags_d = dyadic.ds.amp_flags
    z.fill_(float("nan"))
    L.check(lib.tb_bx_pass1(d.h, L.ptr(d.a_d), L.ptr(aflags_d), L.ptr(z), 0, -1, None))
    written = z.cpu().numpy().reshape(-1, 3)
    assert np.all(np.isfinite(written))
    np.testing.assert_array_equal(written[:, 0], d.zI)

    rng = np.random.default_rng(1)
    known = rng.integers(-64, 65, (d.n_pix, 3)) * 0.25
    z.copy_(torch.from_numpy(known.reshape(z.shape)))
    L.check(lib.tb_bx_pass1(d.h, L.ptr(d.a_d), L.ptr(aflags_d), L.ptr(z), 1, -1, None))
    added = z.cpu().numpy().reshape(-1, 3)
    np.testing.assert_array_equal(added[:, 0], known[:, 0] + d.zI)
    # Q and U: the same sums in another order
    assert_close_norm(added[:, 1:] - known[:, 1:], written[:, 1:], what="pass 1 Q/U, accumulated")

    m = np.zeros((d.n_pix, 3))
    m[:, 0] = rng.integers(-512, 513, d.n_pix) * 2.0 ** -8
    z.copy_(torch.from_numpy(m.reshape(z.shape)))
    q = torch.zeros_like(d.a_d)
    L.check(lib.tb_bx_pass2(d.h, L.ptr(z), L.ptr(q), -1, None))
    np.testing.assert_array_equal(q.cpu().numpy(), d.ref.pass2(m[:, 0]))


@pytest.mark.gpu
def test_pixel_chunked_passes(dyadic):
    """Pass 1 and pass 2 chunk by chunk (tb_obs_set_pixel_chunks) give the whole LHS, with chunk
    bounds on either side of every split block and with one chunk per block."""
    lib = L.load()
    d, ds = dyadic, dyadic.ds
    split = np.flatnonzero(_units(d.entries) > 1)
    around = np.unique(np.minimum(d.n_pix, np.concatenate(
        [[0, d.n_pix], split * BLOCK_PIX, (split + 1) * BLOCK_PIX])))
    every = list(range(0, d.n_pix, BLOCK_PIX)) + [d.n_pix]
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


# the kernel variants of test_gpu_solver.py::test_lhs_path_variants_agree
VARIANTS = (("crossings", dict(blocked=0, crossings=1, pair=1, pairw=1)),
            ("pairw", dict(blocked=0, crossings=0, pair=1, pairw=1)),
            ("pair", dict(blocked=0, crossings=0, pair=1, pairw=0)),
            ("general", dict(blocked=0, crossings=0, pair=0)))
DEFAULT_OPTIONS = dict(blocked=1, crossings=1, pair=1, pairw=1)


@pytest.mark.gpu
def test_lhs_path_variants_are_exact(dyadic):
    """Every other LHS kernel, and the regenerated-pointing form, on the same inputs."""
    lib = L.load()
    d = dyadic
    try:
        for name, opts in VARIANTS:
            for k, v in opts.items():
                L.check(lib.tb_set_option(k.encode(), v))
            dobs = _device_observation(d.obs, d.pb)
            ds = Destriper([dobs], d.pb.n_local_submap, d.pb.n_pix_submap, d.cov, d.pb.offset_var,
                           d.aflags)
            assert not ds._blocked()
            np.testing.assert_array_equal(_lhs(ds, d.a_d), d.lhs, err_msg=name)
    finally:
        for k, v in DEFAULT_OPTIONS.items():
            lib.tb_set_option(k.encode(), v)
    dobs = _device_observation(d.obs, d.pb, expand=False)
    ds = Destriper([dobs], d.pb.n_local_submap, d.pb.n_pix_submap, d.cov, d.pb.offset_var,
                   d.aflags, regen=True)
    np.testing.assert_array_equal(_lhs(ds, d.a_d), d.lhs, err_msg="regen")


@pytest.mark.gpu
@pytest.mark.parametrize("pid", ["split", "split_tail"])
def test_two_observations_accumulate(pid):
    """Two observations on one GPU (what ops.MapMaker runs for several observations): pass 1 of
    the second adds to the map of the first (accumulate = 1), pass 2 runs per observation.  Both
    use the union of their submaps; the second one's amplitudes follow the first one's."""
    n_det = PROBLEMS[pid][1]
    obs = [_observation(pid, det_first=k * n_det) for k in range(2)]
    pbs = [O.build_problem(o, O, rcond_threshold=1e-3) for o in obs]
    hit = pbs[0].hit_submaps | pbs[1].hit_submaps
    _, g2l = O.pixel_distribution(hit)
    n_local, nps = int(np.sum(hit != 0)), pbs[0].n_pix_submap
    n_pix = n_local * nps
    keep = np.zeros((n_local, nps), dtype=bool)
    for pb in pbs:  # the rcond cut of each observation, in the union's pixel numbering
        keep[g2l[pb.local_submaps]] |= pb.rcond.reshape(-1, nps) > 0
    cov = np.zeros((n_local, nps, 6))
    cov[keep, 0] = COV_II
    offsets = [0, pbs[0].n_amp]
    amps = np.concatenate([_dyadic_amplitudes(pb, seed=k)[0] for k, pb in enumerate(pbs)])
    aflags = np.concatenate([pb.amp_flags for pb in pbs])
    aflags[::7] = 1
    ref = DyadicReference([(pb, g2l, off) for pb, off in zip(pbs, offsets)], n_pix, amps, aflags)
    zI, lhs = ref.lhs(cov[..., 0].reshape(-1))
    dobs = []
    for o, pb, off in zip(obs, pbs, offsets):
        dobs.append(_device_observation(o, pb, g2l=g2l, amp_offset=off))
        _check_block_list(pid, dobs[-1], pb, g2l)
    ds = Destriper(dobs, n_local, nps, cov, np.concatenate([pb.offset_var for pb in pbs]),
                   aflags)
    assert ds._blocked()
    a_d = torch.from_numpy(amps).cuda()
    ds.zmap.fill_(float("nan"))
    first = _lhs(ds, a_d)
    np.testing.assert_array_equal(ds.zmap.cpu().numpy().reshape(-1, 3)[:, 0],
                                  cov[..., 0].reshape(-1) * zI)
    np.testing.assert_array_equal(first, lhs)
    np.testing.assert_array_equal(_lhs(ds, a_d), lhs)


# ---- GPU: oracle parity on the problems' own inputs ----------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("pid", ["split", "split_tail", "split_partial"])
def test_oracle_parity(pid):
    """LHS (fused and three-launch), RHS, binned map and ten restarted PCG iterations against the
    oracle, with the problem's own weights, calibration and covariance: the Q/U arithmetic that
    the dyadic inputs leave out."""
    ck = H.checker()
    obs = _observation(pid, dyadic=False)
    pb = O.build_problem(obs, ck, rcond_threshold=1e-3)
    dobs = _device_observation(obs, pb)
    _check_block_list(pid, dobs, pb)
    ds = Destriper([dobs], pb.n_local_submap, pb.n_pix_submap, pb.cov, pb.offset_var,
                   pb.amp_flags)
    assert ds._blocked()
    covapply = ck.cov_apply_diag
    rng = np.random.default_rng(3)
    a = np.where(pb.amp_flags == 0, rng.standard_normal(pb.n_amp), 0.0)
    ref = O.solver_lhs(pb, ck, a, covapply=covapply)
    a_d = torch.from_numpy(a).cuda()
    for fused in (True, False):
        ds.fuse_lhs = fused
        assert_close_norm(_lhs(ds, a_d), ref, what=f"LHS (fused={fused})")
    ds.fuse_lhs = True
    sig = torch.from_numpy(obs["signal"]).cuda()
    rhs_ref = O.solver_rhs(pb, ck, obs["signal"], covapply=covapply)
    assert_close_norm(ds.rhs([sig]).cpu().numpy(), rhs_ref, what="RHS")
    binned_ref = O.bin_map(pb, ck, obs["signal"], covapply)
    assert_close_norm(ds.bin_signal([sig]).cpu().numpy(), binned_ref, what="binned map")
    trace = []
    O.solve(pb, ck, rhs_ref, n_iter_max=10, covapply=covapply, trace=trace)
    assert len(trace) == 10
    H.restart_parity(ds, pb, trace, what=pid)
