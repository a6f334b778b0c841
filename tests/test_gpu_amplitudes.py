"""The amplitude-vector kernels bit for bit: the PCG loop's dot product, update and direction
(tb_amp_dot, tb_pcg_update, tb_pcg_direction) and the Offset template's add / project /
preconditioner (k_offset_*) on the layouts where a grid-stride loop, a grid reduction or a warp
run-sum goes wrong.

The library is built with -fmad=false, so every element-wise result must equal numpy bit for bit,
and the grid reductions are deterministic, so the reduced scalars must equal the numpy model of
their summation order (tests/amplitude_reference.py) bit for bit as well.  Only the Offset
projection sums with atomics: it is held per amplitude to the error bound that every summation
order satisfies, not to a norm-wise tolerance."""

import functools
import math

import numpy as np
import pytest
import torch

import amplitude_reference as AR
import helpers as H
from helpers import O, S
from toast_b200 import kernels as KC
from toast_b200 import lib as L

pytestmark = pytest.mark.gpu

N_VALUES = [0, 1, 31, 255, 256, 257,
            151551, 151552, 151553,  # 592 x 256: the grid stops growing, the stride loop starts
            1000003,
            5529600]                 # 128 detectors x 43 200 baselines: one rank of C4
FLAG_CASES = ["null", "none", "all", "random", "block_runs", "nonfinite"]
REPEATS = 3


# ---- helpers -------------------------------------------------------------------------------------
def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _nan(n):
    return torch.full((n,), float("nan"), dtype=torch.float64, device="cuda")


def assert_same_bits(actual, expected, what=""):
    """Equal bit for bit (signed zeros included); where `expected` is NaN, `actual` must be NaN
    (the device and the host may produce NaNs with different payloads)."""
    actual = np.atleast_1d(np.asarray(actual, dtype=np.float64))
    expected = np.atleast_1d(np.asarray(expected, dtype=np.float64))
    assert actual.shape == expected.shape, (what, actual.shape, expected.shape)
    nan = np.isnan(expected)
    assert np.array_equal(np.isnan(actual), nan), f"{what}: NaNs differ"
    bad = np.flatnonzero(actual[~nan].view(np.int64) != expected[~nan].view(np.int64))
    if bad.size:
        i = np.flatnonzero(~nan)[bad[0]]
        raise AssertionError(f"{what}: {bad.size} of {expected.size} entries differ, first at {i}:"
                             f" {actual[i]!r} != {expected[i]!r}")


@functools.lru_cache(maxsize=1)
def _vectors(n):
    """Seeded inputs of length n (one n at a time: the largest is 350 MB)."""
    rng = np.random.default_rng([n, 2026])
    v = {k: AR.wide_normals(rng, n) for k in ("a", "b", "x", "r", "d", "q")}
    v["var"] = np.exp2(rng.uniform(-20.0, 20.0, n))
    i = np.arange(n)
    blk = i // AR.K_THREADS
    v["flags"] = {
        "none": np.zeros(n, dtype=np.uint8),
        "all": np.ones(n, dtype=np.uint8),
        "random": (rng.random(n) < 0.1).astype(np.uint8),
        # whole blocks, and half blocks that end on a block edge
        "block_runs": ((blk % 3 == 1) | ((blk % 3 == 2) & (i % AR.K_THREADS >= 128)))
        .astype(np.uint8),
    }
    return v


def _case(n, case):
    """(inputs, flags or None) for one flag case; "nonfinite" is "random" with NaN / +-Inf at
    flagged entries of every input the kernels read."""
    v = dict(_vectors(n))
    if case == "null":
        return v, None
    if case != "nonfinite":
        return v, v["flags"][case]
    flags = v["flags"]["random"]
    bad = np.flatnonzero(flags)
    for j, k in enumerate(("a", "b", "r", "q", "var")):
        x = v[k].copy()
        x[bad[j::5]] = np.nan
        x[bad[(j + 1) % 5::5]] = np.inf
        x[bad[(j + 2) % 5::5]] = -np.inf
        v[k] = x
    return v, flags


def _other_n(n):
    """A length whose grid differs from n's: a reduction of it in between two of n's checks that
    the last block resets the completion counter for a launch of another size."""
    return 5000 if AR.red_grid(n) != AR.red_grid(5000) else 300


@functools.lru_cache(maxsize=None)
def _other_inputs(m):
    rng = np.random.default_rng([m, 7])
    a, b = AR.wide_normals(rng, m), AR.wide_normals(rng, m)
    return _dev(a), _dev(b), AR.model_amp_dot(a, b)


def _dot(a, b, flags, n):
    out = _nan(1)
    rc = L.load().tb_amp_dot(L.ptr(a), L.ptr(b), L.ptr(flags), n, L.ptr(out), _stream())
    assert rc == 0, L.last_error()
    return out


def _interleave(n):
    m = _other_n(n)
    a, b, expect = _other_inputs(m)
    assert_same_bits(_dot(a, b, None, m).cpu().numpy(), expect, f"interleaved dot n={m}")


# ---- 1. PCG kernels ------------------------------------------------------------------------------
@pytest.mark.parametrize("case", FLAG_CASES)
@pytest.mark.parametrize("n", N_VALUES)
def test_amp_dot_is_the_model_bit_for_bit(n, case):
    v, flags = _case(n, case)
    expect = AR.model_amp_dot(v["a"], v["b"], flags)
    assert np.isfinite(expect)
    if n == 0 or case == "all":
        assert expect.hex() == "0x0.0p+0"  # +0.0
    a, b = _dev(v["a"]), _dev(v["b"])
    f = None if flags is None else _dev(flags)
    for rep in range(REPEATS):
        got = _dot(a, b, f, n).cpu().numpy()
        assert_same_bits(got, expect, f"dot n={n} {case} run {rep}")
        _interleave(n)


@pytest.mark.parametrize("n", N_VALUES)
def test_amp_dot_of_one_scale_values(n):
    """Unscaled normal deviates: no term dominates, so the rounding of every product and of every
    per-thread addition shows in the sum (with wide values a fused multiply-add in the strided
    accumulation past 592 x 256 entries can hide behind the largest terms)."""
    rng = np.random.default_rng([n, 5])
    a, b = rng.standard_normal(n), rng.standard_normal(n)
    flags = (rng.random(n) < 0.1).astype(np.uint8)
    expect = AR.model_amp_dot(a, b, flags)
    got = _dot(_dev(a), _dev(b), _dev(flags), n).cpu().numpy()
    assert_same_bits(got, expect, f"dot n={n}")


@pytest.mark.parametrize("case", FLAG_CASES[1:])
@pytest.mark.parametrize("n", N_VALUES)
def test_pcg_update_is_numpy_bit_for_bit(n, case):
    v, flags = _case(n, case)
    rng = np.random.default_rng([n, 3])
    delta, dq = float(abs(AR.wide_normals(rng, 1)[0])), float(AR.wide_normals(rng, 1)[0])
    x_ref, r_ref, s_ref, sums_ref = AR.model_pcg_update(delta, dq, v["x"], v["r"], v["d"], v["q"],
                                                        v["var"], flags)
    assert np.all(np.isfinite(sums_ref))
    good = flags == 0
    assert np.all(np.isfinite(x_ref)) and np.all(np.isfinite(r_ref[good]))
    x0, r0, d, q, var, f = (_dev(v["x"]), _dev(v["r"]), _dev(v["d"]), _dev(v["q"]),
                            _dev(v["var"]), _dev(flags))
    sc = _dev(np.array([delta, dq]))
    lib = L.load()
    for rep in range(REPEATS):
        x, r, s, sums = x0.clone(), r0.clone(), _nan(n), _nan(2)
        rc = lib.tb_pcg_update(L.ptr(sc[0:]), L.ptr(sc[1:]), L.ptr(x), L.ptr(r), L.ptr(d),
                               L.ptr(q), L.ptr(s), L.ptr(var), L.ptr(f), n, L.ptr(sums),
                               _stream())
        assert rc == 0, L.last_error()
        what = f"update n={n} {case} run {rep}"
        assert_same_bits(sums.cpu().numpy(), np.array(sums_ref), what + ": (r.r, s.r)")
        assert_same_bits(x.cpu().numpy(), x_ref, what + ": x")
        assert_same_bits(r.cpu().numpy(), r_ref, what + ": r")
        s_h = s.cpu().numpy()
        assert_same_bits(s_h, s_ref, what + ": s")
        assert np.all(s_h[~good].view(np.int64) == 0), what + ": s is not +0.0 where flagged"
        _interleave(n)


@pytest.mark.parametrize("n", N_VALUES)
def test_pcg_direction_is_numpy_bit_for_bit(n):
    v = _vectors(n)
    rng = np.random.default_rng([n, 4])
    dnew, dold = (float(abs(x)) for x in AR.wide_normals(rng, 2))
    expect = AR.model_pcg_direction(dnew, dold, v["d"], v["a"])
    d0, s = _dev(v["d"]), _dev(v["a"])
    sc = _dev(np.array([dnew, dold]))
    for rep in range(REPEATS):
        d = d0.clone()
        rc = L.load().tb_pcg_direction(L.ptr(sc[0:]), L.ptr(sc[1:]), L.ptr(d), L.ptr(s), n,
                                       _stream())
        assert rc == 0, L.last_error()
        assert_same_bits(d.cpu().numpy(), expect, f"direction n={n} run {rep}")
        _interleave(n)


def test_empty_vectors_write_zero_sums():
    """n = 0 with no vectors at all (an empty tensor has no data pointer): out and sums are +0.0,
    and the direction touches nothing."""
    lib = L.load()
    sc = _dev(np.array([2.0, 3.0]))
    out, sums = _nan(1), _nan(2)
    assert lib.tb_amp_dot(None, None, None, 0, L.ptr(out), _stream()) == 0, L.last_error()
    assert lib.tb_pcg_update(L.ptr(sc[0:]), L.ptr(sc[1:]), None, None, None, None, None, None,
                             None, 0, L.ptr(sums), _stream()) == 0, L.last_error()
    assert lib.tb_pcg_direction(L.ptr(sc[0:]), L.ptr(sc[1:]), None, None, 0, _stream()) == 0
    assert_same_bits(out.cpu().numpy(), [0.0], "dot")
    assert_same_bits(sums.cpu().numpy(), [0.0, 0.0], "sums")


def test_pcg_entry_points_refuse_bad_arguments():
    """NULL scalars, NULL vectors of a non-empty call and negative lengths are refused with
    TB_ERR_ARG before anything is launched (nothing is written)."""
    lib = L.load()
    n = 1000
    rng = np.random.default_rng(9)
    vec = [_dev(AR.wide_normals(rng, n)) for _ in range(6)]
    f = _dev(np.zeros(n, dtype=np.uint8))
    sc = _dev(np.array([1.0, 2.0]))
    out = _nan(2)
    p = L.ptr
    dot = [p(vec[0]), p(vec[1]), p(f), n, p(out), _stream()]
    upd = [p(sc[0:]), p(sc[1:]), p(vec[0]), p(vec[1]), p(vec[2]), p(vec[3]), p(vec[4]),
           p(vec[5]), p(f), n, p(out), _stream()]
    dirn = [p(sc[0:]), p(sc[1:]), p(vec[2]), p(vec[4]), n, _stream()]
    saved = [t.cpu().numpy().copy() for t in vec]

    def variants(args, n_pos, pointers, empty_ok):
        """Each pointer NULL in turn, then n = -1; `empty_ok` pointers may be NULL at n = 0."""
        for k in pointers:
            a = list(args)
            a[k] = None
            yield f"arg {k} NULL", a
            if k not in empty_ok:
                a = list(a)
                a[n_pos] = 0
                yield f"arg {k} NULL at n = 0", a
        a = list(args)
        a[n_pos] = -1
        yield "n = -1", a

    calls = [("tb_amp_dot", dot, 3, [0, 1, 4], {0, 1}),
             ("tb_pcg_update", upd, 9, [0, 1, 2, 3, 4, 5, 6, 7, 8, 10], {2, 3, 4, 5, 6, 7, 8}),
             ("tb_pcg_direction", dirn, 4, [0, 1, 2, 3], {2, 3})]
    torch.cuda.synchronize()
    launches = lib.tb_launch_count()
    n_refused = 0
    for name, args, n_pos, pointers, empty_ok in calls:
        for what, a in variants(args, n_pos, pointers, empty_ok):
            rc = getattr(lib, name)(*a)
            assert rc == L.TB_ERR_ARG, (name, what, rc)
            assert "NULL argument" in L.last_error() or "negative" in L.last_error(), (name, what)
            n_refused += 1
    torch.cuda.synchronize()
    assert n_refused == 5 + 14 + 7
    assert lib.tb_launch_count() == launches
    assert np.all(np.isnan(out.cpu().numpy()))
    for t, s in zip(vec, saved):
        assert_same_bits(t.cpu().numpy(), s, "refused call wrote a vector")
    # the same arguments, complete, run
    assert lib.tb_amp_dot(*dot) == 0 and lib.tb_pcg_update(*upd) == 0
    assert lib.tb_pcg_direction(*dirn) == 0
    torch.cuda.synchronize()
    assert lib.tb_launch_count() == launches + 3


# ---- 2. Offset template kernels ------------------------------------------------------------------
STEPS = [1, 7, 31, 32, 33, 256, 1000]
FLAG_MASK = 2


def _edge_intervals(step):
    """Empty and one-sample intervals, gaps and adjacent intervals, lengths that are and are not
    multiples of the step (some shorter than it), one long enough to span several tiles, and the
    last interval ending at n_samp."""
    lengths = [0, 1, 1, 3 * step, 2 * step + 1, max(step - 1, 1), 37, 4000, 0, step + 5, 1, 2500]
    gaps = [0, 0, 2, 5, 0, 7, 1, 3, 0, 11, 2, 0]
    out, pos = [], 0
    for g, ln in zip(gaps, lengths):
        pos += g
        out.append((pos, pos + ln))
        pos += ln
    return out, pos


def _many_intervals(seed, n_view=300):
    """~300 short views (every tenth empty, gaps of 0..5 samples): find_view's binary search has
    nine levels and most warps straddle a view boundary."""
    rng = np.random.default_rng(seed)
    out, pos = [], 0
    for v in range(n_view):
        pos += int(rng.integers(0, 6))
        ln = 0 if v % 10 == 3 else int(rng.integers(1, 61))
        out.append((pos, pos + ln))
        pos += ln
    return out, pos + 3


LAYOUTS = ([("edges", step, 1 + k % 5) for k, step in enumerate(STEPS)]
           + [("many", step, 1 + (k + 2) % 5) for k, step in enumerate(STEPS)])


def _layout(kind, step, n_det):
    """Everything both the kernels and the numpy reference need for one problem."""
    rng = np.random.default_rng([STEPS.index(step), n_det, len(kind)])
    ranges, n_samp = _edge_intervals(step) if kind == "edges" else _many_intervals(step)
    iv = S.make_intervals(ranges)
    nav, det_start, n_amp = O.offset_layout(n_det, iv, step)
    n_buf = n_det + 1                                  # one row no detector maps to
    lay = dict(step=step, n_det=n_det, n_samp=n_samp, iv=iv, ranges=ranges, nav=nav,
               det_start=det_start, n_amp=n_amp, n_buf=n_buf)
    lay["data_index"] = rng.permutation(n_buf)[:n_det].astype(np.int32)
    fi = rng.permutation(n_buf)[:n_det].astype(np.int32)
    if n_det > 1:
        fi[n_det // 2] = -1                            # one detector without sample flags
    lay["flag_index"] = fi
    # flag bytes 0..3, flagged under mask 2 when the byte is 2 or 3; one interval flagged whole
    fl = rng.choice(np.arange(4, dtype=np.uint8), size=(n_buf, n_samp), p=[0.5, 0.25, 0.15, 0.1])
    a, b = ranges[4]
    fl[:, a:b] = 2
    lay["flag_data"] = fl
    aflags = (rng.random(n_amp) < 0.15).astype(np.uint8)
    if n_det > 1:
        aflags[det_start[1]:det_start[1] + n_amp // n_det] = 1   # one detector all flagged
    lay["aflags"] = aflags
    # sample index and detector-relative amplitude of every in-interval sample, view by view
    s_idx, rel, voff = [], [], 0
    for (first, last), na in zip(ranges, nav):
        s_idx.append(np.arange(first, last))
        rel.append(voff + np.arange(last - first) // step)
        voff += int(na)
    lay["s_idx"], lay["rel"] = np.concatenate(s_idx), np.concatenate(rel)
    in_iv = np.zeros(n_samp, dtype=bool)
    in_iv[lay["s_idx"]] = True
    lay["in_interval"] = in_iv
    # per-detector scales 2^-20 .. 2^20: amplitudes of very different sizes in one vector
    lay["det_scale"] = np.exp2(rng.uniform(-20.0, 20.0, n_det))
    lay["rng"] = rng
    return lay


def _samples(lay, k):
    """(sample index, global amplitude index) of detector k's in-interval samples."""
    return lay["s_idx"], lay["det_start"][k] + lay["rel"]


def _add_reference(lay, amps, d):
    """d[data_index[k], s] += amps[amp] for every in-interval sample whose amplitude is not
    flagged, written from the layout."""
    d = d.copy()
    for k in range(lay["n_det"]):
        s, amp = _samples(lay, k)
        keep = lay["aflags"][amp] == 0
        d[lay["data_index"][k], s[keep]] += amps[amp[keep]]
    return d


def _project_terms(lay, d, k):
    """(amplitude, value) of every sample detector k adds to an unflagged amplitude; a detector
    whose flag_index is -1 has no sample flags."""
    s, amp = _samples(lay, k)
    keep = lay["aflags"][amp] == 0
    fi = lay["flag_index"][k]
    if fi >= 0:
        keep &= (lay["flag_data"][fi, s] & FLAG_MASK) == 0
    return amp[keep], d[lay["data_index"][k], s[keep]]


def _project_reference(lay, d, out0):
    """Per amplitude: the exact (fsum) value of out0 plus its unflagged samples, the sample count
    m and the bound gamma_(m+1) (|out0| + sum |d|) that any summation order meets."""
    amp, val = [], []
    for k in range(lay["n_det"]):
        a, v = _project_terms(lay, d, k)
        amp.append(a)
        val.append(v)
    amp, val = np.concatenate(amp), np.concatenate(val)
    order = np.argsort(amp, kind="stable")
    amp, val = amp[order], val[order]
    exact = out0.copy()
    m = np.zeros(lay["n_amp"], dtype=np.int64)
    abs_sum = np.abs(out0)
    uniq, start, count = np.unique(amp, return_index=True, return_counts=True)
    for a, i0, c in zip(uniq.tolist(), start.tolist(), count.tolist()):
        vals = val[i0:i0 + c]
        exact[a] = math.fsum([out0[a]] + vals.tolist())
        m[a] = c
        abs_sum[a] += math.fsum(np.abs(vals).tolist())
    g = (m + 1) * AR.U
    bound = g / (1.0 - g) * abs_sum * (1.0 + 1e-12)
    return exact, m, bound


def _project_violations(lay, got, out0, exact, m, bound):
    """Indices where `got` breaks the per-amplitude check: flagged amplitudes and amplitudes with
    no unflagged sample must keep out0 bit for bit, the others lie within their bound."""
    keep = (lay["aflags"] != 0) | (m == 0)
    moved = keep & (got.view(np.int64) != out0.view(np.int64))
    off = ~keep & ~(np.abs(got - exact) <= bound)
    return np.flatnonzero(moved | off)


def _to(mem, a):
    return _dev(a) if mem == "device" else a.copy()


def _back(a):
    return a.cpu().numpy() if torch.is_tensor(a) else a


def _lid(p):
    return f"{p[0]}-step{p[1]}-det{p[2]}"


@pytest.mark.parametrize("mem", ["host", "device"])
@pytest.mark.parametrize("layout", LAYOUTS, ids=_lid)
def test_offset_add_to_signal_bit_for_bit(layout, mem):
    lay = _layout(*layout)
    rng, n_det = lay["rng"], lay["n_det"]
    amps = AR.wide_normals(rng, lay["n_amp"])
    amps[lay["aflags"] != 0] = np.nan                  # flagged amplitudes are never read
    d0 = rng.standard_normal((lay["n_buf"], lay["n_samp"]))
    d0[:, ~lay["in_interval"]] = np.nan                # samples outside every interval: untouched
    expect = _add_reference(lay, amps, d0)
    assert np.all(np.isfinite(expect[:, lay["in_interval"]]))

    ck = H.checker()
    d_ref = d0.copy()
    for k in range(n_det):
        ck.template_offset_add_to_signal(lay["step"], int(lay["det_start"][k]), lay["nav"], amps,
                                         lay["aflags"], int(lay["data_index"][k]), d_ref,
                                         lay["iv"], False)
    assert_same_bits(d_ref, expect, "oracle add")

    d = _to(mem, d0)
    for k in range(n_det):
        KC.template_offset_add_to_signal(lay["step"], int(lay["det_start"][k]), lay["nav"],
                                         _to(mem, amps), _to(mem, lay["aflags"]),
                                         int(lay["data_index"][k]), d, lay["iv"], False)
    assert_same_bits(_back(d), expect, "add (one call per detector)")
    d = _to(mem, d0)
    KC.template_offset_add_to_signal_batch(lay["step"], lay["det_start"], lay["nav"],
                                           _to(mem, amps), _to(mem, lay["aflags"]),
                                           lay["data_index"], d, lay["iv"], False)
    assert_same_bits(_back(d), expect, "add (batch)")


@pytest.mark.parametrize("mem", ["host", "device"])
@pytest.mark.parametrize("layout", LAYOUTS, ids=_lid)
def test_offset_project_signal_per_amplitude(layout, mem):
    lay = _layout(*layout)
    rng, n_det, step = lay["rng"], lay["n_det"], lay["step"]
    n_amp = lay["n_amp"]
    # wide values on every detector's own scale; NaN wherever a sample must not be read
    d = rng.standard_normal((lay["n_buf"], lay["n_samp"])) * np.exp2(
        rng.uniform(-4.0, 4.0, (lay["n_buf"], lay["n_samp"])))
    d[:, ~lay["in_interval"]] = np.nan
    unused = np.setdiff1d(np.arange(lay["n_buf"]), lay["data_index"])
    d[unused] = np.nan
    for k in range(n_det):
        row = lay["data_index"][k]
        d[row] *= lay["det_scale"][k]
        s, amp = _samples(lay, k)
        unread = lay["aflags"][amp] != 0
        if lay["flag_index"][k] >= 0:
            unread |= (lay["flag_data"][lay["flag_index"][k], s] & FLAG_MASK) != 0
        d[row, s[unread]] = np.nan
    # initial amplitudes on their detector's scale, so that the samples change them
    out0 = rng.standard_normal(n_amp) * np.repeat(lay["det_scale"], n_amp // n_det)
    exact, m, bound = _project_reference(lay, d, out0)
    assert np.all(np.isfinite(exact))
    # the problem reaches the cases it is meant to: flagged amplitudes, unflagged ones with no
    # unflagged sample, sums of several samples
    assert (lay["aflags"] != 0).any() and ((lay["aflags"] == 0) & (m == 0)).any()
    assert m.max() == 1 if step == 1 else m.max() > 1

    ck = H.checker()
    out_ref = out0.copy()
    for k in range(n_det):
        ck.template_offset_project_signal(
            int(lay["data_index"][k]), d, int(lay["flag_index"][k]), lay["flag_data"], FLAG_MASK,
            step, int(lay["det_start"][k]), lay["nav"], out_ref, lay["aflags"], lay["iv"], False)
    assert _project_violations(lay, out_ref, out0, exact, m, bound).size == 0, "oracle"

    fd, dd, af = _to(mem, lay["flag_data"]), _to(mem, d), _to(mem, lay["aflags"])
    out = _to(mem, out0)
    for k in range(n_det):
        KC.template_offset_project_signal(
            int(lay["data_index"][k]), dd, int(lay["flag_index"][k]), fd, FLAG_MASK, step,
            int(lay["det_start"][k]), lay["nav"], out, af, lay["iv"], False)
    got = _back(out)
    bad = _project_violations(lay, got, out0, exact, m, bound)
    assert bad.size == 0, f"project (one call per detector): amplitudes {bad[:8]}"

    outb = _to(mem, out0)
    KC.template_offset_project_signal_batch(lay["data_index"], dd, lay["flag_index"], fd,
                                            FLAG_MASK, step, lay["det_start"], lay["nav"], outb,
                                            af, lay["iv"], False)
    gotb = _back(outb)
    bad = _project_violations(lay, gotb, out0, exact, m, bound)
    assert bad.size == 0, f"project (batch): amplitudes {bad[:8]}"

    # the per-amplitude check is strictly stronger than the norm-wise one: push the smallest
    # summed amplitude off by half the norm-wise tolerance
    summed = np.flatnonzero((lay["aflags"] == 0) & (m > 0))
    i = summed[np.argmin(np.abs(exact[summed]))]
    worse = gotb.copy()
    worse[i] += 0.5 * H.RTOL * np.max(np.abs(exact))
    H.assert_close_norm(worse, exact, what="norm-wise check of a perturbed result")
    assert i in _project_violations(lay, worse, out0, exact, m, bound)


@pytest.mark.parametrize("mem", ["host", "device"])
@pytest.mark.parametrize("n_amp", [1, 255, 256, 257, 4099])
def test_offset_apply_diag_precond_bit_for_bit(n_amp, mem):
    rng = np.random.default_rng([n_amp, 5])
    var = np.exp2(rng.uniform(-20.0, 20.0, n_amp))
    a = AR.wide_normals(rng, n_amp)
    aflags = (rng.random(n_amp) < 0.2).astype(np.uint8)
    aflags[-1] = 1
    bad = np.flatnonzero(aflags)
    a[bad[::2]] = np.nan
    var[bad[1::2]] = np.inf
    expect = np.where(aflags == 0, a * var, 0.0)
    ck = H.checker()
    ref = np.full(n_amp, np.nan)
    ck.template_offset_apply_diag_precond(var, a, aflags, ref, False)
    assert_same_bits(ref, expect, "oracle precond")
    out = _to(mem, np.full(n_amp, np.nan))
    KC.template_offset_apply_diag_precond(_to(mem, var), _to(mem, a), _to(mem, aflags), out, False)
    assert_same_bits(_back(out), expect, "precond")
