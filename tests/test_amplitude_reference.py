"""The CPU references of the amplitude-vector kernels (tests/amplitude_reference.py) checked on
their own: the exact dot against rational arithmetic, the model of the kernels' summation order
against its error bound, and the vectorised model against a scalar, thread-by-thread restatement
of k_amp_dot.  No GPU needed."""

from fractions import Fraction

import numpy as np
import pytest

import amplitude_reference as AR


def _rational_dot(a, b, flags=None):
    s = Fraction(0)
    for i, (x, y) in enumerate(zip(a.tolist(), b.tolist())):
        if flags is None or flags[i] == 0:
            s += Fraction(x) * Fraction(y)
    return s


def _cancelling(rng, n):
    """a.b much smaller than sum |a*b|: pairs (x, y), (x, -y(1 + 2^-40 t)) with x, y wide."""
    x = AR.wide_normals(rng, n)
    y = AR.wide_normals(rng, n)
    t = rng.standard_normal(n)
    a = np.concatenate([x, x])
    b = np.concatenate([y, -(y * (1.0 + 2.0 ** -40 * t))])
    perm = rng.permutation(2 * n)
    return a[perm], b[perm]


def _kernel_loop(a, b, flags):
    """k_amp_dot thread by thread, in plain Python floats: per-thread strided accumulation, the
    full 32-lane __shfl_down_sync tree (lanes past the end read their own value), the sequential
    sum over the 8 warps, and grid_finish's lane-strided sum over the block partials with the
    same tree."""
    a, b = a.tolist(), b.tolist()
    n = len(a)
    grid = AR.red_grid(n)
    stride = grid * AR.K_THREADS

    def tree(v):
        for off in (16, 8, 4, 2, 1):
            v = [v[lane] + (v[lane + off] if lane + off < 32 else v[lane]) for lane in range(32)]
        return v[0]

    partials = []
    for blk in range(grid):
        acc = []
        for tid in range(AR.K_THREADS):
            s = 0.0
            for i in range(blk * AR.K_THREADS + tid, n, stride):
                if flags is None or flags[i] == 0:
                    s += a[i] * b[i]
            acc.append(s)
        sh = [tree(acc[32 * w:32 * (w + 1)]) for w in range(AR.K_THREADS // 32)]
        t = 0.0
        for w in range(AR.K_THREADS // 32):
            t += sh[w]
        partials.append(t)
    lanes = []
    for lane in range(32):
        s = 0.0
        for blk in range(lane, grid, 32):
            s += partials[blk]
        lanes.append(s)
    return tree(lanes)


def _bits(v):
    return np.float64(v).view(np.int64)


def test_red_grid():
    assert [AR.red_grid(n) for n in (0, 1, 256, 257, 151551, 151552, 151553, 5529600)] == \
        [1, 1, 1, 2, 592, 592, 592, 592]


def test_two_product_is_exact():
    rng = np.random.default_rng(1)
    a, b = AR.wide_normals(rng, 500), AR.wide_normals(rng, 500)
    p, e = AR.two_product(a, b)
    for x, y, pp, ee in zip(a.tolist(), b.tolist(), p.tolist(), e.tolist()):
        assert Fraction(pp) + Fraction(ee) == Fraction(x) * Fraction(y)


@pytest.mark.parametrize("case", ["plain", "cancelling", "flagged", "tiny"])
def test_exact_dot_is_the_rational_sum_rounded(case):
    rng = np.random.default_rng(["plain", "cancelling", "flagged", "tiny"].index(case))
    flags = None
    if case == "cancelling":
        a, b = _cancelling(rng, 200)
    elif case == "tiny":
        a, b = AR.wide_normals(rng, 3), AR.wide_normals(rng, 3)
    else:
        a, b = AR.wide_normals(rng, 300), AR.wide_normals(rng, 300)
    if case == "flagged":
        flags = (rng.random(300) < 0.3).astype(np.uint8)
    exact = AR.exact_dot(a, b, flags)
    assert exact == float(_rational_dot(a, b, flags))
    if case == "cancelling":  # the test case really cancels: naive summation is far off
        assert abs(exact) < 1e-6 * AR.abs_dot(a, b)
        assert np.sum(a * b) != exact
    assert AR.exact_dot(a[:0], b[:0]) == 0.0


@pytest.mark.parametrize("n", [1, 31, 255, 256, 257, 10000, 151551, 151552, 151553, 1000003])
def test_model_is_within_its_error_bound(n):
    rng = np.random.default_rng(n)
    if n > 1:
        a, b = _cancelling(rng, n // 2)
        a, b = a[:n], b[:n]
        a = np.concatenate([a, AR.wide_normals(rng, n - len(a))])
        b = np.concatenate([b, AR.wide_normals(rng, n - len(b))])
    else:
        a, b = AR.wide_normals(rng, n), AR.wide_normals(rng, n)
    flags = (rng.random(n) < 0.1).astype(np.uint8)
    for fl in (None, flags):
        model = AR.model_amp_dot(a, b, fl)
        exact = AR.exact_dot(a, b, fl)
        bound = AR.model_error_bound(n, AR.abs_dot(a, b, fl))
        assert abs(model - exact) <= bound, (n, model, exact, bound)


@pytest.mark.parametrize("n", [0, 1, 31, 255, 256, 257, 1000, 8193, 151553])
def test_model_equals_the_thread_by_thread_loop(n):
    rng = np.random.default_rng(100 + n)
    a, b = AR.wide_normals(rng, n), AR.wide_normals(rng, n)
    flags = (rng.random(n) < 0.1).astype(np.uint8)
    for fl in (None, flags):
        assert _bits(AR.model_amp_dot(a, b, fl)) == _bits(_kernel_loop(a, b, fl)), n


def test_update_model_sums_are_the_dot_model():
    """model_pcg_update's (r.r, s.r) are the dot kernel's order over the updated vectors, with
    non-finite values at flagged entries kept out."""
    rng = np.random.default_rng(7)
    n = 3000
    x, r, d, q = (AR.wide_normals(rng, n) for _ in range(4))
    var = rng.random(n)
    flags = (rng.random(n) < 0.2).astype(np.uint8)
    bad = np.flatnonzero(flags)
    r[bad[::2]] = np.nan
    q[bad[1::2]] = np.inf
    var[bad[::3]] = np.nan
    x2, r2, s2, (rr, sr) = AR.model_pcg_update(1.5, -0.75, x, r, d, q, var, flags)
    assert np.isfinite(rr) and np.isfinite(sr)
    assert _bits(rr) == _bits(_kernel_loop(r2, r2, flags))
    assert _bits(sr) == _bits(_kernel_loop(s2, r2, flags))
    assert np.all(s2[bad].view(np.int64) == 0)          # +0.0, not -0.0
    np.testing.assert_array_equal(x2, x + d * -2.0)
