"""CPU references for the amplitude-vector kernels of the PCG loop (tb_solver.cu: k_amp_dot,
k_pcg_update, k_pcg_direction).  No GPU needed.

The library is built with -fmad=false, so every element-wise line of those kernels is an IEEE
multiply followed by an IEEE add, which numpy reproduces bit for bit.  Their reductions are
deterministic by construction: a fixed grid red_grid(n), a per-thread strided accumulation, a
fixed shuffle tree per warp, a sequential sum over the warps of a block and, in the last block to
finish, a fixed lane-strided sum over the block partials followed by the same shuffle tree.
``model_amp_dot`` / ``model_pcg_update`` restate that order in numpy, so the device results must
equal them bit for bit.  ``exact_dot`` is the correctly rounded value of the same sum, which
checks the model itself (``model_error_bound``)."""

import math

import numpy as np

K_THREADS = 256     # kThreads (tb_device.cuh)
K_RED_BLOCKS = 592  # kRedBlocks (tb_solver.cu): 4 x 148 SMs
WARP = 32
U = 2.0 ** -53      # unit roundoff of binary64


def wide_normals(rng, n):
    """Normal deviates scaled by 2^U(-30, 30): sums of their products cancel for real, so a
    different summation order changes the last bits."""
    return rng.standard_normal(n) * np.exp2(rng.uniform(-30.0, 30.0, n))


def red_grid(n):
    """The grid of every amplitude-vector kernel: one thread per entry up to kRedBlocks blocks,
    then a grid-stride loop."""
    return int(min(max((n + K_THREADS - 1) // K_THREADS, 1), K_RED_BLOCKS))


# ---- exact arithmetic ----------------------------------------------------------------------------
def _split(a):
    """Veltkamp split: a == hi + lo exactly, each half with at most 26 significant bits."""
    c = a * 134217729.0  # 2^27 + 1
    hi = c - (c - a)
    return hi, a - hi


def two_product(a, b):
    """Dekker: p = fl(a*b) and e with p + e == a*b exactly (no overflow / underflow assumed)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    p = a * b
    ah, al = _split(a)
    bh, bl = _split(b)
    e = ((ah * bh - p) + ah * bl + al * bh) + al * bl
    return p, e


def _unflagged(a, b, flags):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    if flags is None:
        return a, b
    keep = np.asarray(flags) == 0
    return a[keep], b[keep]


def exact_dot(a, b, flags=None):
    """The correctly rounded value of sum over flags == 0 of a*b (flags None: every entry)."""
    a, b = _unflagged(a, b, flags)
    p, e = two_product(a, b)
    return math.fsum(np.concatenate([p, e]).tolist())


def abs_dot(a, b, flags=None):
    """sum |a*b| over the unflagged entries, rounded upwards by a margin that covers fsum's own
    rounding (the scale of the error bound)."""
    a, b = _unflagged(a, b, flags)
    p, e = two_product(a, b)
    return math.fsum(np.abs(p).tolist() + np.abs(e).tolist()) * (1.0 + 4.0 * U)


def model_error_bound(n, abs_sum):
    """|model - exact| <= gamma_h * sum|a*b|: each product passes through at most h roundings
    (its own multiply, the strided accumulation, 5 shuffle levels, 8 warp sums, the lane-strided
    sum over the partials, 5 more shuffle levels)."""
    grid = red_grid(n)
    h = (-(-n // (grid * K_THREADS)) + 5 + 8 + -(-grid // WARP) + 5 + 1)
    return h * U / (1.0 - h * U) * abs_sum


# ---- the kernels' summation order -----------------------------------------------------------------
def _shuffle_tree(v):
    """`for (off = 16; off > 0; off >>= 1) v += __shfl_down_sync(~0u, v, off)` over the last axis
    (32 lanes); returns lane 0.  Lanes past the end read their own value, but lane 0 never
    depends on them, so keeping the first `off` lanes at each level is exact."""
    off = WARP // 2
    while off > 0:
        v = v[..., :off] + v[..., off:2 * off]
        off //= 2
    return v[..., 0]


def _grid_sum(terms, n):
    """The value k_amp_dot / k_pcg_update store for a per-entry term vector (0.0 where an entry is
    skipped: the accumulators start at +0.0 and can never become -0.0, so adding +0.0 and
    skipping give the same bits)."""
    grid = red_grid(n)
    stride = grid * K_THREADS
    n_pass = max(-(-n // stride), 1)
    padded = np.zeros(n_pass * stride)
    padded[:n] = terms
    padded = padded.reshape(n_pass, stride)
    acc = np.zeros(stride)
    for k in range(n_pass):                     # acc += a[i] * b[i], i += gridDim.x * kThreads
        acc = acc + padded[k]
    warp = _shuffle_tree(acc.reshape(grid, K_THREADS // WARP, WARP))  # [grid, 8]
    part = np.zeros(grid)
    for w in range(K_THREADS // WARP):          # block_sum: t += sh[w] from t = 0.0
        part = part + warp[:, w]
    lanes = np.zeros(WARP)                      # grid_finish: b = lane, lane + 32, ...
    for b0 in range(0, grid, WARP):
        chunk = np.zeros(WARP)
        m = min(WARP, grid - b0)
        chunk[:m] = part[b0:b0 + m]
        lanes = np.where(np.arange(WARP) < m, lanes + chunk, lanes)
    return float(_shuffle_tree(lanes))


def _masked_products(a, b, flags):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        p = a * b
    if flags is not None:
        p = np.where(np.asarray(flags) == 0, p, 0.0)
    return p


def model_amp_dot(a, b, flags=None):
    """What tb_amp_dot writes to out[0], bit for bit."""
    return _grid_sum(_masked_products(a, b, flags), len(a))


def model_pcg_update(delta, dq, x, r, d, q, var, flags):
    """What tb_pcg_update leaves behind: (x, r, s, (r.r, s.r)), bit for bit.
    alpha = delta / dq;  x + d*alpha;  r - q*alpha;  s = flag ? +0.0 : r*var."""
    alpha = np.float64(delta) / np.float64(dq)
    good = np.asarray(flags) == 0
    with np.errstate(invalid="ignore", over="ignore"):
        x_new = x + d * alpha
        r_new = r - q * alpha
        s_new = np.where(good, r_new * var, 0.0)
    rr = _grid_sum(_masked_products(r_new, r_new, flags), len(x))
    sr = _grid_sum(_masked_products(s_new, r_new, flags), len(x))
    return x_new, r_new, s_new, (rr, sr)


def model_pcg_direction(delta_new, delta_old, d, s):
    """What tb_pcg_direction leaves in d: d*beta + s with beta = delta_new / delta_old."""
    beta = np.float64(delta_new) / np.float64(delta_old)
    return d * beta + s
