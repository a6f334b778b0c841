"""Shared helpers for the parity tests."""

import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import toast_oracle as O  # noqa: E402  (the checker; never the thing under test)
from toast_b200 import synthetic as S  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
GOLDEN_FULL_MAX = 4096   # golden arrays up to this many elements are stored whole,
GOLDEN_SAMPLE = 512      # larger ones as a SHA-256 of their bytes plus this many sampled values

# north_star tolerance: fp64 results within 1e-10 relative of the reference COMPILED path.
# Element-wise relative error is meaningless for weights/maps that cross zero (cos 2a -> 0), so
# the bar is norm-wise: max|a - b| <= RTOL * max|b|  (SURVEY.md section 7, hard part 2).
RTOL = 1.0e-10


def assert_close_norm(actual, expected, rtol=RTOL, what=""):
    actual = np.asarray(actual, dtype=np.float64)
    expected = np.asarray(expected, dtype=np.float64)
    assert actual.shape == expected.shape, (what, actual.shape, expected.shape)
    scale = np.max(np.abs(expected)) if expected.size else 0.0
    err = np.max(np.abs(actual - expected)) if expected.size else 0.0
    assert np.all(np.isfinite(actual)), f"{what}: non-finite values"
    assert err <= rtol * max(scale, 1e-300), f"{what}: max|diff| {err:.3e} > {rtol:g} * {scale:.3e}"


def digest(a):
    a = np.ascontiguousarray(a)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()


def _golden_sample_index(n):
    return np.sort(np.random.default_rng(0).choice(n, GOLDEN_SAMPLE, replace=False))


def pack_golden(prefix, arrays):
    """The npz entries that pin ``arrays`` (name -> ndarray) bit for bit, under
    ``prefix/name`` (or ``name`` when ``prefix`` is None)."""
    out = {}
    for key, a in arrays.items():
        a = np.asarray(a)
        name = f"{prefix}/{key}" if prefix else key
        if a.size <= GOLDEN_FULL_MAX:
            out[name] = a
        else:
            out[name + "/sha256"] = np.array(digest(a))
            out[name + "/sample"] = a.reshape(-1)[_golden_sample_index(a.size)]
    return out


def assert_packed(g, name, a):
    """``a`` is bit for bit the array that pack_golden stored as ``name`` in the npz ``g``."""
    a = np.asarray(a)
    if name in g.files:
        np.testing.assert_array_equal(a, g[name], err_msg=name)
    else:
        np.testing.assert_array_equal(a.reshape(-1)[_golden_sample_index(a.size)],
                                      g[name + "/sample"], err_msg=name)
        assert digest(a) == str(g[name + "/sha256"]), name


def checker():
    """The parity checker: the compiled REFERENCE if oracle/_ref is present, else the C port."""
    ref = O.load_ref()
    return ref if ref is not None else O


def scan_fn(K, dtype="float64"):
    return getattr(K, f"ops_scan_map_{dtype}", None) or K.scan_map


def iso_quat(theta, phi, psi):
    """qa.from_iso_angles: Rz(phi) Ry(theta) Rz(psi)."""
    return S.q_mult(S.q_rotation(S.ZAXIS, phi),
                    S.q_mult(S.q_rotation(S.YAXIS, theta), S.q_rotation(S.ZAXIS, psi)))


def healpix_angle_sets():
    """The eps-perturbed pole / meridian angles and the regular grid of
    tests/healpix.py:29-74 (healpy replaced by the compiled reference as the authority)."""
    eps32 = np.finfo(np.float32).eps
    eps64 = np.finfo(np.float64).eps
    theta = [0.0, eps64, eps32, np.radians(90.0) - eps32, np.radians(90.0) - eps64,
             np.radians(90.0), np.radians(90.0) + eps64, np.radians(90.0) + eps32,
             np.radians(180.0) - eps32, np.radians(180.0) - eps64, np.radians(180.0)]
    phi = []
    for pts in [0.0, 90.0, 180.0, 270.0, 360.0]:
        phi += [np.radians(pts) - eps32, np.radians(pts) - eps64, np.radians(pts),
                np.radians(pts) + eps64, np.radians(pts) + eps32]
    ext = np.array([(t, p) for t in theta for p in phi])
    nreg = 100
    reg = np.array([(np.radians(t * 180.0 / nreg), np.radians(p * 360.0 / nreg))
                    for t in range(nreg) for p in range(nreg)])
    both = np.vstack([ext, reg])
    return np.ascontiguousarray(both[:, 0]), np.ascontiguousarray(both[:, 1])


def ang_to_quat(theta, phi):
    return np.ascontiguousarray(iso_quat(theta, phi, np.zeros_like(theta)))


def pcg_envelope(pb, rhs, n_iter, prior=None):
    """How reproducible the reference's OWN residual history is: relative deviation of the
    oracle's history under a 1-ulp random perturbation of the RHS (running maximum).  CG
    amplifies rounding noise exponentially, so beyond the first iterations the history is not
    reproducible to 1e-10 even by the reference itself with a different summation order (its
    project_signal uses OpenMP atomics: template_offset.cpp:301-327)."""
    rng = np.random.default_rng(0)
    rhs2 = rhs * (1.0 + 2.2e-16 * rng.choice([-1.0, 1.0], size=rhs.shape))
    _, h1 = O.solve(pb, O, rhs, n_iter_max=n_iter, prior=prior)
    _, h2 = O.solve(pb, O, rhs2, n_iter_max=n_iter, prior=prior)
    n = min(len(h1), len(h2))
    env = np.abs(np.array(h2[:n]) - np.array(h1[:n])) / np.array(h1[:n])
    return np.maximum.accumulate(env)


def assert_history_matches(hist, hist_ref, env, what=""):
    """PCG residual history parity: 1e-10 relative (north_star) wherever the reference itself is
    reproducible to 1e-13 under a 1-ulp perturbation of its input -- always including the first
    iteration -- and within 1e3 x the reference's own reproducibility envelope elsewhere."""
    hist, hist_ref = np.asarray(hist), np.asarray(hist_ref)
    assert len(hist) == len(hist_ref), (what, len(hist), len(hist_ref))
    dev = np.abs(hist - hist_ref) / hist_ref
    n = min(len(dev), len(env))
    assert dev[0] <= RTOL, f"{what}: first iteration deviates {dev[0]}"
    bound = np.maximum(RTOL, 1.0e3 * env[:n])
    assert np.all(dev[:n] <= bound), f"{what}: history deviates {dev[:n]} > {bound}"


def host_math_lib():
    """g++ build of the product's host/device cores (tests/csrc/host_math.cpp: tb_math.cuh and
    tb_prior.cuh compiled for the host, -ffp-contract=off) for the CPU suite."""
    import ctypes as ct
    import subprocess

    csrc = os.path.join(ROOT, "tests", "csrc")
    so = os.path.join(csrc, "libhostmath.so")
    src = os.path.join(csrc, "host_math.cpp")
    deps = [src] + [os.path.join(ROOT, "toast_b200", "csrc", h)
                    for h in ("tb_math.cuh", "tb_prior.cuh", "tb_wcs.cuh")]
    if (not os.path.exists(so)) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call(["/usr/bin/g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared",
                               "-x", "c++", "-o", so, src, "-lm"])
    lib = ct.CDLL(so)
    lib.tbm_quat2pix.restype = ct.c_int64
    return lib


def first_iteration_over(hist, hist_ref, tol=RTOL):
    """Index of the first PCG iteration whose relative residual deviates from the reference's
    by more than ``tol`` (relative), or None."""
    hist, hist_ref = np.asarray(hist), np.asarray(hist_ref)
    n = min(len(hist), len(hist_ref))
    dev = np.abs(hist[:n] - hist_ref[:n]) / np.abs(hist_ref[:n])
    over = np.flatnonzero(dev > tol)
    return (int(over[0]) if len(over) else None), dev


def restart_parity(ds, pb, trace, rtol=RTOL, what=""):
    """RESTART PARITY of the PCG (the rigorous form of 'residual histories agree to 1e-10'):
    CG amplifies rounding differences exponentially, so two correct implementations drift apart
    when they run freely.  Here the device solver is loaded with the ORACLE's state before
    iteration k (x, r, d, delta: ``trace`` from ``O.solve(..., trace=[])``), runs exactly ONE
    iteration (LHS, d.q, x/r/s update, r.r) and must reproduce what the reference's iteration k
    produced -- q = A d, alpha, the new residual norm and the new x, r -- to 1e-10, for EVERY k.
    Returns the per-iteration worst relative deviation."""
    import torch

    from toast_b200.solver import _PCGState

    st = _PCGState(pb.n_amp, ds.device)
    worst = []
    dev_t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(ds.device)
    nrm = lambda a, b: float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))
    for k, t in enumerate(trace):
        st.x.copy_(dev_t(t["x"]))
        st.r.copy_(dev_t(t["r"]))
        st.d.copy_(dev_t(t["d"]))
        st.delta.fill_(t["delta"])
        ds.lhs_and_dot(st)
        ds.update(st)
        e_q = nrm(st.q.cpu().numpy(), t["q"])
        alpha = t["delta"] / float(st.dq.item())
        e_alpha = abs(alpha - t["alpha"]) / abs(t["alpha"])
        e_rr = abs(float(st.sums[0].item()) - t["sqsum"]) / t["sqsum"]
        x_ref = t["x"] + t["d"] * t["alpha"]
        r_ref = t["r"] - t["q"] * t["alpha"]
        e_x = nrm(st.x.cpu().numpy(), x_ref)
        e_r = nrm(st.r.cpu().numpy(), r_ref) * (np.max(np.abs(r_ref)) / np.max(np.abs(t["r"])))
        w = max(e_q, e_alpha, e_rr, e_x, e_r)
        worst.append(w)
        assert w <= rtol, (f"{what}: restart parity fails at iteration {k}: q {e_q:.2e} "
                           f"alpha {e_alpha:.2e} r.r {e_rr:.2e} x {e_x:.2e} r {e_r:.2e}")
    return worst


def order_tolerance(ref, ref_reversed, rcond=None, what=""):
    """Tolerance for a quantity that passes through the pixel-covariance product.

    north_star asks for 1e-10.  That bar is kept wherever the problem supports it (every test at
    the round-1 thresholds 1e-3 / 1e-5).  At the PRODUCTION threshold (rcond 1e-8: pixels with
    condition numbers up to 1e8 are kept) the product C.z amplifies the rounding of the
    noise-weighted sums z by the condition number, so the result is only DEFINED up to
    kappa * eps = 2e-8 in the worst pixel -- for the reference as much as for anything else: the
    same compiled reference kernels fed the detectors in reverse order (another valid summation
    order) differ from themselves by 1e-11 ... 4e-10 norm-wise on these problems.  The bar is
    therefore the largest of
        1e-10,
        4 x the reference's own order dependence (measured here, per quantity), and
        0.1 x eps / rcond  (a tenth of the forward-error bound kappa * eps of C.z; 2.2e-9 at 1e-8)
    and every test prints / stores both the tolerance used and the reference's self-difference."""
    scale = max(float(np.max(np.abs(ref))), 1e-300)
    self_diff = float(np.max(np.abs(np.asarray(ref) - np.asarray(ref_reversed)))) / scale
    cond = 0.1 * np.finfo(np.float64).eps / rcond if rcond else 0.0
    return max(RTOL, 4.0 * self_diff, cond), self_diff
