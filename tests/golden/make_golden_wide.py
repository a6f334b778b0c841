"""Golden fixtures with >= 1000 hit pixels each (round-1 verdict: the first fixtures have 4-22).

Run in the build container (needs /root/reference compiled by oracle/build_ref.sh):

    python tests/golden/make_golden_wide.py

Inputs are regenerated deterministically by toast_b200.synthetic; the committed files hold the
outputs of the REFERENCE's compiled kernels driven by the oracle's restatement of the Python
glue: pixels (int32, every sample), weights (every 16th sample, as the SHA-256 of those values plus
512 of them, + per-detector column sums), the noise-weighted map, RHS, LHS(1), amplitudes after 2
PCG iterations and the residual history.
"""

import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from helpers import pack_golden  # noqa: E402
from oracle import toast_oracle as O  # noqa: E402
from toast_b200 import synthetic as S  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))

# (fixture, workload, n_det, n_samp, nside)
CASES = [
    ("c1_wide", "c1", 16, 30000, 64),
    ("c2_wide", "c2", 32, 36000, 256),
    ("c4_wide", "c4", 32, 60000, 128),
    ("c5_wide", "c5", 64, 36000, 256),
]
WSTRIDE = 16


def main():
    os.environ["OMP_NUM_THREADS"] = "1"
    R = O.load_ref()
    if R is None:
        raise SystemExit("oracle/_ref is not built: run oracle/build_ref.sh first")
    for name, wl, nd, ns, nside in CASES:
        obs = S.make_observation(wl, n_det=nd, n_samp=ns, eps_max=0.05, nside=nside)
        pb = O.build_problem(obs, R)
        cov = R.cov_apply_diag
        rhs = O.solver_rhs(pb, R, obs["signal"], covapply=cov)
        ones = np.where(pb.amp_flags == 0, 1.0, 0.0)
        lhs1 = O.solver_lhs(pb, R, ones, covapply=cov)
        amps2, _ = O.solve(pb, R, rhs, n_iter_max=2, covapply=cov)
        _, hist = O.solve(pb, R, rhs, n_iter_max=12, covapply=cov)
        idx = np.arange(nd, dtype=np.int32)
        zmap = np.zeros((pb.n_local_submap, pb.n_pix_submap, 3))
        R.build_noise_weighted(pb.global2local, zmap, idx, pb.pixels, idx, pb.weights, idx,
                               obs["signal"], idx, pb.solver_flags, pb.det_scale, 1,
                               pb.intervals, pb.shared_flags, 1, False)
        nz = np.flatnonzero(np.any(zmap.reshape(-1, 3) != 0, axis=1))
        assert len(nz) >= 1000, (name, len(nz))
        np.savez_compressed(
            os.path.join(HERE, f"{name}.npz"),
            workload=wl, n_det=nd, n_samp=ns, nside=nside, weight_stride=WSTRIDE,
            pixels=pb.pixels.astype(np.int32),
            **pack_golden(None, {"weights_strided": pb.weights[:, ::WSTRIDE, :]}),
            weights_colsum=pb.weights.sum(axis=1),
            hit_submaps=pb.hit_submaps,
            zmap_index=nz.astype(np.int32),
            zmap_values=zmap.reshape(-1, 3)[nz],
            rhs=rhs, lhs_of_ones=lhs1, amplitudes_iter2=amps2, history=np.array(hist),
        )
        print(name, "hit pixels", len(nz), "unflagged", float(np.mean(pb.solver_flags == 0)),
              "n_amp", pb.n_amp, "history", hist[0], "->", hist[-1],
              os.path.getsize(os.path.join(HERE, f"{name}.npz")) // 1024, "KiB")


if __name__ == "__main__":
    main()
