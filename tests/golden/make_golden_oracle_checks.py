"""Generate tests/golden/oracle_checks.npz: what the comparisons of tests/test_oracle.py with the
compiled reference (pointing, solver chain, covariance accumulation, eigen-inversion) are held to
on machines where oracle/_ref cannot be built.

The outputs come from the compiled reference when oracle/_ref is present.  Without it they come
from the C restatement (oracle/toast_oracle.c), which those same comparisons held bit for bit to
the compiled reference on exactly these inputs (the eigen-inversion within the tolerance of
``_check_cov_inverse``).  The entry ``source`` records which one wrote the file.  Arrays of more
than 4096 elements are stored as a SHA-256 of their bytes plus 512 sampled values.

    python tests/golden/make_golden_oracle_checks.py
"""

import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
os.environ["OMP_NUM_THREADS"] = "1"   # the reference's OpenMP atomics: single thread only


def main():
    import test_oracle as T
    from helpers import O, pack_golden

    K = T.REF if T.REF is not None else O
    out = {"source": np.array("reference" if K is not O else "restatement")}
    for name, n_det, n_samp in T.POINTING_CASES:
        out.update(pack_golden(f"pointing_{name}", T.pointing_outputs(K, name, n_det, n_samp)))
    out.update(pack_golden("solver_chain", T.solver_chain_outputs(K)))
    out.update(pack_golden("covariance", T.covariance_outputs(K)))
    inv, rc = T.eigendecompose_outputs(K)
    out["eigendecompose/inverse"] = inv
    out["eigendecompose/rcond"] = rc
    np.savez_compressed(T.CHECKS, **out)
    print(str(out["source"]), len(out), "entries,", os.path.getsize(T.CHECKS), "bytes")


if __name__ == "__main__":
    main()
