import os
import sys

import pytest
import threadpoolctl

# The reference's CPU project_signal accumulates with OpenMP atomics (template_offset.cpp:
# 301-327): only a single-threaded oracle is deterministic / bit-comparable.
# Forced (not setdefault): a caller's OMP_NUM_THREADS > 1 would make the bit-for-bit checks against
# the compiled reference flaky.  TB_TEST_OMP_THREADS overrides it for experiments.
os.environ["OMP_NUM_THREADS"] = os.environ.get("TB_TEST_OMP_THREADS", "1")

# numpy's OpenBLAS splits a dot product of more than 10 000 elements into one partial sum per
# thread, so the oracle's PCG results on the larger golden fixtures (c2/c4/c5_wide) depend on its
# thread count: they were stored with 8 threads.  numpy is already loaded when this file runs, so
# the count is set through the library rather than through OPENBLAS_NUM_THREADS.
threadpoolctl.threadpool_limits(8, user_api="blas")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_sessionstart(session):
    """Build whatever is missing (nvcc cross-compiles without a GPU): the CUDA library, the
    pybind11 module and the oracle's C restatement.  `__graft_entry__.build()` does the same."""
    from toast_b200 import build as tb_build

    tb_build.build()
    tb_build.build_pybind()
    from oracle import toast_oracle

    toast_oracle.build()


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: test needs a CUDA device (run on the B200 box)")


def _has_gpu():
    try:
        from toast_b200 import lib

        return lib.accel_enabled()
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    # GPU tests are selected with `-m gpu`; when selected on a machine without a device they
    # fail loudly (no silent skip): the product has no CPU fallback.
    return
