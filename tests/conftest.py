import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_report_header(config):
    import oracle
    if oracle.have_reference():
        return "parity comparator (ref_planner): the compiled unmodified reference, oracle/_ref"
    return ("parity comparator (ref_planner): the C restatement oracle/dymu_oracle.c "
            "(oracle/_ref not built)")


@pytest.fixture(scope="session")
def pkg():
    import dymu_b200
    return dymu_b200.load()


@pytest.fixture(scope="session")
def oracle_mod():
    import oracle
    oracle.build(ref=True, port=True)
    return oracle


@pytest.fixture(scope="session")
def ref_lib(oracle_mod):
    if not oracle_mod.have_reference():
        pytest.skip("oracle/_ref/libdymu_ref.so not built (needs /root/reference at build time)")
    return oracle_mod.reference()


@pytest.fixture(scope="session")
def ref_planner(oracle_mod):
    """Planner factory the GPU parity tests compare with: the compiled unmodified reference where
    it is built, otherwise the plain-C restatement oracle/dymu_oracle.c, which reproduces the
    reference's stored outputs bit for bit (tests/test_golden_cpu.py) and is pinned against the
    compiled reference by tests/test_oracle_vs_reference.py where that is built.  The report
    header names the one in use."""
    if oracle_mod.have_reference():
        return oracle_mod.reference().DyMuPathPlanner
    return oracle_mod.Port


def rel_err(a, b):
    """max |a-b| / |b| over cells where b is finite and non-zero; masks must agree."""
    a, b = np.asarray(a), np.asarray(b)
    fin = np.isfinite(b) & (b != 0)
    if not fin.any():
        return 0.0
    return float(np.max(np.abs(a[fin] - b[fin]) / np.abs(b[fin])))
