import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE, os.path.join(HERE, "golden")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def fixtures():
    import golden_store
    return golden_store.load("fixtures")


@pytest.fixture(scope="session")
def golden():
    import golden_store
    return golden_store.load("golden_ref")


def case_inputs(name, fixtures, golden):
    """(gn, psf, bkg, divergence, kwargs) of a parity case; flux / betaParam of the synthetic cases come
    from the golden file (they were arguments of the reference run)."""
    from cases import CASES
    dkey, div, kw, _ = CASES[name]
    kw = dict(kw)
    if dkey.startswith("tile"):
        base = f"tile{(int(dkey[4:]) // 5) * 5}"
        gn, psf, bkg = fixtures[base + "/gn"], fixtures["tile0/psf"], fixtures[base + "/bkg"]
    elif dkey.startswith("cutout31_"):
        gn, psf, bkg = fixtures[dkey + "/gn"], fixtures["cutout31_0/psf"], fixtures[dkey + "/bkg"]
    else:
        gn, psf, bkg = fixtures[dkey + "/gn"], fixtures[dkey + "/psf"], fixtures[dkey + "/bkg"]
    if name + "/flux_in" in golden.files:
        kw["flux"] = np.float64(golden[name + "/flux_in"])
    if name + "/beta0" in golden.files:
        kw["betaParam"] = float(golden[name + "/beta0"])
    if bkg.ndim == 0:
        bkg = np.float64(bkg)
    return gn, psf, bkg, div, kw


@pytest.fixture(scope="session")
def get_case(fixtures, golden):
    return lambda name: case_inputs(name, fixtures, golden)
