import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, "tests", "golden")
# The original project (fast_monte_carlo_cfb.py, sim_helpers.py, edge_finder.py, PregameSPPlus2025_1.csv and its model
# artifacts) is not part of this repository; the tests that run it side by side with ours need FMC_REFERENCE_DIR.
from oracle.ref_harness import REFERENCE_DIR as REFERENCE   # noqa: E402


def has_reference(name: str) -> bool:
    return bool(REFERENCE) and os.path.exists(os.path.join(REFERENCE, name))


NO_REFERENCE = "the original project is not here: set FMC_REFERENCE_DIR to its directory"


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (runs through the C-ABI / CUDA kernels)")


@pytest.fixture(scope="session")
def models():
    from fast_monte_carlo_b200 import artifacts as art
    return art.load_default_models()


@pytest.fixture(scope="session")
def models_s2(models):
    from fast_monte_carlo_b200 import synth
    return synth.with_synthetic_stage2(models)


@pytest.fixture(scope="session")
def oracle(models_s2):
    """The C oracle with every forest (incl. the synthetic stage 2) loaded."""
    from oracle import c_oracle as co
    co.build()
    co.load_models(models_s2)
    return co


@pytest.fixture(scope="session")
def native_lib():
    from fast_monte_carlo_b200 import build, native
    build.build()
    return native.load_library()


@pytest.fixture(scope="session")
def engine(models_s2, native_lib):
    """GPU engine with the shipped configuration (heuristic play-call, stage-2 stand-in)."""
    from fast_monte_carlo_b200.engine import Engine
    e = Engine(models_s2, device=0, stage2="standin")
    yield e
    e.close()


KSU = (15.6, 35.7, 20.0)
ISU = (11.0, 31.5, 20.6)
