"""pytest configuration: the `gpu` marker and loaders for the package and the oracle.

`-m "not gpu"` tests run on a CPU-only box: oracle vs golden fixtures, host mirror vs oracle,
C-ABI symbol checks, gloo multi-process logic.  `-m gpu` tests are the parity tests proper and
call the CUDA path through the C ABI; they never read /root/reference.
"""
import importlib.util
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def load_agpt():
    """Import ag-pathtracer_b200/ (hyphenated directory) under the module name agpt_b200."""
    if "agpt_b200" in sys.modules:
        return sys.modules["agpt_b200"]
    pkg_dir = os.path.join(ROOT, "ag-pathtracer_b200")
    spec = importlib.util.spec_from_file_location("agpt_b200", os.path.join(pkg_dir, "__init__.py"),
                                                  submodule_search_locations=[pkg_dir])
    mod = importlib.util.module_from_spec(spec)
    sys.modules["agpt_b200"] = mod
    spec.loader.exec_module(mod)
    return mod


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def agpt():
    return load_agpt()


@pytest.fixture(scope="session")
def ref():
    from oracle import ref_binding
    if not ref_binding.available():
        pytest.skip("oracle/_ref/libagpt_ref.so not built (needs /root/reference at build time)")
    return ref_binding


@pytest.fixture(scope="session")
def ref_live():
    """The reference's own code where oracle/_ref is built, else None: the test then compares with what
    tests/golden/make_golden_fullsize.py stored (ref_golden)."""
    from oracle import ref_binding
    return ref_binding if ref_binding.available() else None


@pytest.fixture(scope="session")
def ref_golden():
    def load(name):
        g = np.load(os.path.join(ROOT, "tests", "golden", name))
        print(f"compared with tests/golden/{name} (source: {g['source']})")
        return g
    return load


@pytest.fixture(scope="session")
def gpu_ctx(agpt):
    if agpt.device_count() == 0:
        pytest.fail("no CUDA device visible: -m gpu tests must run on the GPU box")
    ctx = agpt.Context(0)
    yield ctx
    ctx.close()
