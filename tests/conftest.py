import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

ORACLE_LIB = os.path.join(ROOT, "oracle", "_ref", "libsailor_pt_ref.so")
ORACLE_COUNT_LIB = os.path.join(ROOT, "oracle", "_ref", "libsailor_pt_ref_count.so")
REFERENCE = "/root/reference"


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def _build_oracle_if_possible():
    if os.path.exists(ORACLE_LIB) and os.path.exists(ORACLE_COUNT_LIB):
        return True
    if os.path.isdir(os.path.join(REFERENCE, "Runtime", "Raytracing")):
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import build_ref
        build_ref.build(REFERENCE, False)
        build_ref.build(REFERENCE, True)
        return True
    return False


@pytest.fixture
def oracle(request):
    """The reference's own code behind the C-ABI (test checker).  Where it cannot be built, its recorded results stand in
    (tests/recorded_oracle.py), computed by the library a GPU test checks or else by the host-compiled kernel bodies."""
    from sailor_b200.capi import Library
    import recorded_oracle
    return recorded_oracle.for_tests(Library(ORACLE_LIB) if _build_oracle_if_possible() else None,
                                     lambda: request.getfixturevalue("gpu" if request.node.get_closest_marker("gpu") else "emu"))


@pytest.fixture(scope="session")
def oracle_count():
    from sailor_b200.capi import Library
    if not _build_oracle_if_possible():
        pytest.skip("oracle not available")
    return Library(ORACLE_COUNT_LIB)


@pytest.fixture(scope="session")
def emu():
    """Kernel bodies + host orchestration compiled for the host (tests/emu); a test tool, not a product path."""
    from sailor_b200.capi import Library
    sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
    import build_emu
    # SAILOR_EMU_LIB: another build of the same sources, e.g. one compiled with -fsanitize=address (tools/asan_emu.sh)
    return Library(os.environ.get("SAILOR_EMU_LIB") or build_emu.build())


@pytest.fixture(scope="session")
def gpu():
    """The product library. No skip when CUDA is missing: a GPU test without the CUDA path must fail loudly."""
    import sailor_b200
    from sailor_b200 import build as product_build
    product_build.build()
    return sailor_b200.library()


@pytest.fixture(scope="session")
def G():
    return np.load(os.path.join(ROOT, "tests", "golden", "golden.npz"))


@pytest.fixture(scope="session")
def digests():
    return json.load(open(os.path.join(ROOT, "tests", "golden", "digests.json")))


@pytest.fixture(scope="session")
def scene_dir(tmp_path_factory):
    return str(tmp_path_factory.mktemp("scenes"))
