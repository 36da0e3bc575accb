import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def ref_lib():
    """oracle/_ref/libenv_ref.so — prebuilt by __graft_entry__.build(); rebuilt here if the reference is present."""
    from oracle import build_ref
    from oracle.ref_env import REF_LIB

    if not os.path.exists(REF_LIB):
        if not build_ref.reference_available():
            pytest.skip("oracle/_ref not built and reference tree absent")
        build_ref.build()
    return REF_LIB


@pytest.fixture(scope="session")
def asset_pack():
    from procgen_b200 import assets

    if not os.path.exists(assets.DEFAULT_PACK):
        assets.build_pack_from_images()
    return assets.DEFAULT_PACK


@pytest.fixture(scope="session")
def hostsim_lib(asset_pack):
    """CPU debug build of the device code (tests only; the package never loads it)."""
    from procgen_b200 import build as B

    return B.build_hostsim()


@pytest.fixture(scope="session")
def product_lib():
    from procgen_b200 import build as B

    # never test a library older than the sources it was built from
    if B.needs_build():
        B.build_library()
    return B.LIB_PATH
