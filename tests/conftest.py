import os
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def built():
    """Builds (if stale) and returns the two shared libraries."""
    import __graft_entry__ as g

    return {"cuda": g.build_cuda(), "oracle": g.build_oracle()}


@pytest.fixture(scope="session")
def oracle_lib(built):
    from pokegym_b200 import _capi

    return _capi.GbEnvLib(built["oracle"], "oracle_")


@pytest.fixture(scope="session")
def cuda_lib(built):
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pokegym_b200 import _capi

    return _capi.GbEnvLib(built["cuda"], "gbenv_")


@pytest.fixture(scope="session")
def roms():
    from pokegym_b200.tools import synth_rom

    cache = {}

    def get(name):
        if name not in cache:
            fn, kw = synth_rom.rom_catalog()[name]
            cache[name] = fn(**kw)
        return cache[name]

    return get
