import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    # torch CPU ops crawl when they spawn one thread per hardware thread of a 100+ core box
    import torch

    torch.set_num_threads(min(16, os.cpu_count() or 1))
    config.addinivalue_line("markers", "gpu: needs a CUDA (sm_100a) device; run with -m gpu on the B200 box")


def ckpt_path(name: str, seed: int = 0) -> str:
    from beat_this_b200 import synthetic

    return synthetic.write_checkpoint(os.path.join(synthetic.cache_dir(), f"{name}_s{seed}.ckpt"), name, seed)


@pytest.fixture(scope="session")
def small0_ckpt():
    return ckpt_path("small0")


@pytest.fixture(scope="session")
def final0_ckpt():
    return ckpt_path("final0")


@pytest.fixture(scope="session")
def lib_built():
    """The CUDA library, built in-tree if missing (nvcc cross-compiles without a GPU)."""
    from beat_this_b200 import _lib

    _lib.build()
    return _lib.load()
