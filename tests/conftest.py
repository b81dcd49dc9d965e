import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")
    config.addinivalue_line("markers", "slow: multi-GB allocations (full llama2-7B shape)")


@pytest.fixture(scope="session")
def stories15m():
    """The real 61 MB stories15M.bin, too large to keep in the repository: tests that need its
    trained weights run when it has been copied to assets/stories15M.bin."""
    p = os.path.join(ROOT, "assets", "stories15M.bin")
    if not os.path.exists(p):
        pytest.skip("stories15M.bin is not in assets/")
    return p


@pytest.fixture(scope="session")
def oracle():
    import oracle_lib
    oracle_lib.build_oracle()
    return oracle_lib


@pytest.fixture(scope="session")
def l2b():
    import llama2_zig_b200
    return llama2_zig_b200
