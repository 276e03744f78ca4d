import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


# product defaults of the per-thread library options (api.cu); a test that changes one must put it back
OPTION_DEFAULTS = {"gemm": 0, "corr": 0, "attn": 0, "prec.corr": 2, "prec.fc1": 3, "fuse": 1}


@pytest.fixture(autouse=True)
def _options_do_not_leak(request):
    """GPU tests share one process: a leaked verification option would silently move every later test off the
    product path.  After each gpu-marked test the options must be back at their defaults."""
    yield
    if request.node.get_closest_marker("gpu") is None:
        return
    from cotracker_b200 import engine
    leaked = {k: engine.get_option(k) for k in OPTION_DEFAULTS if engine.get_option(k) != OPTION_DEFAULTS[k]}
    for k in leaked:
        engine.set_option(k, OPTION_DEFAULTS[k])
    assert not leaked, f"{request.node.nodeid} left library options changed: {leaked}"
