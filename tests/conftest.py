import os
import sys
import tempfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# the remote code of converted checkpoints that transformers caches (``trust_remote_code``) goes to a temporary directory, not
# to a home directory that may not be writable; set here, before any test imports transformers, so that sub-processes inherit it
os.environ["HF_HOME"] = os.path.join(tempfile.gettempdir(), f"internevo-tests-hf-{os.getuid()}")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `pytest -m gpu`)")


def pytest_collection_modifyitems(config, items):
    import torch

    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(autouse=True)
def _restore_global_config():
    """Tests that run in-process (no spawned ranks) set partial configs on the global context; give every test the config it
    found so the outcome does not depend on which tests share an xdist worker."""
    from internevo_b200.core.context import global_context as gpc

    saved = gpc._config
    yield
    gpc._config = saved
