import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu under gpurun)")
    config.addinivalue_line("markers", "reference: needs /root/reference (build container only)")


def pytest_collection_modifyitems(config, items):
    import torch
    has_gpu = torch.cuda.is_available()
    skip_gpu = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords and not has_gpu:
            item.add_marker(skip_gpu)


@pytest.fixture(autouse=True)
def cpu_tests_build_on_the_cpu(request, monkeypatch):
    """A test not marked gpu runs on the CPU also where a GPU is visible: networks and models are created on the CPU
    (the package puts them on cuda whenever a GPU is present), as on a machine without one."""
    if request.node.get_closest_marker("gpu") is None:
        import torch
        from mra_gan_b200 import networks3D
        from mra_gan_b200.models import base_model
        monkeypatch.setattr(networks3D, "device", torch.device("cpu"))
        monkeypatch.setattr(base_model, "device", torch.device("cpu"))


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN
