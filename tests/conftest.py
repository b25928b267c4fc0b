import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "spff-unet-spcct_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)


@pytest.fixture
def reference_threads():
    """Run on 8 intra-op threads, the count the reference's golden vectors were computed with. Torch's CPU reductions
    (float64 sums, convolution weight gradients) split their work by thread count; the init checksums are compared
    bit for bit, and the small bottleneck gradients of the golden cases are ill-conditioned enough that another split
    moves single entries past their elementwise tolerance.

    The 8 is not recorded in the golden files: oracle/make_golden*.py run on `torch.set_num_threads(os.cpu_count())`,
    and the host that wrote tests/golden/init_seed42.npz and case*.npz had 8 cores (with 8 threads these tests pass,
    with 1, 4 or 16 they do not). Goldens regenerated on another host need this count changed to that host's."""
    import torch

    n = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(n)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (sm_100) GPU; run with -m gpu on the GPU box")


def pytest_collection_modifyitems(config, items):
    try:
        import torch

        has_gpu = torch.cuda.is_available()
    except Exception:  # pragma: no cover
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)
