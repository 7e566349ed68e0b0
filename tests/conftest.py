import os
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]
# random-init parity experiments: both sides tokenize with the same deterministic stand-in (arp_b200/tokenizer.py)
os.environ.setdefault("ARP_ALLOW_STANDIN_TOKENIZER", "1")
for p in (str(ROOT), str(ROOT / "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")
    config.addinivalue_line("markers", "reference: needs /root/reference mounted (build container only)")


def pytest_collection_modifyitems(config, items):
    import torch
    from oracle import stubs
    has_gpu = torch.cuda.is_available()
    ref = stubs.reference_available()
    for item in items:
        if "gpu" in item.keywords and not has_gpu:
            item.add_marker(pytest.mark.skip(reason="no CUDA device"))
        if "reference" in item.keywords and not ref:
            item.add_marker(pytest.mark.skip(reason="/root/reference not mounted"))


@pytest.fixture(scope="session")
def built_lib():
    """The native library, built in-tree (nvcc cross-compiles without a GPU)."""
    from arp_b200.build import build
    return build()
