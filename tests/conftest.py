import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


# `-m gpu -x` stops at the first failure: run the headline path first (encode parity, edge cases, user surface, Mixtral
# forward, KV cache), then the training path (backward, GradCache, joint step), so that a problem in a later stage never
# hides the evidence of an earlier one.  Stable within a file; CPU-only files keep their alphabetical order.
GPU_FILE_ORDER = ["test_gpu_parity.py", "test_gpu_edges.py", "test_gpu_surface.py", "test_gpu_mixtral.py", "test_gpu_kvcache.py",
                  "test_gpu_training.py", "test_gpu_backward.py", "test_gpu_gradcache.py", "test_gpu_decode_inplace.py",
                  "test_gpu_mixtral_backward.py", "test_gpu_p2p_gather.py", "test_gpu_devices.py"]


def pytest_collection_modifyitems(config, items):
    rank = {name: i for i, name in enumerate(GPU_FILE_ORDER)}
    items.sort(key=lambda it: rank.get(Path(str(it.fspath)).name, -1))   # list.sort is stable
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:  # pragma: no cover
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def golden():
    """The Mistral fixture of tests/golden/make_golden.py, stored as three archives to keep each file small."""
    import numpy as np
    out = {}
    for part in ("", "_eager", "_logits"):
        out.update(np.load(ROOT / "tests" / "golden" / f"gritlm_ref_tiny{part}.npz"))
    return out
