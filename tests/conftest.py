import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200, sm_100a); run with -m gpu on the GPU box")


@pytest.fixture(scope="session")
def golden():
    import json
    import numpy as np
    with np.load(os.path.join(ROOT, "tests", "golden", "unet_sampler_golden.npz")) as z:
        g = dict(z)
    # the tiny-UNet inputs are not stored: tests/golden/make_golden.py drew them first from default_rng(7), so they are
    # regenerated bit for bit, as the weights are from their seeds
    rng = np.random.default_rng(7)
    for tag in ("tiny", "tiny_cond", "tiny_sr"):
        cfg = json.loads(bytes(g[f"{tag}_cfg"]).decode())
        S = cfg["image_size"]
        g[f"{tag}_x"] = rng.standard_normal((len(g[f"{tag}_t"]), cfg["in_channels"], S, S)).astype(np.float32)
    return g


@pytest.fixture(scope="session", autouse=True)
def _built_library():
    """Build (or reuse) the in-tree sm_100a library once per session; nvcc cross-compiles without a GPU."""
    from ivid_b200 import build
    build.build()
