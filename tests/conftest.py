import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box via gpurun)")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def load_golden(name):
    with np.load(os.path.join(GOLDEN, name), allow_pickle=False) as z:
        return {k: z[k] for k in z.files}


def golden_inputs(g):
    """The inputs of a reduced-size golden case (CPU tensors), re-drawn by synthetic.make_inputs from the stored
    seed and checked bit for bit against the stored SHA-256 of the inputs the golden results were computed on."""
    import hashlib
    from kccotgan_b200.synthetic import INPUT_ORDER, make_inputs
    inp = make_inputs(int(g["B"]), int(g["T"]), int(g["H"]), int(g["W"]), int(g["C"]), J=int(g["J"]), ctx=int(g["ctx"]),
                      kind=str(g["kind"]), seed=int(g["seed"]))
    for k in INPUT_ORDER:
        assert hashlib.sha256(inp[k].numpy().tobytes()).hexdigest() == str(g["sha256_" + k]), k
    return inp


def rel_l2(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    den = np.linalg.norm(b)
    return float(np.linalg.norm(a - b) / den) if den > 0 else float(np.linalg.norm(a - b))
