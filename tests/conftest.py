import hashlib
import json
import os
import shutil
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
# Q3_CKPT_DIR: keep the exported synthetic checkpoints between sessions (by default each session exports its own into a
# temporary directory that it removes at the end)
CKPT_DIR = os.environ.get("Q3_CKPT_DIR")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "slow: multi-GB checkpoints / long CPU oracle runs")


def _sha(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for blk in iter(lambda: f.read(1 << 20), b""):
            h.update(blk)
    return h.hexdigest()


@pytest.fixture(scope="session")
def golden():
    return np.load(os.path.join(GOLDEN_DIR, "golden.npz"))


@pytest.fixture(scope="session")
def golden_meta():
    with open(os.path.join(GOLDEN_DIR, "golden_meta.json")) as f:
        return json.load(f)


@pytest.fixture(scope="session")
def ckpt(tmp_path_factory):
    """ckpt(shape_name, group_size, seed) -> path of the exported synthetic checkpoint (cached)."""
    from qwen3_rs_b200 import synth

    d = CKPT_DIR or str(tmp_path_factory.mktemp("ckpt"))
    os.makedirs(d, exist_ok=True)

    def get(name: str, gs: int = 64, seed: int = 0) -> str:
        if (name, gs, seed) == ("micro", 32, 7):
            return os.path.join(GOLDEN_DIR, "micro_gs32.bin")
        path = os.path.join(d, f"{name}_gs{gs}_s{seed}.bin")
        want = synth.checkpoint_bytes(synth.SHAPES[name], gs)
        if not (os.path.exists(path) and os.path.getsize(path) == want):
            tmp = path + f".tmp{os.getpid()}"
            synth.export_synthetic(synth.SHAPES[name], tmp, gs, seed=seed)
            os.replace(tmp, path)
        return path

    yield get
    if not CKPT_DIR:
        shutil.rmtree(d, ignore_errors=True)  # the Qwen3-0.6B checkpoint alone is 0.6 GB


GOLDEN_CASES = [("micro", 32, 7), ("tiny", 64, 0), ("tiny-untied", 64, 1), ("small", 128, 2)]


def has_cuda() -> bool:
    try:
        import torch

        return torch.cuda.is_available()
    except Exception:
        return False
