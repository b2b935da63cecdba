"""pytest configuration: the `gpu` marker, golden loaders, shared fixtures.

`-m "not gpu"` runs here (no GPU): oracle vs the reference-generated goldens, host logic,
C-ABI symbol checks, gloo world_size-2 paths.  `-m gpu` runs on a B200 and compares the
CUDA path (through the C-ABI) with the oracle and the goldens.  Every input is in the
repository (tests/golden) or generated from a seed.
"""
import json
import os
import sys

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)
GOLDEN = os.path.join(REPO, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); deselected on the CPU box")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        have_gpu = torch.cuda.is_available()
    except Exception:
        have_gpu = False
    for item in items:
        if "gpu" in item.keywords and not have_gpu:
            item.add_marker(pytest.mark.skip(reason="no CUDA device"))


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


@pytest.fixture(scope="session")
def word():
    """The bundled reference_word.wav (SURVEY §2 row 14) as float32 = int16/32768."""
    g = load_golden("reference_word.npz")
    return g["pcm_i16"].astype(np.float32) / np.float32(32768.0)


@pytest.fixture(scope="session")
def word_i16():
    return load_golden("reference_word.npz")["pcm_i16"]


@pytest.fixture(scope="session")
def golden_matcher():
    return load_golden("matcher.npz")


@pytest.fixture(scope="session")
def golden_detect():
    g = load_golden("detect.npz")
    cases = json.loads(str(g["cases_json"]))
    return g, cases


@pytest.fixture(scope="session")
def golden_dense():
    return load_golden("dense.npz")


@pytest.fixture(scope="session")
def golden_vad():
    return load_golden("vad.npz")
