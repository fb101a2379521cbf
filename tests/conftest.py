"""Shared pytest plumbing: the ``gpu`` marker, repo-root imports and the golden fixtures."""
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import golden_files  # noqa: E402

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden():
    """(arrays, meta) produced by oracle/make_golden.py from the unmodified reference."""
    arrays = golden_files.load(GOLDEN_DIR, "rawboost_golden")
    with open(os.path.join(GOLDEN_DIR, "rawboost_golden.json")) as f:
        meta = json.load(f)
    return arrays, meta


def stream_digest():
    """Same fingerprint of the global numpy stream that make_golden.py records."""
    import hashlib
    _, key, pos, has_gauss, cached = np.random.get_state()
    return {
        "pos": int(pos),
        "key_sha1": hashlib.sha1(np.asarray(key, dtype=np.uint32).tobytes()).hexdigest(),
        "has_gauss": int(has_gauss),
        "cached_gaussian": float(cached),
    }


@pytest.fixture(scope="session")
def golden2():
    """Round-2 fixtures (oracle/make_golden.py --round2): inputs above full scale, float64 / zero / NaN inputs, utterances
    longer than 65536 samples, the reverb augmentor and whole Dataset items -- all from the unmodified reference."""
    arrays = golden_files.load(GOLDEN_DIR, "round2_golden")
    with open(os.path.join(GOLDEN_DIR, "round2_golden.json")) as f:
        meta = json.load(f)
    return arrays, meta


def sha1_of(a):
    import hashlib
    return hashlib.sha1(np.ascontiguousarray(a).tobytes()).hexdigest()
