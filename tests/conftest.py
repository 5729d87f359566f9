import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

GOLDEN = os.path.join(ROOT, "tests", "golden")
SCENES = ("small", "medium", "large")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu")


@pytest.fixture(scope="session")
def oracle():
    from cpu_checkers import Oracle
    return Oracle()


@pytest.fixture(scope="session")
def r1():
    import rays1bench_b200
    return rays1bench_b200


@pytest.fixture(scope="session")
def golden_rays():
    return {name: dict(np.load(os.path.join(GOLDEN, "rays_%s.npz" % name))) for name in SCENES + ("synth4096",)}


@pytest.fixture(scope="session")
def golden_render():
    return {name: dict(np.load(os.path.join(GOLDEN, "render_%s.npz" % name))) for name in SCENES + ("synth4096",)}


@pytest.fixture(scope="session")
def ref_stats():
    import json
    return json.load(open(os.path.join(GOLDEN, "ref_stats.json")))


def rmse(a, b):
    """per-channel RMSE in 8-bit units"""
    d = a.astype(np.float64) - b.astype(np.float64)
    return float(np.sqrt((d * d).mean()))
