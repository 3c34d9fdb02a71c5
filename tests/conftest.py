"""Shared fixtures.  GPU tests are marked @pytest.mark.gpu."""
import importlib
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")
PKG_NAME = "klt-feature-tracker-acceleration-gpus_b200"


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def load_pkg():
    return importlib.import_module(PKG_NAME)


@pytest.fixture(scope="session")
def pkg():
    return load_pkg()


@pytest.fixture(scope="session")
def capi(pkg):
    return pkg.capi


@pytest.fixture(scope="session")
def oracle():
    from oracle import oracle_py
    oracle_py.build()
    return oracle_py.Oracle()


@pytest.fixture(scope="session")
def oracle_mod():
    from oracle import oracle_py
    return oracle_py


@pytest.fixture(scope="session")
def provided(capi):
    """The 10 frames of data/images_provided (config 1), copied to tests/golden."""
    return [capi.read_pgm_numpy(os.path.join(GOLDEN, "images_provided", "img%d.pgm" % i))
            for i in range(10)]


@pytest.fixture(scope="session")
def golden_ft():
    raw = open(os.path.join(GOLDEN, "features2.ft"), "rb").read()
    assert raw[:6] == b"KLTFT1"
    nframes, nfeat = np.frombuffer(raw[6:14], np.int32)
    tab = np.frombuffer(raw[14:], dtype=[("x", "f4"), ("y", "f4"), ("val", "i4")])
    return raw, tab.reshape(nfeat, nframes)


def synth_image(w, h, seed, shift=(0.0, 0.0)):
    """Small smooth-ish random texture (numpy only) for stage tests."""
    rng = np.random.default_rng(seed)
    acc = np.zeros((h, w), np.float64)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float64)
    xx = xx + shift[0]
    yy = yy + shift[1]
    for cell, wgt in ((23, 0.5), (9, 0.3), (4, 0.2)):
        gw, gh = w // cell + 4, h // cell + 4
        lat = rng.random((gh, gw))
        fx, fy = xx / cell + 1.0, yy / cell + 1.0
        x0, y0 = np.floor(fx).astype(int), np.floor(fy).astype(int)
        ax, ay = fx - x0, fy - y0
        x0 = np.clip(x0, 0, gw - 2); y0 = np.clip(y0, 0, gh - 2)
        v = (lat[y0, x0] * (1 - ax) * (1 - ay) + lat[y0, x0 + 1] * ax * (1 - ay)
             + lat[y0 + 1, x0] * (1 - ax) * ay + lat[y0 + 1, x0 + 1] * ax * ay)
        acc += wgt * v
    return np.clip(acc * 255.0, 0, 255).astype(np.uint8)
