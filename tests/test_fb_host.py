"""Host side of the forward-backward check (KLTB200SetForwardBackward, include/klt_b200.h) and its
oracle (tests/fb_oracle.py): no GPU needed.  The setter only touches the context's state record, so
nothing here creates a device."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.conftest import synth_image
from tests.fb_oracle import track_fb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def L(pkg):
    from importlib import import_module
    lib = import_module(pkg.__name__ + ".runtime").load()
    lib.KLTSetVerbosity(0)
    return lib


def _run(code, env_extra=None):
    env = dict(os.environ)
    env.pop("KLT_B200_FB_MAX_ERROR", None)
    env.update(env_extra or {})
    code = ("import importlib,numpy as np;"
            "m=importlib.import_module('klt-feature-tracker-acceleration-gpus_b200.runtime');"
            "L=m.load();L.KLTSetVerbosity(0);" + code)
    return subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, env=env)


def test_set_get_round_trip(L):
    tc = L.KLTCreateTrackingContext()
    assert L.KLTB200GetForwardBackward(tc) == 0.0           # off by default
    for v in (0.5, 1.0, -2.0, 0.0, math.inf):
        L.KLTB200SetForwardBackward(tc, v)
        assert L.KLTB200GetForwardBackward(tc) == np.float32(v)
    L.KLTFreeTrackingContext(tc)


def test_environment_default():
    r = _run("tc=L.KLTCreateTrackingContext();print(L.KLTB200GetForwardBackward(tc))",
             {"KLT_B200_FB_MAX_ERROR": "0.75"})
    assert r.returncode == 0, r.stderr
    assert float(r.stdout.split()[-1]) == 0.75
    r = _run("tc=L.KLTCreateTrackingContext();print(L.KLTB200GetForwardBackward(tc))",
             {"KLT_B200_FB_MAX_ERROR": "inf"})
    assert r.returncode == 0 and r.stdout.split()[-1] == "inf", r.stderr


@pytest.mark.parametrize("how", ["setter", "environment"])
def test_nan_is_refused(how):
    if how == "setter":
        r = _run("tc=L.KLTCreateTrackingContext();L.KLTB200SetForwardBackward(tc,float('nan'));print('SURVIVED')")
    else:
        r = _run("tc=L.KLTCreateTrackingContext();L.KLTB200GetForwardBackward(tc);print('SURVIVED')",
                 {"KLT_B200_FB_MAX_ERROR": "nan"})
    assert r.returncode == 1
    assert "KLT Error" in r.stderr and "SURVIVED" not in r.stdout


def test_result_without_a_checked_call_fails():
    r = _run("tc=L.KLTCreateTrackingContext();L.KLTB200SetForwardBackward(tc,1.0);"
             "L.forward_backward(tc,4);print('SURVIVED')")
    assert r.returncode == 1
    assert "KLT Error" in r.stderr and "SURVIVED" not in r.stdout


def test_oracle_track_fb_infinite_threshold_keeps_every_round_trip(oracle):
    """max_error = inf on a pure translation: a feature is dropped exactly when its backward leg
    fails; everything kept is the forward leg's answer, with the round-trip distance recorded."""
    img1 = synth_image(160, 120, 3)
    img2 = synth_image(160, 120, 3, shift=(1.3, -0.7))
    p = oracle.default_params()
    oracle.change_pyramid(p, 15)
    oracle.update_border(p)
    x0, y0, v0 = oracle.select(img1, p, 60)
    pyr1, pyr2 = oracle.build_pyramids(img1, p), oracle.build_pyramids(img2, p)
    xf, yf, vf = oracle.track(pyr1, pyr2, p, x0, y0, v0)
    x, y, v, xb, yb, err, bv = track_fb(oracle, pyr1, pyr2, p, x0, y0, v0, math.inf)
    fwd = vf == 0
    assert fwd.sum() > 30
    assert np.array_equal(bv[~fwd], np.ones((~fwd).sum(), np.int32))
    assert (err[~fwd] == -1).all() and (xb[~fwd] == -1).all()
    kept = fwd & (bv == 0)
    assert kept.sum() > 30
    assert x[kept].tobytes() == xf[kept].tobytes() and y[kept].tobytes() == yf[kept].tobytes()
    assert (v[kept] == 0).all() and (v[fwd & (bv != 0)] == -6).all()
    assert np.array_equal(v[~fwd], vf[~fwd])
    dx, dy = xb[kept] - x0[kept], yb[kept] - y0[kept]
    assert err[kept].tobytes() == np.sqrt(dx * dx + dy * dy).tobytes()
    assert float(err[kept].max()) < 0.1            # a clean translation comes home
    # a threshold below every round-trip distance rejects every feature the forward leg kept
    _, _, v2, _, _, _, _ = track_fb(oracle, pyr1, pyr2, p, x0, y0, v0, 1e-9)
    assert (v2[kept & (err > 1e-9)] == -6).all()
