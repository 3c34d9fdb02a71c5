"""Host side of the motion prior (KLTB200SetPrediction, include/klt_b200.h) and its oracle
(tests/predict_oracle.py): no GPU needed.  The mode setter only touches the context's state record,
so nothing here creates a device."""
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.predict_oracle import pan_frames, pan_survival, track_guided

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def L(pkg):
    from importlib import import_module
    lib = import_module(pkg.__name__ + ".runtime").load()
    lib.KLTSetVerbosity(0)
    return lib


def _run(code, env_extra=None):
    env = dict(os.environ)
    env.pop("KLT_B200_PREDICT", None)
    env.update(env_extra or {})
    code = ("import importlib,numpy as np;"
            "m=importlib.import_module('klt-feature-tracker-acceleration-gpus_b200.runtime');"
            "L=m.load();L.KLTSetVerbosity(0);" + code)
    return subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, env=env)


def test_set_get_round_trip(L):
    tc = L.KLTCreateTrackingContext()
    assert L.KLTB200GetPrediction(tc) == 0                  # off by default
    for m in (1, 0, 1):
        L.KLTB200SetPrediction(tc, m)
        assert L.KLTB200GetPrediction(tc) == m
    L.KLTFreeTrackingContext(tc)


def test_bad_mode_is_refused():
    r = _run("tc=L.KLTCreateTrackingContext();L.KLTB200SetPrediction(tc,2);print('SURVIVED')")
    assert r.returncode == 1
    assert "KLT Error" in r.stderr and "SURVIVED" not in r.stdout


@pytest.mark.parametrize("value,mode", [("velocity", 1), ("none", 0)])
def test_environment_default(value, mode):
    r = _run("tc=L.KLTCreateTrackingContext();print(L.KLTB200GetPrediction(tc))", {"KLT_B200_PREDICT": value})
    assert r.returncode == 0, r.stderr
    assert int(r.stdout.split()[-1]) == mode


def test_environment_bad_value_is_refused():
    r = _run("tc=L.KLTCreateTrackingContext();L.KLTB200GetPrediction(tc);print('SURVIVED')",
             {"KLT_B200_PREDICT": "imu"})
    assert r.returncode == 1
    assert "KLT Error" in r.stderr and "SURVIVED" not in r.stdout


def test_result_without_a_predicted_call_fails():
    r = _run("tc=L.KLTCreateTrackingContext();L.prediction(tc,4);print('SURVIVED')")
    assert r.returncode == 1
    assert "KLT Error" in r.stderr and "SURVIVED" not in r.stdout


@pytest.mark.parametrize("lighting", [0, 1])
def test_guess_at_start_equals_oracle_track(oracle, capi, provided, lighting):
    """the composed descent with g = x0 is klto_track, bit for bit, on real frames"""
    p = oracle.default_params()
    p.lighting_insensitive = lighting
    x, y, v = oracle.select(provided[0], p, 300)
    v[::13] = -1
    p1, p2 = oracle.build_pyramids(provided[0], p), oracle.build_pyramids(provided[1], p)
    want = oracle.track(p1, p2, p, x, y, v)
    got = track_guided(oracle, p1, p2, p, x, y, v, x, y)
    assert all(u.tobytes() == w.tobytes() for u, w in zip(got, want))
    nan = np.full(len(x), np.nan, np.float32)
    got = track_guided(oracle, p1, p2, p, x, y, v, nan, nan)
    assert all(u.tobytes() == w.tobytes() for u, w in zip(got, want))
    assert (want[2] == 0).sum() > 200


def test_velocity_keeps_features_on_a_fast_pan(oracle, oracle_mod):
    """3 px/frame^2 up to 48 px/frame at 640x480 with the default context (2 levels, subsampling 4,
    7x7), 300 features, no replacement: tracked results summed over 16 frame pairs were 2733 without
    the prior and 3375 with it"""
    frames, _ = pan_frames(accel=3, frames=17)
    off = pan_survival(oracle, oracle_mod, frames, 300, velocity=False, replace=False)
    on = pan_survival(oracle, oracle_mod, frames, 300, velocity=True, replace=False)
    assert off <= 2800 and on >= 3300 and on >= 1.2 * off, (off, on)
