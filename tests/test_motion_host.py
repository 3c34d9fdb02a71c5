"""Host side of the global motion check (KLTB200SetMotionCheck, include/klt_b200.h) and its oracle
(tests/motion_oracle.py): no GPU needed.  The setter only touches the context's state record, so
nothing here creates a device."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import motion_oracle as mo
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
    env.pop("KLT_B200_MOTION_MAX_ERROR", None)
    env.update(env_extra or {})
    code = ("import importlib,ctypes as C,numpy as np;"
            "m=importlib.import_module('klt-feature-tracker-acceleration-gpus_b200.runtime');"
            "L=m.load();L.KLTSetVerbosity(0);" + code)
    return subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, env=env)


def _get(L, tc):
    import ctypes as C
    h = C.c_int(0)
    return L.KLTB200GetMotionCheck(tc, C.byref(h)), h.value


def test_set_get_round_trip(L):
    tc = L.KLTCreateTrackingContext()
    assert _get(L, tc) == (0.0, 1024)                         # off by default, 1024 hypotheses
    for e, h, want in ((1.0, 0, 1024), (0.5, 1, 1), (2.5, 65536, 65536), (-1.0, 300, 300), (math.inf, 7, 7)):
        L.KLTB200SetMotionCheck(tc, e, h)
        assert _get(L, tc) == (np.float32(e), want)
    L.KLTFreeTrackingContext(tc)


def test_environment_default():
    r = _run("tc=L.KLTCreateTrackingContext();h=C.c_int(0);print(L.KLTB200GetMotionCheck(tc,C.byref(h)),h.value)",
             {"KLT_B200_MOTION_MAX_ERROR": "1.25"})
    assert r.returncode == 0, r.stderr
    assert r.stdout.split()[-2:] == ["1.25", "1024"]


@pytest.mark.parametrize("how", ["nan", "environment", "negative", "too_many"])
def test_bad_settings_are_refused(how):
    if how == "nan":
        r = _run("tc=L.KLTCreateTrackingContext();L.KLTB200SetMotionCheck(tc,float('nan'),0);print('SURVIVED')")
    elif how == "environment":
        r = _run("tc=L.KLTCreateTrackingContext();L.KLTB200GetMotionCheck(tc,None);print('SURVIVED')",
                 {"KLT_B200_MOTION_MAX_ERROR": "nan"})
    else:
        h = -1 if how == "negative" else 65537
        r = _run("tc=L.KLTCreateTrackingContext();L.KLTB200SetMotionCheck(tc,1.0,%d);print('SURVIVED')" % h)
    assert r.returncode == 1
    assert "KLT Error" in r.stderr and "SURVIVED" not in r.stdout


@pytest.mark.parametrize("call", ["result", "models"])
def test_results_without_a_checked_call_fail(call):
    what = "L.motion_result(tc,4)" if call == "result" else "L.motion_models(tc,1)"
    r = _run("tc=L.KLTCreateTrackingContext();L.KLTB200SetMotionCheck(tc,1.0,0);%s;print('SURVIVED')" % what)
    assert r.returncode == 1
    assert "KLT Error" in r.stderr and "SURVIVED" not in r.stdout


def test_sampler_is_reproducible():
    assert mo.mix32(0) == 0 and mo.mix32(1) != 1
    a = [mo.sample(h, 300) for h in range(64)]
    assert a == [mo.sample(h, 300) for h in range(64)]
    assert all(s is not None and len(set(s)) == 4 and max(s) < 300 for s in a)
    assert len({tuple(s) for s in a}) == 64                  # different hypotheses, different samples
    assert mo.sample(5, 0) is None and mo.sample(5, 3) is None


def test_minimal_solve_recovers_a_homography_with_outliers():
    """noise-free correspondences of a known homography, 30 % replaced by random ones: the check finds
    the model to the float32 resolution of its entries at the corners (the float64 solve before that
    rounding: 1e-6 px, next test) and drops exactly the replaced ones"""
    W, H = 640, 480
    Ht = mo.scene_homography()
    rng = np.random.default_rng(3)
    n = 400
    p0 = np.c_[rng.uniform(20, W - 20, n), rng.uniform(20, H - 20, n)].astype(np.float32)
    p1 = mo.project(Ht, p0.astype(np.float64))
    bad = rng.random(n) < 0.3
    p1[bad] += rng.uniform(-40, 40, (bad.sum(), 2))
    p1 = p1.astype(np.float32)
    v = np.zeros(n, np.int32)
    r = mo.motion_check(p0[:, 0], p0[:, 1], v, p1[:, 0], p1[:, 1], v, W, H, 0.5, 256)
    assert r["valid"] == 1 and r["m"] == n and r["refined"]
    c = mo.corners(W, H)
    assert np.abs(mo.project(r["H"], c) - mo.project(Ht, c)).max() < 1e-6 * 640 + 1e-4
    assert set(np.nonzero(r["out"][2] == mo.MOTION_OUTLIER)[0]) == set(np.nonzero(bad)[0])
    assert (r["err"][~bad] < 0.01).all()


def test_float64_solve_is_exact_before_rounding():
    Ht = mo.scene_homography()
    pts = np.array([[10.0, 20.0], [600.0, 40.0], [580.0, 450.0], [30.0, 400.0]])
    q = mo.project(Ht, pts)
    geo = mo.geometry(640, 480)
    A = []
    for (x, y), (u, v) in zip(pts, q):
        A += mo._rows(mo._norm(x, geo[0], geo[2]), mo._norm(y, geo[1], geo[2]),
                      mo._norm(u, geo[0], geo[2]), mo._norm(v, geo[1], geo[2]))
    n = mo.solve8(A)
    c = mo.corners(640, 480)
    Hd = np.array(n + [1.0]).reshape(3, 3)
    s, cx, cy = geo[2], geo[0], geo[1]
    T = np.array([[s, 0, -s * cx], [0, s, -s * cy], [0, 0, 1]])
    Hp = np.linalg.inv(T) @ Hd @ T
    assert np.abs(mo.project(Hp / Hp[2, 2], c) - mo.project(Ht, c)).max() < 1e-6


def test_degenerate_sample_is_rejected():
    # three collinear points in frame 1
    x = [mo._norm(v, 320.0, 1 / 320) for v in (100.0, 200.0, 300.0, 150.0)]
    y = [mo._norm(v, 240.0, 1 / 320) for v in (100.0, 100.0, 100.0, 300.0)]
    assert mo.degenerate(x, y)
    y[2] = mo._norm(101.0, 240.0, 1 / 320)
    assert not mo.degenerate(x, y)
    # every sample of collinear correspondences is rejected: no model, nothing dropped
    n = 50
    xs = np.linspace(10, 600, n).astype(np.float32)
    ys = (0.5 * xs + 20).astype(np.float32)
    v = np.zeros(n, np.int32)
    r = mo.motion_check(xs, ys, v, xs + 1, ys, v, 640, 480, 1.0, 64)
    assert r["winner"] == -1 and r["valid"] == 0 and (r["counts"] == -1).all()
    assert (r["out"][2] == 0).all() and (r["err"] == -1).all()


def test_effect_scenario(oracle):
    """640x480, 300 features, the default context, max_error 1.0: the check drops the features on the
    moving rectangle and keeps the background; the forward-backward check alone keeps the rectangle"""
    img1, img2 = mo.scene()
    p = oracle.default_params()
    x0, y0, v0 = oracle.select(img1, p, 300)
    pyr1, pyr2 = oracle.build_pyramids(img1, p), oracle.build_pyramids(img2, p)
    x1, y1, v1 = oracle.track(pyr1, pyr2, p, x0, y0, v0)
    r = mo.motion_check(x0, y0, v0, x1, y1, v1, mo.SCENE_W, mo.SCENE_H, 1.0)
    rect, bg = mo.scene_groups(x0, y0, x1, y1, (v0 >= 0) & (v1 == 0), p.window_width // 2)
    flagged = r["out"][2] == mo.MOTION_OUTLIER
    assert rect.sum() >= 10 and bg.sum() >= 150
    assert flagged[rect].mean() >= 0.9
    assert flagged[bg].mean() <= 0.01
    c = mo.corners(mo.SCENE_W, mo.SCENE_H)
    assert np.abs(mo.project(r["H"], c) - mo.project(mo.scene_homography(), c)).max() <= 0.25
    _, _, vf, _, _, _, _ = track_fb(oracle, pyr1, pyr2, p, x0, y0, v0, 0.5)
    assert (vf[rect] == 0).mean() >= 0.8        # consistent forward and back: only the global model sees them
