"""GPU tests of the motion prior (KLTB200SetPrediction / KLTB200SetGuesses, include/klt_b200.h): the
descent starts from a per-feature guess inside the tracker's own launch (csrc/klt_dev.cu track_kernel,
csrc/klt_track_fast.cuh track_fast_kernel / track7w_kernel, PRED = true).

Exact mode is compared bit for bit with the oracle's composition of the guided descent
(tests/predict_oracle.py); fma mode goes through the usual parity gate with the same guesses."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.conftest import synth_image
from tests.gpu_common import check_fma_step, params_from_tc
from tests.predict_oracle import (EXPLICIT, NONE, VELOCITY, VelocityDriver, pan_frames, track_fb_guided,
                                  track_guided)
from tests.test_gpu_fb import PATHS, _set_window, occluded_pair

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def L(pkg):
    from importlib import import_module
    lib = import_module(pkg.__name__ + ".runtime").load()
    lib.require_gpu()
    lib.KLTSetVerbosity(0)
    return lib


def _call(L, capi, tc, img1, img2, x, y, v, gx=None, gy=None):
    """one KLTTrackFeatures call, with explicit guesses when given -> (x, y, val)"""
    fl = L.KLTCreateFeatureList(len(x))
    capi.arrays_to_featurelist(fl, x, y, v)
    if gx is not None:
        L.set_guesses(tc, gx, gy)
    L.track(tc, img1, img2, fl)
    out = capi.featurelist_to_arrays(fl)
    L.KLTFreeFeatureList(fl)
    return out


def shift_pair(w=640, h=480, dx=40.0, seed=3):
    """frame 2 is frame 1 moved by -dx in x: too far for the default pyramid alone"""
    return synth_image(w, h, seed), synth_image(w, h, seed, shift=(dx, 0.0))


def _pairs(capi, provided):
    from tests.conftest import GOLDEN
    t = [capi.read_pgm_numpy(os.path.join(GOLDEN, "images_traffic", "img%d.pgm" % i)) for i in (1, 2)]
    return {"provided": (provided[0], provided[1], 0.0), "traffic": (t[0], t[1], 0.0),
            "shift40": shift_pair() + (-40.0,)}


def _guesses(x, y, v, motion, seed=0, spread=1.5):
    """x0 + the true motion + noise; NaN (no guess) for every 7th feature"""
    rng = np.random.default_rng(seed)
    gx = (x + np.float32(motion) + rng.uniform(-spread, spread, len(x))).astype(np.float32)
    gy = (y + rng.uniform(-spread, spread, len(x))).astype(np.float32)
    gx[::7] = np.nan
    return gx, gy


def _expected_records(x, y, v, gx, gy):
    has = np.isfinite(gx) & np.isfinite(gy) & (v >= 0)
    return (np.where(has, gx, np.float32(-1)).astype(np.float32), np.where(has, gy, np.float32(-1)).astype(np.float32),
            np.where(has, EXPLICIT, NONE).astype(np.int32))


@pytest.mark.parametrize("fb", [0.0, 0.5])
@pytest.mark.parametrize("exact", [0, 1])
@pytest.mark.parametrize("path", sorted(PATHS))
def test_guess_at_start_is_identity(L, capi, oracle, path, exact, fb):
    a, b = occluded_pair(640, 480, seed=5)
    res, launches = [], []
    for guided in (False, True):
        tc = L.KLTCreateTrackingContext()
        PATHS[path](L, tc)
        L.KLTB200SetExact(tc, exact)
        L.KLTB200SetForwardBackward(tc, fb)
        p = params_from_tc(oracle, tc)
        x, y, v = oracle.select(a, p, 600)
        v[::11] = -3; x[::11] = -1.0; y[::11] = -1.0
        dev = L.KLTB200Device(tc)
        _call(L, capi, tc, a, b, x, y, v)                       # warm: buffers allocated
        c0 = L.klt_dev_launch_count(dev)
        res.append(_call(L, capi, tc, a, b, x, y, v, *((x, y) if guided else (None, None))))
        launches.append(L.klt_dev_launch_count(dev) - c0)
        if guided:
            gx, gy, src = L.prediction(tc, len(x))
            assert np.array_equal(src, np.where(v >= 0, EXPLICIT, NONE))
        L.KLTFreeTrackingContext(tc)
    assert all(u.tobytes() == w.tobytes() for u, w in zip(*res)), path
    assert launches[0] == launches[1] > 0
    assert (res[0][2] == 0).sum() > 300


@pytest.mark.parametrize("config", ["default", "lighting", "window9", "window7x9"])
def test_exact_mode_matches_oracle(L, capi, oracle, provided, config):
    seen = {"only_with_guess": 0, "guess_left_frame": 0}
    for name, (a, b, motion) in _pairs(capi, provided).items():
        tc = L.KLTCreateTrackingContext()
        L.KLTB200SetExact(tc, 1)
        if config == "lighting":
            tc.contents.lighting_insensitive = 1
        elif config == "window9":
            _set_window(L, tc, 9, 9)
        elif config == "window7x9":
            _set_window(L, tc, 7, 9)
        p = params_from_tc(oracle, tc)
        x, y, v = oracle.select(a, p, 300)
        gx, gy = _guesses(x, y, v, motion, seed=len(name))
        p1, p2 = oracle.build_pyramids(a, p), oracle.build_pyramids(b, p)
        got = _call(L, capi, tc, a, b, x, y, v, gx, gy)
        want = track_guided(oracle, p1, p2, p, x, y, v, gx, gy)
        for k, what in enumerate(("x", "y", "val")):
            assert got[k].tobytes() == want[k].tobytes(), (name, what, np.nonzero(got[k] != want[k])[0][:8])
        rec = L.prediction(tc, len(x))
        assert all(u.tobytes() == w.tobytes() for u, w in zip(rec, _expected_records(x, y, v, gx, gy)))
        plain = oracle.track(p1, p2, p, x, y, v)[2]
        g = np.isfinite(gx)
        seen["only_with_guess"] += int((g & (got[2] == 0) & (plain != 0)).sum())
        seen["guess_left_frame"] += int((g & (got[2] == -4) & (gx < p.borderx)).sum())
        L.KLTFreeTrackingContext(tc)
    assert min(seen.values()) > 0, seen


class _Guided:
    """an oracle whose track() starts each feature from its guess, looked up by its start position"""

    def __init__(self, oracle, x, y, gx, gy):
        self.o = oracle
        self.g = {(float(a), float(b)): (c, d) for a, b, c, d in zip(x, y, gx, gy)}

    def track(self, p1, p2, p, x, y, v):
        nan = np.float32(np.nan)
        g = [self.g.get((float(a), float(b)), (nan, nan)) for a, b in zip(x, y)]
        gx = np.array([q[0] for q in g], np.float32); gy = np.array([q[1] for q in g], np.float32)
        return track_guided(self.o, p1, p2, p, x, y, v, gx, gy)

    def __getattr__(self, k):
        return getattr(self.o, k)


@pytest.mark.parametrize("path", sorted(PATHS))
def test_fma_mode_parity(L, capi, oracle, provided, path):
    for a, b, motion in (shift_pair() + (-40.0,), (provided[0], provided[1], 0.0)):
        tc = L.KLTCreateTrackingContext()
        PATHS[path](L, tc)
        p = params_from_tc(oracle, tc)
        x, y, v = oracle.select(a, p, 400)
        gx, gy = _guesses(x, y, v, motion, seed=1, spread=0.8)
        gv = _call(L, capi, tc, a, b, x, y, v, gx, gy)
        p1, p2 = oracle.build_pyramids(a, p), oracle.build_pyramids(b, p)
        g = _Guided(oracle, x, y, gx, gy)
        ox, oy, ov = g.track(p1, p2, p, x, y, v)
        check_fma_step(g, p, p1, p2, x, y, v, gv[0], gv[1], gv[2], ox, oy, ov, path)
        L.KLTFreeTrackingContext(tc)


def test_forward_backward_with_guesses(L, capi, oracle, provided):
    for name, (a, b, motion) in _pairs(capi, provided).items():
        tc = L.KLTCreateTrackingContext()
        L.KLTB200SetExact(tc, 1)
        L.KLTB200SetForwardBackward(tc, 0.5)
        p = params_from_tc(oracle, tc)
        x, y, v = oracle.select(a, p, 300)
        gx, gy = _guesses(x, y, v, motion, seed=2)
        got = _call(L, capi, tc, a, b, x, y, v, gx, gy) + L.forward_backward(tc, len(x))
        p1, p2 = oracle.build_pyramids(a, p), oracle.build_pyramids(b, p)
        want = track_fb_guided(oracle, p1, p2, p, x, y, v, gx, gy, 0.5)
        for k, what in enumerate(("x", "y", "val", "xb", "yb", "err", "back_val")):
            assert got[k].tobytes() == want[k].tobytes(), (name, what, np.nonzero(got[k] != want[k])[0][:8])
        rec = L.prediction(tc, len(x))
        assert all(u.tobytes() == w.tobytes() for u, w in zip(rec, _expected_records(x, y, v, gx, gy)))
        if name == "shift40":
            assert (got[2] == 0).sum() > 100
        L.KLTFreeTrackingContext(tc)


@pytest.mark.parametrize("replace", [False, True])
def test_velocity_loop_matches_oracle(L, capi, oracle, oracle_mod, replace):
    frames, _ = pan_frames(accel=3, frames=13)
    n = 300
    tc = L.KLTCreateTrackingContext()
    L.KLTB200SetExact(tc, 1)
    L.KLTB200SetPrediction(tc, 1)
    p = params_from_tc(oracle, tc)
    x, y, v = oracle.select(frames[0], p, n, sort_kind=oracle_mod.SORT_STABLE)
    drv = VelocityDriver(n)
    prev = oracle.build_pyramids(frames[0], p)
    sources = np.zeros(3, int)
    for k in range(1, len(frames)):
        if k == 6:                                   # the caller moves some features: no velocity for them
            x[3::17] = np.where(v[3::17] == 0, x[3::17] + np.float32(0.25), x[3::17])
        cur = oracle.build_pyramids(frames[k], p)
        gx0 = _call(L, capi, tc, frames[k - 1], frames[k], x, y, v)
        grec = L.prediction(tc, n)
        (ox, oy, ov), orec = drv.step(oracle, prev, cur, p, x, y, v)
        for u, w, what in zip(gx0 + grec, (ox, oy, ov) + orec, ("x", "y", "val", "gx", "gy", "source")):
            assert u.tobytes() == w.tobytes(), (k, what, np.nonzero(u != w)[0][:8])
        moved = np.zeros(n, bool)
        if k == 6:
            moved[3::17] = v[3::17] == 0
            assert moved.any() and (grec[2][moved] == NONE).all()
        if replace and k > 1:
            assert (grec[2][v > 0] == NONE).all()
        sources += np.bincount(grec[2], minlength=3)
        x, y, v = ox, oy, ov
        if replace:
            x, y, v = oracle.select(frames[k], p, n, sort_kind=oracle_mod.SORT_STABLE, replace=True,
                                    last=cur, x=x, y=y, val=v)
            assert (v > 0).any()
        prev = cur
    assert sources[VELOCITY] > 1000, sources
    # a change of frame size forgets every velocity
    small = [f[:240, :320].copy() for f in frames[-2:]]
    xs, ys, vs = oracle.select(small[0], p, n)
    _call(L, capi, tc, small[0], small[1], xs, ys, vs)
    assert (L.prediction(tc, n)[2] == NONE).all()
    L.KLTFreeTrackingContext(tc)


def _loop(L, capi, frames, n, exact, replace, fb, affine):
    tc = L.KLTCreateTrackingContext()
    tc.contents.sequentialMode = 1
    if affine:
        tc.contents.affineConsistencyCheck = 2
    L.KLTB200SetExact(tc, exact)
    L.KLTB200SetForwardBackward(tc, fb)
    L.KLTB200SetPrediction(tc, 1)
    fl = L.KLTCreateFeatureList(n)
    ft = L.KLTCreateFeatureTable(len(frames), n)
    L.select(tc, frames[0], fl)
    L.KLTStoreFeatureList(fl, ft, 0)
    vel = 0
    for k in range(1, len(frames)):
        L.track(tc, frames[k - 1], frames[k], fl)
        rec = L.prediction(tc, n)
        vel += int((rec[2] == VELOCITY).sum())
        if replace:
            L.replace(tc, frames[k], fl)
        L.KLTStoreFeatureList(fl, ft, k)
    assert vel > 100, vel
    out = capi.featuretable_to_array(ft), capi.featurelist_to_arrays(fl), rec
    L.KLTFreeFeatureTable(ft)
    L.KLTFreeFeatureList(fl)
    L.KLTFreeTrackingContext(tc)
    return out


@pytest.mark.parametrize("exact", [0, 1])
@pytest.mark.parametrize("variant", ["plain", "replace", "fb", "affine"])
def test_sequence_call_equals_per_call_loop(L, capi, exact, variant):
    frames, _ = pan_frames(accel=3, frames=11)
    n = 200
    replace, fb, affine = variant == "replace", 0.3 if variant == "fb" else 0.0, variant == "affine"
    tab, fin, rec = _loop(L, capi, frames, n, exact, replace, fb, affine)
    tc = L.KLTCreateTrackingContext()
    tc.contents.sequentialMode = 1
    if affine:
        tc.contents.affineConsistencyCheck = 2
    L.KLTB200SetExact(tc, exact)
    L.KLTB200SetForwardBackward(tc, fb)
    L.KLTB200SetPrediction(tc, 1)
    fl = L.KLTCreateFeatureList(n)
    ft = L.KLTCreateFeatureTable(len(frames), n)
    L.select(tc, frames[0], fl)
    L.KLTStoreFeatureList(fl, ft, 0)
    L.track_sequence(tc, frames[:6], fl, ft, 0, replace)
    L.track_sequence(tc, frames[5:], fl, ft, 5, replace)
    assert capi.featuretable_to_array(ft).tobytes() == tab.tobytes()
    assert all(u.tobytes() == w.tobytes() for u, w in zip(capi.featurelist_to_arrays(fl), fin))
    assert all(u.tobytes() == w.tobytes() for u, w in zip(L.prediction(tc, n), rec))
    L.KLTFreeFeatureTable(ft)
    L.KLTFreeFeatureList(fl)
    L.KLTFreeTrackingContext(tc)


@pytest.mark.parametrize("exact", [0, 1])
def test_resident_pipeline_equals_per_call_loop(L, capi, exact):
    frames, _ = pan_frames(accel=3, frames=11)
    n = 200
    tab, fin, rec = _loop(L, capi, frames, n, exact, False, 0.3, False)
    tc = L.KLTCreateTrackingContext()
    tc.contents.sequentialMode = 1
    L.KLTB200SetExact(tc, exact)
    L.KLTB200SetForwardBackward(tc, 0.3)
    L.KLTB200SetPrediction(tc, 1)
    fl = L.KLTCreateFeatureList(n)
    L.select(tc, frames[0], fl)
    h, w = frames[0].shape
    L.KLTB200ResidentBegin(tc, frames[0].ctypes.data, 0, w, w, h, fl)
    for k in range(1, len(frames)):
        L.KLTB200ResidentStep(tc, frames[k].ctypes.data, 0, w, w, h)
    L.KLTB200ResidentEnd(tc, fl)
    assert all(u.tobytes() == w_.tobytes() for u, w_ in zip(capi.featurelist_to_arrays(fl), fin))
    assert all(u.tobytes() == w_.tobytes() for u, w_ in zip(L.prediction(tc, n), rec))
    L.KLTFreeFeatureList(fl)
    L.KLTFreeTrackingContext(tc)


@pytest.mark.parametrize("source", ["host", "tensor"])
def test_explicit_guesses_through_resident_step(L, capi, source):
    """an IMU-style prior: each frame's guesses are the start positions moved by the known pan"""
    import torch
    frames, motion = pan_frames(accel=4, frames=9)
    n = 200
    h, w = frames[0].shape
    # the per-call loop: its start positions give the guesses the resident run is handed
    tc = L.KLTCreateTrackingContext()
    tc.contents.sequentialMode = 1
    fl = L.KLTCreateFeatureList(n)
    L.select(tc, frames[0], fl)
    guesses, recs = [], []
    for k in range(1, len(frames)):
        x, y, _ = capi.featurelist_to_arrays(fl)
        guesses.append(((x + np.float32(motion[k])).astype(np.float32), y.copy()))
        L.set_guesses(tc, *guesses[-1])
        L.track(tc, frames[k - 1], frames[k], fl)
        recs.append(L.prediction(tc, n))
    want = capi.featurelist_to_arrays(fl)
    L.KLTFreeFeatureList(fl)
    L.KLTFreeTrackingContext(tc)
    assert (want[2] == 0).sum() > 50

    tc = L.KLTCreateTrackingContext()
    tc.contents.sequentialMode = 1
    fl = L.KLTCreateFeatureList(n)
    L.select(tc, frames[0], fl)
    L.KLTB200ResidentBegin(tc, frames[0].ctypes.data, 0, w, w, h, fl)
    keep = []
    for k in range(1, len(frames)):
        gx, gy = guesses[k - 1]
        if source == "tensor":
            tx, ty = torch.from_numpy(gx).cuda(), torch.from_numpy(gy).cuda()
            torch.cuda.synchronize()
            keep.append((tx, ty))
            L.set_guesses(tc, tx, ty, on_device=True)
        else:
            L.set_guesses(tc, gx, gy)
        L.KLTB200ResidentStep(tc, frames[k].ctypes.data, 0, w, w, h)
        got = L.prediction(tc, n)
        assert all(u.tobytes() == v.tobytes() for u, v in zip(got, recs[k - 1])), k
    L.KLTB200ResidentEnd(tc, fl)
    assert all(u.tobytes() == v.tobytes() for u, v in zip(capi.featurelist_to_arrays(fl), want))
    L.KLTFreeFeatureList(fl)
    L.KLTFreeTrackingContext(tc)


@pytest.mark.parametrize("source", ["host", "tensor"])
def test_explicit_guesses_queued_without_synchronisation(L, capi, source):
    """a pipelined driver: the guesses of every step are queued right behind the step before, nothing
    synchronises until the end, and each step's guesses differ from the last (an accelerating pan);
    the result equals the per-call loop's"""
    import torch
    frames, motion = pan_frames(accel=4, frames=13)
    n = 300
    h, w = frames[0].shape
    tc = L.KLTCreateTrackingContext()
    tc.contents.sequentialMode = 1
    fl = L.KLTCreateFeatureList(n)
    L.select(tc, frames[0], fl)
    x0, y0, v0 = capi.featurelist_to_arrays(fl)
    # guesses that depend on the step only, so that both runs can be handed them up front
    guesses = [((x0 + np.float32(sum(motion[1:k + 1]))).astype(np.float32), y0.copy()) for k in range(1, len(frames))]
    for k in range(1, len(frames)):
        L.set_guesses(tc, *guesses[k - 1])
        L.track(tc, frames[k - 1], frames[k], fl)
    want = capi.featurelist_to_arrays(fl)
    L.KLTFreeFeatureList(fl)
    L.KLTFreeTrackingContext(tc)
    assert (want[2] == 0).sum() > 50

    tc = L.KLTCreateTrackingContext()
    tc.contents.sequentialMode = 1
    fl = L.KLTCreateFeatureList(n)
    capi.arrays_to_featurelist(fl, x0, y0, v0)
    L.KLTB200ResidentBegin(tc, frames[0].ctypes.data, 0, w, w, h, fl)
    keep = []
    if source == "tensor":
        keep = [(torch.from_numpy(gx).cuda(), torch.from_numpy(gy).cuda()) for gx, gy in guesses]
        torch.cuda.synchronize()
    for k in range(1, len(frames)):
        if source == "tensor":
            L.set_guesses(tc, *keep[k - 1], on_device=True)
        else:
            L.set_guesses(tc, *guesses[k - 1])
        L.KLTB200ResidentStep(tc, frames[k].ctypes.data, 0, w, w, h)
    L.KLTB200ResidentEnd(tc, fl)
    assert all(u.tobytes() == v.tobytes() for u, v in zip(capi.featurelist_to_arrays(fl), want))
    L.KLTFreeFeatureList(fl)
    L.KLTFreeTrackingContext(tc)


def _run(code):
    env = dict(os.environ)
    env.pop("KLT_B200_PREDICT", None)
    code = ("import importlib,numpy as np;"
            "m=importlib.import_module('klt-feature-tracker-acceleration-gpus_b200.runtime');"
            "L=m.load();L.KLTSetVerbosity(0);"
            "rng=np.random.default_rng(0);"
            "a=(rng.random((120,160))*255).astype(np.uint8);b=np.roll(a,1,axis=1).copy();"
            "tc=L.KLTCreateTrackingContext();tc.contents.sequentialMode=1;fl=L.KLTCreateFeatureList(50);"
            "L.select(tc,a,fl);" + code)
    return subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, env=env)


@pytest.mark.parametrize("case", ["mismatched_n", "mismatched_n_resident", "sequence_with_guesses",
                                  "sequence_with_device_level_guesses"])
def test_errors(case):
    code = {
        "mismatched_n": "L.set_guesses(tc,np.zeros(3,np.float32),np.zeros(3,np.float32));L.track(tc,a,b,fl);",
        "mismatched_n_resident": ("L.KLTB200ResidentBegin(tc,a.ctypes.data,0,160,160,120,fl);"
                                  "L.set_guesses(tc,np.zeros(3,np.float32),np.zeros(3,np.float32));"
                                  "L.KLTB200ResidentStep(tc,b.ctypes.data,0,160,160,120);L.KLTB200ResidentEnd(tc,fl);"),
        "sequence_with_guesses": ("L.set_guesses(tc,np.zeros(50,np.float32),np.zeros(50,np.float32));"
                                  "L.track_sequence(tc,[a,b],fl);"),
        "sequence_with_device_level_guesses": ("g=np.zeros(50,np.float32);"
                                               "L.dev_check(L.KLTB200Device(tc),L.lib.klt_dev_set_guesses("
                                               "L.KLTB200Device(tc),50,g.ctypes.data,g.ctypes.data,0));"
                                               "L.track_sequence(tc,[a,b],fl);"),
    }[case]
    r = _run(code + "print('SURVIVED')")
    assert r.returncode == 1, (r.stdout, r.stderr)
    assert "KLT Error" in r.stderr and "SURVIVED" not in r.stdout


def test_guard_mode(L, capi):
    frames = [synth_image(643, 487, 5, shift=(9.0 * k, -1.3 * k)) for k in range(8)]
    tc = L.KLTCreateTrackingContext()
    tc.contents.sequentialMode = 1
    dev = L.KLTB200Device(tc)
    L.klt_dev_set_guard(dev, 1)
    L.KLTB200SetForwardBackward(tc, 0.2)
    L.KLTB200SetPrediction(tc, 1)
    fl = L.KLTCreateFeatureList(300)
    ft = L.KLTCreateFeatureTable(len(frames), 300)
    L.select(tc, frames[0], fl)
    for k in (1, 2, 3):
        x, y, _ = capi.featurelist_to_arrays(fl)
        if k == 2:
            L.set_guesses(tc, x - np.float32(9.0), y)
        L.track(tc, frames[k - 1], frames[k], fl)
        L.replace(tc, frames[k], fl)
    L.track_sequence(tc, frames[3:], fl, ft, 3, True)
    assert (L.prediction(tc, 300)[2] == VELOCITY).sum() > 50
    bad, band = C.c_longlong(-1), C.c_int(-1)
    assert L.klt_dev_check_guards(dev, C.byref(bad), C.byref(band)) == 0
    assert bad.value == 0, (bad.value, band.value)
    L.KLTFreeFeatureTable(ft)
    L.KLTFreeFeatureList(fl)
    L.KLTFreeTrackingContext(tc)
