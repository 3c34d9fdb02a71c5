"""GPU tests of the global motion check (KLTB200SetMotionCheck, include/klt_b200.h;
csrc/klt_motion.cuh).  Teacher-forced: a twin context with the check off gives the tracker's results,
and those with the start positions are the oracle's input (tests/motion_oracle.py), so nothing here
depends on tracker parity."""
import ctypes as C
import os

import numpy as np
import pytest

from tests import motion_oracle as mo
from tests.conftest import GOLDEN
from tests.gpu_common import params_from_tc
from tests.test_gpu_fb import PATHS

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def L(pkg):
    from importlib import import_module
    lib = import_module(pkg.__name__ + ".runtime").load()
    lib.require_gpu()
    lib.KLTSetVerbosity(0)
    return lib


def _pairs(capi, synth):
    t = [capi.read_pgm_numpy(os.path.join(GOLDEN, "images_traffic", "img%d.pgm" % i)) for i in (1, 2)]
    return {"scene": mo.scene(),
            "translation": (synth.frame(640, 480, seed=3, t=0.0), synth.frame(640, 480, seed=3, t=1.0)),
            "rotate_zoom": (synth.frame(640, 480, seed=4, t=0.0),
                            synth.frame(640, 480, seed=4, t=0.0, rot_deg=1.5, scale=1.02)),
            "traffic": (t[0], t[1])}


def _call(L, capi, tc, a, b, x, y, v):
    fl = L.KLTCreateFeatureList(len(x))
    capi.arrays_to_featurelist(fl, x, y, v)
    L.track(tc, a, b, fl)
    out = capi.featurelist_to_arrays(fl)
    L.KLTFreeFeatureList(fl)
    return out


def _twins(L, setup=None, exact=0, max_error=1.0, hyps=0, fb=0.0):
    res = []
    for on in (0, 1):
        tc = L.KLTCreateTrackingContext()
        if setup:
            setup(L, tc)
        L.KLTB200SetExact(tc, exact)
        L.KLTB200SetForwardBackward(tc, fb)
        L.KLTB200SetMotionCheck(tc, max_error if on else 0.0, hyps)
        res.append(tc)
    return res


def _forced(L, capi, oracle, a, b, n=300, exact=0, max_error=1.0, hyps=0, setup=None):
    """-> (start, twin result, checked result, err, model, counts, oracle run)"""
    off, on = _twins(L, setup, exact, max_error, hyps)
    p = params_from_tc(oracle, off)
    x0, y0, v0 = oracle.select(a, p, n)
    v0[::17] = -2; x0[::17] = -1.0; y0[::17] = -1.0            # lost on entry: not a correspondence
    t = _call(L, capi, off, a, b, x0, y0, v0)
    g = _call(L, capi, on, a, b, x0, y0, v0)
    err = L.motion_result(on, len(x0))
    model = L.motion_models(on, 1)
    m, counts = L.dev_motion_counts(L.KLTB200Device(on), hyps or 1024)
    r = mo.motion_check(x0, y0, v0, *t, a.shape[1], a.shape[0], max_error, hyps or 1024)
    for tc in (off, on):
        L.KLTFreeTrackingContext(tc)
    return (x0, y0, v0), t, g, err, model, (m, counts), r


@pytest.mark.parametrize("exact", [0, 1])
def test_matches_oracle(L, capi, oracle, exact):
    import importlib
    synth = importlib.import_module("klt-feature-tracker-acceleration-gpus_b200.synth")
    near_total = 0
    for name, (a, b) in _pairs(capi, synth).items():
        s, t, g, err, model, (m, counts), r = _forced(L, capi, oracle, a, b, exact=exact)
        # bit-exact intermediate state: m, every hypothesis' count, the winner, validity
        assert m == r["m"] and model["tracked"][0] == r["m"], name
        assert np.array_equal(counts, r["counts"]), (name, np.nonzero(counts != r["counts"])[0][:8])
        assert model["hypothesis"][0] == r["winner"] and model["valid"][0] == r["valid"], name
        assert r["valid"] == 1, name
        # refined model: the corners within 1e-3 px of the oracle's
        c = mo.corners(a.shape[1], a.shape[0])
        assert np.abs(mo.project(model["H"][0], c) - mo.project(r["H"], c)).max() <= 1e-3, name
        # final classification: identical except next to the threshold
        near = np.abs(r["d2"].astype(np.float64) - r["e2"]) <= 1e-3 * r["e2"]
        near_total += int(near.sum())
        assert near.mean() < 0.005, name
        idx = r["idx"]
        gv, ov = g[2][idx], r["out"][2][idx]
        assert np.array_equal(gv[~near], ov[~near]), name
        assert model["inliers"][0] == int((gv == 0).sum()), name
        # everything else is the twin's result, and err is the oracle's within the model's tolerance
        assert np.array_equal(g[2][g[2] != mo.MOTION_OUTLIER], t[2][g[2] != mo.MOTION_OUTLIER]), name
        other = np.setdiff1d(np.arange(len(err)), idx)
        assert (err[other] == -1).all(), name
        assert np.abs(err[idx] - r["err"][idx]).max() <= 2e-3, name
    print("motion check (exact=%d): %d correspondences within 1e-3 relative of max_error^2" % (exact, near_total))


@pytest.mark.parametrize("exact", [0, 1])
@pytest.mark.parametrize("path", sorted(PATHS) + ["fb", "velocity"])
def test_check_only_removes(L, capi, oracle, path, exact):
    a, b = mo.scene()
    setup = {"fb": lambda L, tc: L.KLTB200SetForwardBackward(tc, 0.5),
             "velocity": lambda L, tc: L.KLTB200SetPrediction(tc, 1)}.get(path) or PATHS[path]
    off, on = _twins(L, setup, exact, fb=0.5 if path == "fb" else 0.0)
    p = params_from_tc(oracle, off)
    x0, y0, v0 = oracle.select(a, p, 400)
    v0[::13] = -3; x0[::13] = -1.0; y0[::13] = -1.0
    t = _call(L, capi, off, a, b, x0, y0, v0)
    g = _call(L, capi, on, a, b, x0, y0, v0)
    out = g[2] == mo.MOTION_OUTLIER
    assert out.sum() > 0 and (g[0][out] == -1).all() and (g[1][out] == -1).all()
    assert (t[2][out] == 0).all() and (v0[out] >= 0).all()
    keep = ~out
    assert g[0][keep].tobytes() == t[0][keep].tobytes() and g[1][keep].tobytes() == t[1][keep].tobytes()
    assert np.array_equal(g[2][keep], t[2][keep])
    for tc in (off, on):
        L.KLTFreeTrackingContext(tc)


def test_effect_scenario(L, capi, oracle):
    a, b = mo.scene()
    off, on = _twins(L)
    p = params_from_tc(oracle, off)
    x0, y0, v0 = oracle.select(a, p, 300)
    t = _call(L, capi, off, a, b, x0, y0, v0)
    g = _call(L, capi, on, a, b, x0, y0, v0)
    rect, bg = mo.scene_groups(x0, y0, t[0], t[1], (v0 >= 0) & (t[2] == 0), p.window_width // 2)
    flagged = g[2] == mo.MOTION_OUTLIER
    assert rect.sum() >= 10 and bg.sum() >= 150
    assert flagged[rect].mean() >= 0.9 and flagged[bg].mean() <= 0.01
    c = mo.corners(mo.SCENE_W, mo.SCENE_H)
    H = L.motion_models(on, 1)["H"][0]
    assert np.abs(mo.project(H, c) - mo.project(mo.scene_homography(), c)).max() <= 0.25
    for tc in (off, on):
        L.KLTFreeTrackingContext(tc)


def _frames(synth, k=6):
    return [synth.frame(320, 240, seed=9, t=0.7 * i, rot_deg=0.4 * i, scale=1.0 + 0.004 * i) for i in range(k)]


def _loop(L, capi, tc, frames, x, y, v, replace):
    fl = L.KLTCreateFeatureList(len(x))
    capi.arrays_to_featurelist(fl, x, y, v)
    table = []
    for k in range(1, len(frames)):
        L.track(tc, frames[k - 1], frames[k], fl)
        if replace:
            L.replace(tc, frames[k], fl)
        table.append(capi.featurelist_to_arrays(fl))
    final = capi.featurelist_to_arrays(fl)
    L.KLTFreeFeatureList(fl)
    return table, final


@pytest.mark.parametrize("affine", [0, 1])
@pytest.mark.parametrize("replace", [0, 1])
def test_sequence_matches_per_call_loop(L, capi, oracle, replace, affine):
    import importlib
    synth = importlib.import_module("klt-feature-tracker-acceleration-gpus_b200.synth")
    frames = _frames(synth)
    res = []
    for how in ("loop", "sequence"):
        tc = L.KLTCreateTrackingContext()
        tc.contents.sequentialMode = 1
        if affine:
            tc.contents.affineConsistencyCheck = 1
        L.KLTB200SetMotionCheck(tc, 0.5, 256)
        fl0 = L.KLTCreateFeatureList(200)
        L.select(tc, frames[0], fl0)
        x, y, v = capi.featurelist_to_arrays(fl0)
        L.KLTFreeFeatureList(fl0)
        if how == "loop":
            table, final = _loop(L, capi, tc, frames, x, y, v, replace)
        else:
            fl = L.KLTCreateFeatureList(len(x))
            capi.arrays_to_featurelist(fl, x, y, v)
            ft = L.KLTCreateFeatureTable(len(frames), len(x))
            L.track_sequence(tc, frames, fl, ft, 0, replace=bool(replace))
            tab = capi.featuretable_to_array(ft)
            table = [(tab["x"][:, k].copy(), tab["y"][:, k].copy(), tab["val"][:, k].copy())
                     for k in range(1, len(frames))]
            final = capi.featurelist_to_arrays(fl)
            L.KLTFreeFeatureTable(ft); L.KLTFreeFeatureList(fl)
        models = L.motion_models(tc, len(frames) - 1)
        res.append((table, final, models))
        L.KLTFreeTrackingContext(tc)
    (ta, fa, ma), (tb, fb, mb) = res
    for k, (ca, cb) in enumerate(zip(ta, tb)):
        for u, w in zip(ca, cb):
            assert u.tobytes() == w.tobytes(), "frame %d" % (k + 1)
    for u, w in zip(fa, fb):
        assert u.tobytes() == w.tobytes()
    for key in ma:
        assert ma[key].tobytes() == mb[key].tobytes(), key
    assert (ma["valid"] == 1).all()


def test_resident_matches_per_call_loop(L, capi):
    import importlib
    synth = importlib.import_module("klt-feature-tracker-acceleration-gpus_b200.synth")
    frames = _frames(synth)
    res = []
    for how in ("loop", "resident"):
        tc = L.KLTCreateTrackingContext()
        tc.contents.sequentialMode = 1
        L.KLTB200SetMotionCheck(tc, 0.5, 0)
        fl = L.KLTCreateFeatureList(300)
        L.select(tc, frames[0], fl)
        x, y, v = capi.featurelist_to_arrays(fl)
        if how == "loop":
            _, final = _loop(L, capi, tc, frames, x, y, v, 0)
        else:
            L.KLTB200ResidentBegin(tc, frames[0].ctypes.data, 0, 320, 320, 240, fl)
            for f in frames[1:]:
                L.KLTB200ResidentStep(tc, f.ctypes.data, 0, 320, 320, 240)
            L.KLTB200ResidentEnd(tc, fl)
            final = capi.featurelist_to_arrays(fl)
        res.append((final, L.motion_models(tc, len(frames) - 1), L.motion_result(tc, 300)))
        L.KLTFreeFeatureList(fl)
        L.KLTFreeTrackingContext(tc)
    (fa, ma, ea), (fb, mb, eb) = res
    for u, w in zip(fa, fb):
        assert u.tobytes() == w.tobytes()
    for key in ma:
        assert ma[key].tobytes() == mb[key].tobytes(), key
    assert ea.tobytes() == eb.tobytes()


def test_edge_cases(L, capi):
    import importlib
    synth = importlib.import_module("klt-feature-tracker-acceleration-gpus_b200.synth")
    a, b = synth.frame(320, 240, seed=5, t=0.0), synth.frame(320, 240, seed=5, t=1.0)
    tc = L.KLTCreateTrackingContext()
    L.KLTB200SetMotionCheck(tc, 1.0, 0)
    # n = 0
    fl = L.KLTCreateFeatureList(0)
    L.track(tc, a, b, fl)
    L.KLTFreeFeatureList(fl)
    mdl = L.motion_models(tc, 1)
    assert mdl["valid"][0] == 0 and mdl["tracked"][0] == 0 and mdl["hypothesis"][0] == -1
    assert np.isnan(mdl["H"][0]).all()
    # all features lost on entry; then m < 8
    for lost in (20, 14):
        x = np.linspace(40, 280, 20).astype(np.float32); y = np.full(20, 120.0, np.float32)
        v = np.zeros(20, np.int32); v[:lost] = -1
        g = _call(L, capi, tc, a, b, x, y, v)
        mdl = L.motion_models(tc, 1)
        assert mdl["valid"][0] == 0 and mdl["tracked"][0] <= 20 - lost
        assert (g[2] != mo.MOTION_OUTLIER).all()
        assert (L.motion_result(tc, 20)[:lost] == -1).all()
    # constant frames: nothing tracks, no model, nothing dropped
    c = np.full((240, 320), 128, np.uint8)
    x = np.linspace(40, 280, 50).astype(np.float32); y = np.linspace(40, 200, 50).astype(np.float32)
    g = _call(L, capi, tc, c, c, x, y, np.zeros(50, np.int32))
    mdl = L.motion_models(tc, 1)
    assert mdl["valid"][0] == 0 and (g[2] != mo.MOTION_OUTLIER).all()
    # history: 4 checked calls so far; more fails, a call without the check clears it
    assert len(L.motion_models(tc, 4)["valid"]) == 4
    with pytest.raises(RuntimeError):
        L.dev_motion_models(L.KLTB200Device(tc), 5)
    with pytest.raises(RuntimeError):                    # the last call had 50 features
        L.dev_motion_results(L.KLTB200Device(tc), 51)
    assert len(L.dev_motion_results(L.KLTB200Device(tc), 50)) == 50
    L.KLTB200SetMotionCheck(tc, 0.0, 0)
    _call(L, capi, tc, a, b, x, y, np.zeros(50, np.int32))
    with pytest.raises(RuntimeError):
        L.dev_motion_models(L.KLTB200Device(tc), 1)
    with pytest.raises(RuntimeError):
        L.dev_motion_results(L.KLTB200Device(tc), 50)
    L.KLTFreeTrackingContext(tc)


def test_guard_mode(L, capi, oracle):
    a, b = mo.scene()
    tc = L.KLTCreateTrackingContext()
    dev = L.KLTB200Device(tc)
    L.klt_dev_set_guard(dev, 1)
    L.KLTB200SetMotionCheck(tc, 1.0, 300)
    p = params_from_tc(oracle, tc)
    xs, ys, vs = oracle.select(a, p, 1200)
    rng = np.random.default_rng(1)
    for n in (1, 7, 1025, 5000):
        k = rng.integers(0, len(xs), n)
        x, y, v = xs[k].copy(), ys[k].copy(), vs[k].copy()
        _call(L, capi, tc, a, b, x, y, v)
        L.motion_result(tc, n)
    damaged, first = C.c_longlong(0), C.c_int(0)
    L.dev_check(dev, L.klt_dev_check_guards(dev, C.byref(damaged), C.byref(first)))
    assert damaged.value == 0
    assert len(L.motion_models(tc, 4)["valid"]) == 4
    L.KLTFreeTrackingContext(tc)


def test_launch_count(L, capi, oracle):
    a, b = mo.scene()
    tc = L.KLTCreateTrackingContext()
    p = params_from_tc(oracle, tc)
    x, y, v = oracle.select(a, p, 300)
    dev = L.KLTB200Device(tc)
    per = []
    for e in (0.0, 1.0, 0.0, 1.0):
        L.KLTB200SetMotionCheck(tc, e, 0)
        c0 = L.klt_dev_launch_count(dev)
        _call(L, capi, tc, a, b, x, y, v)
        per.append(L.klt_dev_launch_count(dev) - c0)
    assert per[0] == per[2] and per[1] == per[3] == per[0] + 3
    L.KLTFreeTrackingContext(tc)
