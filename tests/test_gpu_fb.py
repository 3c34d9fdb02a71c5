"""GPU tests of the forward-backward check (KLTB200SetForwardBackward, include/klt_b200.h): the
backward leg runs in the tracker's own launch (csrc/klt_dev.cu track_kernel, csrc/klt_track_fast.cuh
track_fast_kernel / track7w_kernel, FB = true).

Exact mode is compared bit for bit with the oracle's composition of two reference tracking calls
(tests/fb_oracle.py); fma mode keeps the usual parity gate on the backward leg; on every tracker path
the check may only remove features, by the float32 rule recomputed here."""
import ctypes as C
import math

import numpy as np
import pytest

from tests.conftest import synth_image
from tests.fb_oracle import track_fb
from tests.gpu_common import check_fma_step, params_from_tc

pytestmark = pytest.mark.gpu

FB_INCONSISTENT = -6


@pytest.fixture(scope="module")
def L(pkg):
    from importlib import import_module
    lib = import_module(pkg.__name__ + ".runtime").load()
    lib.require_gpu()
    lib.KLTSetVerbosity(0)
    return lib


def occluded_pair(w, h, seed=11):
    """a shifted synthetic texture whose frame 2 has a rectangle of another texture pasted in: features
    there track forward somewhere and fail or miss on the way back"""
    a = synth_image(w, h, seed)
    b = synth_image(w, h, seed, shift=(2.4, -1.7))
    o = synth_image(w, h, seed + 100)
    b[h // 4: h // 2, w // 3: 2 * w // 3] = o[h // 4: h // 2, w // 3: 2 * w // 3]
    return a, b


def _pairs(capi, provided):
    import os
    from tests.conftest import GOLDEN
    t = [capi.read_pgm_numpy(os.path.join(GOLDEN, "images_traffic", "img%d.pgm" % i)) for i in (1, 2)]
    return {"provided": (provided[0], provided[1]), "traffic": (t[0], t[1]), "occluded": occluded_pair(320, 240)}


def _call(L, capi, tc, img1, img2, x, y, v):
    """one KLTTrackFeatures call on the given features -> (x, y, val) and, with the check on, its records"""
    n = len(x)
    fl = L.KLTCreateFeatureList(n)
    capi.arrays_to_featurelist(fl, x, y, v)
    L.track(tc, img1, img2, fl)
    out = capi.featurelist_to_arrays(fl)
    L.KLTFreeFeatureList(fl)
    if L.KLTB200GetForwardBackward(tc) > 0:
        return out + L.forward_backward(tc, n)
    return out


def _decision(x0, y0, xb, yb, bv, max_error):
    """the float32 rule: kept <=> back_val == 0 and !(d2 > max_error^2); err = sqrt(d2)"""
    dx = (xb - x0).astype(np.float32); dy = (yb - y0).astype(np.float32)
    d2 = dx * dx + dy * dy
    keep = (bv == 0) & ~(d2 > np.float32(max_error) * np.float32(max_error))
    return keep, np.sqrt(d2)


def test_exact_mode_matches_oracle(L, capi, oracle, provided):
    seen = {"kept": 0, "distance": 0, "backward": 0}
    for name, (a, b) in _pairs(capi, provided).items():
        tc = L.KLTCreateTrackingContext()
        L.KLTB200SetExact(tc, 1)
        p = params_from_tc(oracle, tc)
        x, y, v = oracle.select(a, p, 300)
        p1, p2 = oracle.build_pyramids(a, p), oracle.build_pyramids(b, p)
        for t in (0.1, 1.0, math.inf):
            L.KLTB200SetForwardBackward(tc, t)
            g = _call(L, capi, tc, a, b, x, y, v)
            o = track_fb(oracle, p1, p2, p, x, y, v, t)
            for k, what in enumerate(("x", "y", "val", "xb", "yb", "err", "back_val")):
                assert g[k].tobytes() == o[k].tobytes(), (name, t, what, np.nonzero(g[k] != o[k])[0][:8])
            gv, bv = g[2], g[6]
            seen["kept"] += int(((gv == 0) & (bv == 0)).sum())
            seen["distance"] += int(((gv == FB_INCONSISTENT) & (bv == 0)).sum())
            seen["backward"] += int(((gv == FB_INCONSISTENT) & (bv < 0)).sum())
        L.KLTFreeTrackingContext(tc)
    assert min(seen.values()) > 0, seen


def _set_window(L, tc, w, h):
    tc.contents.window_width, tc.contents.window_height = w, h
    L.KLTUpdateTCBorder(tc)


PATHS = {
    "track7w": lambda L, tc: None,
    "track_fast7": lambda L, tc: L.klt_dev_disable_track7w(L.KLTB200Device(tc), 1),
    "track_fast5": lambda L, tc: _set_window(L, tc, 5, 5),
    "track_fast9": lambda L, tc: _set_window(L, tc, 9, 9),
    "track_fast15": lambda L, tc: _set_window(L, tc, 15, 15),
    "generic7x9": lambda L, tc: _set_window(L, tc, 7, 9),
    "force_generic": lambda L, tc: L.klt_dev_force_generic(L.KLTB200Device(tc), 1),
    "lighting": lambda L, tc: setattr(tc.contents, "lighting_insensitive", 1),
}


@pytest.mark.parametrize("exact", [0, 1])
@pytest.mark.parametrize("path", sorted(PATHS))
def test_check_only_removes(L, capi, oracle, path, exact):
    a, b = occluded_pair(640, 480, seed=5)
    res = []
    for t in (0.0, 0.5):
        tc = L.KLTCreateTrackingContext()
        PATHS[path](L, tc)
        L.KLTB200SetExact(tc, exact)
        L.KLTB200SetForwardBackward(tc, t)
        p = params_from_tc(oracle, tc)
        x, y, v = oracle.select(a, p, 600)
        v[::11] = -3; x[::11] = -1.0; y[::11] = -1.0           # lost on entry: not touched, not checked
        res.append(_call(L, capi, tc, a, b, x, y, v))
        L.KLTFreeTrackingContext(tc)
    (fx, fy, fv), (gx, gy, gv, xb, yb, err, bv) = res
    fwd = fv == 0
    assert fwd.sum() > 300 and (~fwd).sum() > 0
    same = (gx.tobytes() == fx.tobytes(), gy.tobytes() == fy.tobytes())
    assert np.array_equal(gv[~fwd], fv[~fwd]) and (bv[~fwd] == 1).all()
    assert (gx[~fwd] == fx[~fwd]).all() and (gy[~fwd] == fy[~fwd]).all() and (err[~fwd] == -1).all()
    kept = fwd & (gv == 0)
    rej = fwd & (gv == FB_INCONSISTENT)
    assert (kept | rej)[fwd].all()
    assert kept.sum() > 200 and rej.sum() > 0, (kept.sum(), rej.sum())
    assert (gx[kept] == fx[kept]).all() and (gy[kept] == fy[kept]).all(), same
    assert (bv[kept] == 0).all() and (err[kept] <= 0.5).all()
    assert (gx[rej] == -1).all() and (gy[rej] == -1).all()
    keep, e = _decision(x[fwd], y[fwd], xb[fwd], yb[fwd], bv[fwd], 0.5)
    assert np.array_equal(keep, kept[fwd])
    ok = bv[fwd] == 0
    assert err[fwd][ok].tobytes() == e[ok].tobytes()
    assert (err[fwd][~ok] == -1).all() and (xb[fwd][~ok] == -1).all()


def test_fma_backward_leg_matches_oracle(L, capi, oracle, provided):
    """the GPU's backward leg, teacher-forced from its own forward positions, through the fma gate"""
    for a, b in ((provided[0], provided[1]), occluded_pair(640, 480, seed=5)):
        tc = L.KLTCreateTrackingContext()
        p = params_from_tc(oracle, tc)
        x, y, v = oracle.select(a, p, 400)
        fl = L.KLTCreateFeatureList(len(x))
        capi.arrays_to_featurelist(fl, x, y, v)
        L.track(tc, a, b, fl)
        fx, fy, fv = capi.featurelist_to_arrays(fl)
        L.KLTFreeFeatureList(fl)
        L.KLTB200SetForwardBackward(tc, math.inf)
        gx, gy, gv, xb, yb, err, bv = _call(L, capi, tc, a, b, x, y, v)
        m = np.nonzero(bv != 1)[0]
        assert np.array_equal(m, np.nonzero(fv == 0)[0]) and len(m) > 200
        p1, p2 = oracle.build_pyramids(a, p), oracle.build_pyramids(b, p)
        z = np.zeros(len(m), np.int32)
        ox, oy, ov = oracle.track(p2, p1, p, fx[m], fy[m], z)
        check_fma_step(oracle, p, p2, p1, fx[m], fy[m], z, xb[m], yb[m], bv[m], ox, oy, ov, "backward leg")
        L.KLTFreeTrackingContext(tc)


def test_launch_count_unchanged(L, capi, provided):
    counts = []
    for t in (0.0, 0.5):
        tc = L.KLTCreateTrackingContext()
        tc.contents.sequentialMode = 1
        L.KLTB200SetForwardBackward(tc, t)
        dev = L.KLTB200Device(tc)
        fl = L.KLTCreateFeatureList(200)
        L.select(tc, provided[0], fl)
        L.track(tc, provided[0], provided[1], fl)
        c0 = L.klt_dev_launch_count(dev)
        L.track(tc, provided[1], provided[2], fl)
        counts.append(L.klt_dev_launch_count(dev) - c0)
        L.KLTFreeFeatureList(fl)
        L.KLTFreeTrackingContext(tc)
    assert counts[0] == counts[1] and counts[0] > 0, counts


class _FloatImage(C.Structure):
    _fields_ = [("ncols", C.c_int), ("nrows", C.c_int), ("data", C.POINTER(C.c_float))]


def _template(fl, i):
    r = fl.contents.feature[i].contents
    if not r.aff_img:
        return None
    return [np.ctypeslib.as_array(C.cast(q, C.POINTER(_FloatImage)).contents.data, shape=(17 * 17,)).copy()
            for q in (r.aff_img, r.aff_img_gradx, r.aff_img_grady)]


@pytest.mark.parametrize("exact", [0, 1])
@pytest.mark.parametrize("check", [0, 1, 2])
def test_affine_check_after_fb(L, capi, provided, check, exact):
    """frame 0 -> 1 without the check in both contexts, frame 1 -> 2 with it in one: a kept feature
    leaves what the check-off affine run leaves, a rejected one what a lost feature leaves"""
    lists, states = [], []
    for fb in (0.0, 0.1):
        tc = L.KLTCreateTrackingContext()
        tc.contents.sequentialMode = 1
        tc.contents.affineConsistencyCheck = check
        L.KLTB200SetExact(tc, exact)
        fl = L.KLTCreateFeatureList(150)
        L.select(tc, provided[0], fl)
        L.track(tc, provided[0], provided[1], fl)
        before = capi.featurelist_affine(fl)
        L.KLTB200SetForwardBackward(tc, fb)
        L.track(tc, provided[1], provided[2], fl)
        lists.append((tc, fl))
        states.append(before)
    (_, fa), (_, fb_) = lists
    ax, ay, av = capi.featurelist_to_arrays(fa)
    bx, by, bv = capi.featurelist_to_arrays(fb_)
    aa, ba = capi.featurelist_affine(fa), capi.featurelist_affine(fb_)
    kept = bv != FB_INCONSISTENT
    rej = ~kept
    assert rej.sum() > 0 and kept.sum() > 50
    assert ax[kept].tobytes() == bx[kept].tobytes() and ay[kept].tobytes() == by[kept].tobytes()
    assert np.array_equal(av[kept], bv[kept])
    assert aa[kept].tobytes() == ba[kept].tobytes()
    for i in np.nonzero(kept)[0]:
        ta, tb = _template(fa, int(i)), _template(fb_, int(i))
        assert (ta is None) == (tb is None), int(i)
        if ta is not None:
            assert all(u.tobytes() == w.tobytes() for u, w in zip(ta, tb)), int(i)
    assert (bx[rej] == -1).all() and (by[rej] == -1).all()
    assert (ba["has"][rej] == 0).all()
    assert all(_template(fb_, int(i)) is None for i in np.nonzero(rej)[0])
    for k in ("aff_x", "aff_y", "Axx", "Ayx", "Axy", "Ayy"):
        assert ba[k][rej].tobytes() == states[1][k][rej].tobytes(), k
    for tc, fl in lists:
        L.KLTFreeFeatureList(fl)
        L.KLTFreeTrackingContext(tc)


def _loop(L, capi, frames, n, exact, replace, fb):
    tc = L.KLTCreateTrackingContext()
    tc.contents.sequentialMode = 1
    L.KLTB200SetExact(tc, exact)
    L.KLTB200SetForwardBackward(tc, fb)
    fl = L.KLTCreateFeatureList(n)
    ft = L.KLTCreateFeatureTable(len(frames), n)
    L.select(tc, frames[0], fl)
    L.KLTStoreFeatureList(fl, ft, 0)
    rejected = 0
    for k in range(1, len(frames)):
        L.track(tc, frames[k - 1], frames[k], fl)
        rec = L.forward_backward(tc, n)
        rejected += int((capi.featurelist_to_arrays(fl)[2] == FB_INCONSISTENT).sum())
        if replace:
            L.replace(tc, frames[k], fl)
        L.KLTStoreFeatureList(fl, ft, k)
    assert rejected > 0
    out = capi.featuretable_to_array(ft), capi.featurelist_to_arrays(fl), rec
    L.KLTFreeFeatureTable(ft)
    L.KLTFreeFeatureList(fl)
    L.KLTFreeTrackingContext(tc)
    return out


@pytest.mark.parametrize("exact", [0, 1])
@pytest.mark.parametrize("replace", [False, True])
def test_sequence_call_equals_per_call_loop(L, capi, provided, exact, replace):
    n = 150
    tab, fin, rec = _loop(L, capi, provided, n, exact, replace, 0.3)
    tc = L.KLTCreateTrackingContext()
    tc.contents.sequentialMode = 1
    L.KLTB200SetExact(tc, exact)
    L.KLTB200SetForwardBackward(tc, 0.3)
    fl = L.KLTCreateFeatureList(n)
    ft = L.KLTCreateFeatureTable(len(provided), n)
    L.select(tc, provided[0], fl)
    L.KLTStoreFeatureList(fl, ft, 0)
    L.track_sequence(tc, provided[:6], fl, ft, 0, replace)
    L.track_sequence(tc, provided[5:], fl, ft, 5, replace)
    got = capi.featuretable_to_array(ft)
    assert got.tobytes() == tab.tobytes()
    assert all(u.tobytes() == w.tobytes() for u, w in zip(capi.featurelist_to_arrays(fl), fin))
    assert all(u.tobytes() == w.tobytes() for u, w in zip(L.forward_backward(tc, n), rec))
    L.KLTFreeFeatureTable(ft)
    L.KLTFreeFeatureList(fl)
    L.KLTFreeTrackingContext(tc)


@pytest.mark.parametrize("replace", [False, True])
def test_exact_loop_matches_oracle_loop(L, capi, oracle, oracle_mod, provided, replace):
    n = 150
    tab, _, _ = _loop(L, capi, provided, n, 1, replace, 0.3)
    tc = L.KLTCreateTrackingContext()
    p = params_from_tc(oracle, tc)
    L.KLTFreeTrackingContext(tc)
    x, y, v = oracle.select(provided[0], p, n, sort_kind=oracle_mod.SORT_STABLE)
    prev = oracle.build_pyramids(provided[0], p)
    for k in range(1, len(provided)):
        cur = oracle.build_pyramids(provided[k], p)
        x, y, v = track_fb(oracle, prev, cur, p, x, y, v, 0.3)[:3]
        if replace:
            x, y, v = oracle.select(provided[k], p, n, sort_kind=oracle_mod.SORT_STABLE, replace=True,
                                    last=cur, x=x, y=y, val=v)
        assert tab["x"][:, k].tobytes() == x.tobytes() and tab["y"][:, k].tobytes() == y.tobytes(), k
        assert np.array_equal(tab["val"][:, k], v), k
        prev = cur


def test_resident_pipeline_equals_per_call_loop(L, capi, provided):
    n = 150
    tab, fin, rec = _loop(L, capi, provided, n, 0, False, 0.3)
    tc = L.KLTCreateTrackingContext()
    tc.contents.sequentialMode = 1
    L.KLTB200SetForwardBackward(tc, 0.3)
    fl = L.KLTCreateFeatureList(n)
    L.select(tc, provided[0], fl)
    frames = [np.ascontiguousarray(f) for f in provided]
    h, w = frames[0].shape
    L.KLTB200ResidentBegin(tc, frames[0].ctypes.data, 0, w, w, h, fl)
    for k in range(1, len(frames)):
        L.KLTB200ResidentStep(tc, frames[k].ctypes.data, 0, w, w, h)
    L.KLTB200ResidentEnd(tc, fl)
    assert all(u.tobytes() == w_.tobytes() for u, w_ in zip(capi.featurelist_to_arrays(fl), fin))
    assert all(u.tobytes() == w_.tobytes() for u, w_ in zip(L.forward_backward(tc, n), rec))
    L.KLTFreeFeatureList(fl)
    L.KLTFreeTrackingContext(tc)


def test_guard_mode(L, capi):
    frames = [synth_image(643, 487, 5, shift=(1.9 * k, -1.3 * k)) for k in range(8)]
    tc = L.KLTCreateTrackingContext()
    tc.contents.sequentialMode = 1
    dev = L.KLTB200Device(tc)
    L.klt_dev_set_guard(dev, 1)
    L.KLTB200SetForwardBackward(tc, 0.2)
    fl = L.KLTCreateFeatureList(300)
    ft = L.KLTCreateFeatureTable(len(frames), 300)
    L.select(tc, frames[0], fl)
    for k in (1, 2, 3):
        L.track(tc, frames[k - 1], frames[k], fl)
        L.replace(tc, frames[k], fl)
    L.track_sequence(tc, frames[3:], fl, ft, 3, True)
    L.forward_backward(tc, 300)
    bad, band = C.c_longlong(-1), C.c_int(-1)
    assert L.klt_dev_check_guards(dev, C.byref(bad), C.byref(band)) == 0
    assert bad.value == 0, (bad.value, band.value)
    L.KLTFreeFeatureTable(ft)
    L.KLTFreeFeatureList(fl)
    L.KLTFreeTrackingContext(tc)


def test_environment_default_switches_the_check_on(L, capi, provided, monkeypatch):
    monkeypatch.setenv("KLT_B200_FB_MAX_ERROR", "0.3")
    tc = L.KLTCreateTrackingContext()
    fl = L.KLTCreateFeatureList(150)
    L.select(tc, provided[0], fl)
    x, y, v = capi.featurelist_to_arrays(fl)
    L.track(tc, provided[0], provided[1], fl)
    gx, gy, gv = capi.featurelist_to_arrays(fl)
    xb, yb, err, bv = L.forward_backward(tc, 150)
    monkeypatch.delenv("KLT_B200_FB_MAX_ERROR")
    tc2 = L.KLTCreateTrackingContext()
    L.KLTB200SetForwardBackward(tc2, 0.3)
    assert all(u.tobytes() == w.tobytes() for u, w in zip(_call(L, capi, tc2, provided[0], provided[1], x, y, v),
                                                          (gx, gy, gv, xb, yb, err, bv)))
    assert (gv == FB_INCONSISTENT).sum() > 0
    L.KLTFreeFeatureList(fl)
    L.KLTFreeTrackingContext(tc)
    L.KLTFreeTrackingContext(tc2)
