"""Oracle of the motion prior (KLTB200SetPrediction / KLTB200SetGuesses, include/klt_b200.h) -- TEST
INFRASTRUCTURE ONLY.  The prior is not part of the reference, so it is not part of the oracle's
restatement of it (oracle/): it is composed here from the oracle's exported single-level solver,
klto_track_level_li (oracle/klt_oracle.c), restating the feature loop of klto_track with the descent
started from the guess.  Every position is float32 and every operation separately rounded, as in the
library."""
import ctypes as C

import numpy as np

TRACKED, SMALL_DET, OOB = 0, -2, -4
FB_INCONSISTENT = -6
NONE, VELOCITY, EXPLICIT = 0, 1, 2

_f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")


def _lib(oracle):
    L = oracle.lib
    if not getattr(L, "_predict_bound", False):
        L.klto_track_level_li.argtypes = ([C.c_float, C.c_float, C.POINTER(C.c_float), C.POINTER(C.c_float)]
                                          + [_f32p] * 6 + [C.c_int] * 4
                                          + [C.c_float, C.c_int, C.c_float, C.c_float, C.c_float, C.c_int])
        L.klto_track_level_li.restype = C.c_int
        L._predict_bound = True
    return L


def _levels(pyr):
    if not hasattr(pyr, "_levels"):
        pyr._levels = [tuple(np.ascontiguousarray(pyr.view(w, l)) for w in range(3)) for l in range(pyr.nlevels)]
    return pyr._levels


def descend(oracle, pyr1, pyr2, p, x, y, gx, gy):
    """klto_track's descent for one feature from (x, y), with xout starting from the guess (gx, gy)
    scaled through the levels as (x, y) is, then the border test -> (x, y, val) as klto_track records"""
    L = _lib(oracle)
    f = np.float32
    ss = f(p.subsampling)
    xl, yl, xo, yo = f(x), f(y), f(gx), f(gy)
    for _ in range(p.nPyramidLevels):
        xl, yl, xo, yo = f(xl / ss), f(yl / ss), f(xo / ss), f(yo / ss)
    lv1, lv2 = _levels(pyr1), _levels(pyr2)
    v = TRACKED
    for r in range(p.nPyramidLevels - 1, -1, -1):
        xl, yl, xo, yo = f(xl * ss), f(yl * ss), f(xo * ss), f(yo * ss)
        x2, y2 = C.c_float(xo), C.c_float(yo)
        i1, g1x, g1y = lv1[r]
        i2, g2x, g2y = lv2[r]
        v = L.klto_track_level_li(xl, yl, C.byref(x2), C.byref(y2), i1, g1x, g1y, i2, g2x, g2y,
                                  i1.shape[1], i1.shape[0], p.window_width, p.window_height, p.step_factor,
                                  p.max_iterations, p.min_determinant, p.min_displacement, p.max_residue,
                                  p.lighting_insensitive)
        xo, yo = f(x2.value), f(y2.value)
        if v in (SMALL_DET, OOB):
            break
    nr, nc = lv1[0][0].shape
    if v == OOB or xo < p.borderx or xo > nc - 1 - p.borderx or yo < p.bordery or yo > nr - 1 - p.bordery:
        return f(-1), f(-1), OOB
    if v != TRACKED:
        return f(-1), f(-1), v
    return xo, yo, TRACKED


def _has(gx, gy):
    return np.isfinite(gx) & np.isfinite(gy)


def track_guided(oracle, pyr1, pyr2, p, x, y, val, gx, gy):
    """klto_track with a guess per feature (NaN: none) -> (x, y, val)"""
    x = np.array(x, np.float32); y = np.array(y, np.float32); val = np.array(val, np.int32)
    gx = np.asarray(gx, np.float32); gy = np.asarray(gy, np.float32)
    has = _has(gx, gy)
    for i in np.nonzero(val >= 0)[0]:
        g = (gx[i], gy[i]) if has[i] else (x[i], y[i])
        x[i], y[i], val[i] = descend(oracle, pyr1, pyr2, p, x[i], y[i], *g)
    return x, y, val


def track_fb_guided(oracle, pyr1, pyr2, p, x, y, val, gx, gy, max_error):
    """track_guided plus the forward-backward check (tests/fb_oracle.py's rule); the backward leg of a
    feature with a guess g starts from the mirrored prior xout - (g - x0)
    -> (x, y, val, xb, yb, err, back_val)"""
    x0 = np.array(x, np.float32); y0 = np.array(y, np.float32); v0 = np.array(val, np.int32)
    gx = np.asarray(gx, np.float32); gy = np.asarray(gy, np.float32)
    xf, yf, vf = track_guided(oracle, pyr1, pyr2, p, x0, y0, v0, gx, gy)
    n = len(xf)
    xb = np.full(n, -1.0, np.float32); yb = np.full(n, -1.0, np.float32)
    err = np.full(n, -1.0, np.float32); bv = np.ones(n, np.int32)
    if not max_error > 0:
        return xf, yf, vf, xb, yb, err, bv
    has = _has(gx, gy)
    thr2 = np.float32(max_error) * np.float32(max_error)
    for i in np.nonzero((v0 >= 0) & (vf == 0))[0]:
        g = (xf[i] - (gx[i] - x0[i]), yf[i] - (gy[i] - y0[i])) if has[i] else (xf[i], yf[i])
        bx, by, b = descend(oracle, pyr2, pyr1, p, xf[i], yf[i], *g)
        xb[i], yb[i], bv[i] = bx, by, b
        keep = False
        if b == TRACKED:
            dx, dy = bx - x0[i], by - y0[i]
            d2 = dx * dx + dy * dy
            err[i] = np.sqrt(d2)
            keep = not d2 > thr2
        if not keep:
            xf[i], yf[i], vf[i] = -1.0, -1.0, FB_INCONSISTENT
    return xf, yf, vf, xb, yb, err, bv


class VelocityDriver:
    """the per-call rule of KLT_B200_PREDICT_VELOCITY in numpy float32: one record {px, py, dx, dy} per
    feature index; a feature with input val == 0 that still starts at (px, py) gets g = x0 + (dx, dy);
    an explicit guess takes precedence.  step() tracks one frame pair and returns (x, y, val) and the
    per-feature (gx, gy, source) that KLTB200PredictionResult reports."""

    def __init__(self, n):
        self.px = np.full(n, np.nan, np.float32); self.py = np.full(n, np.nan, np.float32)
        self.dx = np.zeros(n, np.float32); self.dy = np.zeros(n, np.float32)

    def forget(self):
        self.px[:] = np.nan

    def guesses(self, x, y, val, ex=None, ey=None):
        x = np.asarray(x, np.float32); y = np.asarray(y, np.float32); val = np.asarray(val)
        n = len(x)
        gx = np.full(n, np.nan, np.float32); gy = np.full(n, np.nan, np.float32)
        src = np.zeros(n, np.int32)
        vel = (val == 0) & (x == self.px) & (y == self.py)
        gx[vel] = x[vel] + self.dx[vel]; gy[vel] = y[vel] + self.dy[vel]; src[vel] = VELOCITY
        if ex is not None:
            e = _has(np.asarray(ex, np.float32), np.asarray(ey, np.float32))
            gx[e] = np.asarray(ex, np.float32)[e]; gy[e] = np.asarray(ey, np.float32)[e]; src[e] = EXPLICIT
        live = val >= 0
        src[~live] = NONE; gx[~live] = np.nan; gy[~live] = np.nan
        return gx, gy, src

    def step(self, oracle, pyr1, pyr2, p, x, y, val, ex=None, ey=None, fb=0.0):
        x0 = np.array(x, np.float32); y0 = np.array(y, np.float32); v0 = np.array(val, np.int32)
        gx, gy, src = self.guesses(x0, y0, v0, ex, ey)
        if fb > 0:
            x1, y1, v1 = track_fb_guided(oracle, pyr1, pyr2, p, x0, y0, v0, gx, gy, fb)[:3]
        else:
            x1, y1, v1 = track_guided(oracle, pyr1, pyr2, p, x0, y0, v0, gx, gy)
        ok = v1 == TRACKED
        self.px = np.where(ok, x1, np.float32(np.nan)).astype(np.float32)
        self.py = np.where(ok, y1, np.float32(np.nan)).astype(np.float32)
        self.dx = np.where(ok, x1 - x0, 0).astype(np.float32)
        self.dy = np.where(ok, y1 - y0, 0).astype(np.float32)
        rx = np.where(src > 0, gx, np.float32(-1)).astype(np.float32)
        ry = np.where(src > 0, gy, np.float32(-1)).astype(np.float32)
        return (x1, y1, v1), (rx, ry, src)


def pan_frames(w=640, h=480, accel=2, frames=17, seed=21):
    """an accelerating horizontal pan: frame k is a w x h crop of one larger synthetic texture, moved
    right by k*accel pixels more than the frame before (scene motion -accel, -2 accel, ... px/frame),
    so the content never runs out -> (frames, per-frame scene displacement in x)"""
    from tests.conftest import synth_image
    v = [accel * k for k in range(frames)]
    off = np.cumsum(v)
    big = synth_image(w + int(off[-1]) + 8, h, seed)
    return [np.ascontiguousarray(big[:, o:o + w]) for o in off], [-float(s) for s in v]


def pan_survival(oracle, oracle_mod, frames, n, velocity, replace=True):
    """the per-call loop over frames with the default context, with or without the velocity prior
    -> number of KLT_TRACKED results summed over all frame pairs"""
    p = oracle.default_params()
    x, y, v = oracle.select(frames[0], p, n, sort_kind=oracle_mod.SORT_STABLE)
    drv = VelocityDriver(n)
    prev = oracle.build_pyramids(frames[0], p)
    tracked = 0
    for k in range(1, len(frames)):
        cur = oracle.build_pyramids(frames[k], p)
        if velocity:
            (x, y, v), _ = drv.step(oracle, prev, cur, p, x, y, v)
        else:
            x, y, v = oracle.track(prev, cur, p, x, y, v)
        tracked += int((v == 0).sum())
        if replace:
            x, y, v = oracle.select(frames[k], p, n, sort_kind=oracle_mod.SORT_STABLE, replace=True,
                                    last=cur, x=x, y=y, val=v)
        prev = cur
    return tracked
