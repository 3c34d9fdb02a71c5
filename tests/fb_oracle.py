"""Oracle of the forward-backward check (KLTB200SetForwardBackward, include/klt_b200.h) -- TEST
INFRASTRUCTURE ONLY, and an extension: the check is not part of the reference, so it is not part of
the oracle's restatement of it (oracle/).  It is composed here from two reference tracking calls of
the oracle and the float32 decision."""
import numpy as np

FB_INCONSISTENT = -6


def track_fb(oracle, pyr1, pyr2, p, x, y, val, max_error):
    """Forward leg = klto_track(pyr1, pyr2), backward leg = klto_track(pyr2, pyr1) from the forward
    result of every feature the forward leg tracked, then the decision in float32 with every
    operation rounded separately (numpy does not contract a*a + b*b): kept <=> the backward leg
    tracked and !(d2 > max_error^2).  -> (x, y, val, xb, yb, err, back_val); xb = yb = err = -1,
    back_val = 1 where the check did not run, xb = yb = err = -1 where the backward leg lost it."""
    x0 = np.array(x, np.float32); y0 = np.array(y, np.float32); v0 = np.array(val, np.int32)
    xf, yf, vf = oracle.track(pyr1, pyr2, p, x0, y0, v0)
    n = len(xf)
    xb = np.full(n, -1.0, np.float32); yb = np.full(n, -1.0, np.float32)
    err = np.full(n, -1.0, np.float32); bv = np.ones(n, np.int32)
    if not max_error > 0:
        return xf, yf, vf, xb, yb, err, bv
    run = np.nonzero((v0 >= 0) & (vf == 0))[0]
    if len(run):
        bx, by, bval = oracle.track(pyr2, pyr1, p, xf[run], yf[run], np.zeros(len(run), np.int32))
        xb[run], yb[run], bv[run] = bx, by, bval
        ok = bval == 0
        dx = bx - x0[run]; dy = by - y0[run]
        d2 = dx * dx + dy * dy
        err[run[ok]] = np.sqrt(d2[ok])
        thr2 = np.float32(max_error) * np.float32(max_error)
        drop = run[~(ok & ~(d2 > thr2))]
        xf[drop] = -1.0; yf[drop] = -1.0; vf[drop] = FB_INCONSISTENT
    return xf, yf, vf, xb, yb, err, bv
