"""Oracle of the global motion check (KLTB200SetMotionCheck, include/klt_b200.h) -- TEST
INFRASTRUCTURE ONLY, and an extension: the check is not part of the reference, so it is not part of
the oracle's restatement of it (oracle/).  It restates the algorithm of csrc/klt_motion.cuh (DESIGN.md
4, "Global motion check") step by step: Python floats are IEEE doubles with every operation rounded
separately, as the kernels' __dadd_rn / __dmul_rn / __ddiv_rn, and numpy float32 arrays do not
contract, as the kernels' __fmul_rn / __fadd_rn.  Only the refinement's reduction order differs (here
numpy's), so the refined model is compared with a tolerance."""
import math

import numpy as np

MOTION_OUTLIER = -7
DRAWS = 16
COLLINEAR = 1e-6
PIVOT = 1e-10
MIN_KEEP = 8
DEFAULT_HYPOTHESES = 1024
_M32 = 0xFFFFFFFF


def mix32(x):
    """lowbias32"""
    x &= _M32
    x ^= x >> 16
    x = (x * 0x7FEB352D) & _M32
    x ^= x >> 15
    x = (x * 0x846CA68B) & _M32
    x ^= x >> 16
    return x


def sample(h, m):
    """hypothesis h's 4 distinct correspondence indices (draw order), None after 16 draws without"""
    s = []
    for j in range(DRAWS):
        i = (mix32(h * 16 + j) * m) >> 32
        if len(s) < 4 and i not in s:
            s.append(i)
    return s if len(s) == 4 else None


def geometry(W, H):
    """normalisation (p - (cx, cy)) * s"""
    return W / 2.0, H / 2.0, 2.0 / max(W, H)


def _norm(p, c, s):
    return (float(p) - c) * s


def _cross(x, y, a, b, c):
    return (x[b] - x[a]) * (y[c] - y[a]) - (y[b] - y[a]) * (x[c] - x[a])


def degenerate(x, y):
    return any(abs(_cross(x, y, *t)) < COLLINEAR for t in ((0, 1, 2), (0, 1, 3), (0, 2, 3), (1, 2, 3)))


def solve8(A):
    """Gaussian elimination with partial pivoting (largest |a|, first on ties) of the 8 x 9 augmented
    system A; None when a pivot is below PIVOT"""
    A = [list(map(float, r)) for r in A]
    for k in range(8):
        p, best = k, abs(A[k][k])
        for i in range(k + 1, 8):
            if abs(A[i][k]) > best:
                best, p = abs(A[i][k]), i
        if not best >= PIVOT:
            return None
        A[k], A[p] = A[p], A[k]
        for i in range(k + 1, 8):
            f = A[i][k] / A[k][k]
            for j in range(k + 1, 9):
                A[i][j] = A[i][j] - f * A[k][j]
    h = [0.0] * 8
    for i in range(7, -1, -1):
        s = A[i][8]
        for j in range(i + 1, 8):
            s = s - A[i][j] * h[j]
        h[i] = s / A[i][i]
    return h


def denorm(n, geo):
    """T^-1 n T in pixel coordinates, scaled to H[8] = 1, rounded to float32 (8 entries); None when the
    scale is not finite and nonzero or an entry is not finite"""
    cx, cy, s = geo
    ox, oy = s * cx, s * cy
    M = [0.0] * 9
    for r in range(3):
        a, b, c = n[3 * r], n[3 * r + 1], (1.0 if r == 2 else n[3 * r + 2])
        M[3 * r] = a * s
        M[3 * r + 1] = b * s
        M[3 * r + 2] = c - (a * ox + b * oy)
    D = [0.0] * 9
    for j in range(3):
        D[j] = M[j] / s + cx * M[6 + j]
        D[3 + j] = M[3 + j] / s + cy * M[6 + j]
        D[6 + j] = M[6 + j]
    w = D[8]
    if not (math.isfinite(w) and w != 0.0):
        return None
    with np.errstate(over="ignore"):
        H = np.array([D[k] / w for k in range(8)], np.float64).astype(np.float32)
    return H if np.isfinite(H).all() else None


def _rows(x, y, u, v):
    return [[x, y, 1.0, 0.0, 0.0, 0.0, -(u * x), -(u * y), u],
            [0.0, 0.0, 0.0, x, y, 1.0, -(v * x), -(v * y), v]]


def hypothesis(h, corr, geo):
    """the float32 model (8 entries) of hypothesis h over corr (m x 4 float32: x0, y0, x1, y1), or None"""
    cx, cy, s = geo
    idx = sample(h, len(corr))
    if idx is None:
        return None
    px = [_norm(corr[i, 0], cx, s) for i in idx]; py = [_norm(corr[i, 1], cy, s) for i in idx]
    qx = [_norm(corr[i, 2], cx, s) for i in idx]; qy = [_norm(corr[i, 3], cy, s) for i in idx]
    if degenerate(px, py) or degenerate(qx, qy):
        return None
    A = []
    for k in range(4):
        A += _rows(px[k], py[k], qx[k], qy[k])
    n = solve8(A)
    return None if n is None else denorm(n, geo)


def d2(H, corr):
    """(squared reprojection distance, w > 0) per correspondence, separately rounded float32"""
    h = [np.float32(v) for v in H[:8]]
    x, y, x1, y1 = (np.ascontiguousarray(corr[:, i], np.float32) for i in range(4))
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        u = (h[0] * x + h[1] * y) + h[2]
        v = (h[3] * x + h[4] * y) + h[5]
        w = (h[6] * x + h[7] * y) + np.float32(1.0)
        dx = u / w - x1
        dy = v / w - y1
        return dx * dx + dy * dy, w > 0


def inliers(H, corr, e2):
    q, front = d2(H, corr)
    return front & ~(q > e2)


def refine(Hmin, corr, keep, geo):
    """one least-squares DLT (h22 = 1) over corr[keep] in normalised coordinates, float64 normal
    equations, the same elimination; the minimal model when singular"""
    cx, cy, s = geo
    c = corr[keep].astype(np.float64)
    x, y = (c[:, 0] - cx) * s, (c[:, 1] - cy) * s
    u, v = (c[:, 2] - cx) * s, (c[:, 3] - cy) * s
    z, o = np.zeros_like(x), np.ones_like(x)
    A = np.concatenate([np.stack([x, y, o, z, z, z, -u * x, -u * y], 1),
                        np.stack([z, z, z, x, y, o, -v * x, -v * y], 1)])
    b = np.concatenate([u, v])
    n = solve8(np.concatenate([A.T @ A, (A.T @ b)[:, None]], 1))
    R = None if n is None else denorm(n, geo)
    return (Hmin, False) if R is None else (R, True)


def motion_check(x0, y0, v0, x1, y1, v1, W, H, max_error, hypotheses=DEFAULT_HYPOTHESES):
    """The check on one call: start positions (x0, y0, v0) and the tracker's result (x1, y1, v1).
    -> dict: out (x, y, val after the check), err per feature, m, counts (-1: no model), winner,
    H_min, H (final, 3 x 3 float32, NaN unless valid), refined, valid, inliers, idx (feature index of
    each correspondence), d2 (per correspondence under the final model)."""
    x0, y0, x1, y1 = (np.asarray(a, np.float32) for a in (x0, y0, x1, y1))
    v0, v1 = np.asarray(v0, np.int32), np.asarray(v1, np.int32)
    n = len(x0)
    idx = np.nonzero((v0 >= 0) & (v1 == 0))[0]
    corr = np.stack([x0[idx], y0[idx], x1[idx], y1[idx]], 1).astype(np.float32)
    m = len(idx)
    geo = geometry(W, H)
    e2 = np.float32(max_error) * np.float32(max_error)
    counts = np.full(hypotheses, -1, np.int64)
    models = {}
    for h in range(hypotheses):
        Hh = hypothesis(h, corr, geo)
        if Hh is not None:
            models[h] = Hh
            counts[h] = int(inliers(Hh, corr, e2).sum())
    x, y, val = x1.copy(), y1.copy(), v1.copy()
    err = np.full(n, -1.0, np.float32)
    r = {"m": m, "counts": counts, "idx": idx, "corr": corr, "winner": -1, "H_min": None, "refined": False,
         "valid": 0, "inliers": 0, "H": np.full((3, 3), np.nan, np.float32), "d2": None, "e2": e2}
    if models:
        win = int(np.argmax(counts))                 # first maximum: the lowest h on ties
        Hmin = models[win]
        Hf, refined = refine(Hmin, corr, inliers(Hmin, corr, e2), geo)
        q, front = d2(Hf, corr)
        keep = front & ~(q > e2)
        err[idx] = np.where(front, np.sqrt(q), np.float32(np.inf))
        valid = int(keep.sum() >= MIN_KEEP)
        if valid:
            drop = idx[~keep]
            x[drop], y[drop], val[drop] = -1.0, -1.0, MOTION_OUTLIER
            r["H"] = np.append(Hf, np.float32(1.0)).reshape(3, 3)
        r.update(winner=win, H_min=Hmin, H_final=Hf, refined=refined, valid=valid, inliers=int(keep.sum()), d2=q)
    r.update(out=(x, y, val), err=err)
    return r


def project(H, pts):
    """pts (k x 2) through the 3 x 3 homography H, in float64"""
    H = np.asarray(H, np.float64)
    p = np.c_[pts, np.ones(len(pts))] @ H.T
    return p[:, :2] / p[:, 2:]


def corners(W, H):
    return np.array([[0, 0], [W - 1, 0], [W - 1, H - 1], [0, H - 1]], np.float64)


def warped_scene(W, H, Htrue, rect, shift, seed=21):
    """A frame pair: background texture (synth_image) warped by the 3 x 3 homography Htrue, and a
    rectangle (x0, y0, x1, y1) of another texture that moves by its own translation `shift` instead.
    Bilinear resampling (scipy.ndimage.map_coordinates, order 1). -> (img1, img2) uint8"""
    from scipy.ndimage import map_coordinates
    from tests.conftest import synth_image
    bg = synth_image(W, H, seed).astype(np.float64)
    ob = synth_image(W, H, seed + 100).astype(np.float64)
    rx0, ry0, rx1, ry1 = rect
    img1 = bg.copy()
    img1[ry0:ry1, rx0:rx1] = ob[ry0:ry1, rx0:rx1]
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float64)
    src = project(np.linalg.inv(Htrue), np.c_[xx.ravel(), yy.ravel()])
    img2 = map_coordinates(bg, [src[:, 1], src[:, 0]], order=1, mode="nearest").reshape(H, W)
    sx, sy = shift
    inside = (xx >= rx0 + sx) & (xx < rx1 + sx) & (yy >= ry0 + sy) & (yy < ry1 + sy)
    moved = map_coordinates(ob, [yy - sy, xx - sx], order=1, mode="nearest")
    img2[inside] = moved[inside]
    return (np.clip(np.rint(img1), 0, 255).astype(np.uint8), np.clip(np.rint(img2), 0, 255).astype(np.uint8))


# the effect scenario of the tests and tools/motion_bench.py: a slight rotation, zoom and pan of the
# background, and a rectangle moving against it
SCENE_W, SCENE_H = 640, 480
SCENE_RECT = (220, 160, 420, 320)
SCENE_SHIFT = (6.0, 4.0)


def scene_homography():
    a, z = math.radians(0.8), 1.01
    c, s = z * math.cos(a), z * math.sin(a)
    cx, cy = SCENE_W / 2.0, SCENE_H / 2.0
    return np.array([[c, -s, cx - c * cx + s * cy + 3.0],
                     [s, c, cy - s * cx - c * cy - 2.0],
                     [2e-6, -1e-6, 1.0]])


def scene():
    return warped_scene(SCENE_W, SCENE_H, scene_homography(), SCENE_RECT, SCENE_SHIFT)


def scene_groups(x0, y0, x1, y1, tracked, half_window):
    """(rectangle features: start inside the rectangle shrunk by the window half-width; background
    features tracked correctly: start outside the rectangle grown by the half-width and the shift,
    end within 0.5 px of the true motion).  The second group is narrower than "every feature outside
    the rectangle" on purpose: features whose window meets the rectangle in either frame, and
    background features the tracker got wrong, disagree with the background's homography, and
    dropping them is the check doing its job.  The tests' bound on wrongly flagged features (1 %)
    applies to this group only."""
    rx0, ry0, rx1, ry1 = SCENE_RECT
    hw = half_window
    inner = (x0 >= rx0 + hw) & (x0 < rx1 - hw) & (y0 >= ry0 + hw) & (y0 < ry1 - hw)
    g = hw + max(abs(v) for v in SCENE_SHIFT) + 1
    outer = (x0 >= rx0 - g) & (x0 < rx1 + g) & (y0 >= ry0 - g) & (y0 < ry1 + g)
    truth = project(scene_homography(), np.c_[x0, y0])
    good = np.hypot(x1 - truth[:, 0], y1 - truth[:, 1]) < 0.5
    return tracked & inner, tracked & ~outer & good
