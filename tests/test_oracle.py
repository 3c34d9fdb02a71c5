"""Pin the oracle (oracle/klt_oracle.c) before trusting it.

 * against the reference's golden run src/V1/feat/features2.ft (byte for byte)
 * against what the unmodified reference CPU sources return, stage by stage and bit for bit:
   tests/golden/reference_digests.json holds a SHA-256 digest of every array these tests
   compare (the reference sources are not part of the repository; see tests/golden/README.md).
CPU only.
"""
import hashlib
import json
import os

import numpy as np
import pytest

from tests.conftest import GOLDEN, synth_image

DIGESTS_PATH = os.path.join(GOLDEN, "reference_digests.json")
RECORD = os.environ.get("KLT_RECORD_DIGESTS") == "1"
_DIGESTS = json.load(open(DIGESTS_PATH)) if os.path.exists(DIGESTS_PATH) else {}


@pytest.fixture(scope="module", autouse=True)
def _record_digests():
    yield
    if RECORD:
        with open(DIGESTS_PATH, "w") as fh:
            json.dump(dict(sorted(_DIGESTS.items())), fh, indent=0)
            fh.write("\n")


def _pin(key, *arrays):
    """the arrays, bit for bit, equal what the reference returned (stored digest `key`)"""
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(("%s%s" % (a.dtype.str, a.shape)).encode())
        h.update(a.tobytes())
    if RECORD:
        _DIGESTS[key] = h.hexdigest()
    else:
        assert h.hexdigest() == _DIGESTS[key], key


def _v1_flow_oracle(oracle, oracle_mod, imgs, n=150, sort_kind=None):
    """reference src/V1/example3.c:35-65 restated on the oracle API."""
    sort_kind = oracle_mod.SORT_QUICK if sort_kind is None else sort_kind
    p = oracle.default_params()
    nframes = len(imgs)
    table = np.zeros((n, nframes), dtype=[("x", "f4"), ("y", "f4"), ("val", "i4")])
    x, y, v = oracle.select(imgs[0], p, n, sort_kind=sort_kind)
    table["x"][:, 0], table["y"][:, 0], table["val"][:, 0] = x, y, v
    prev = oracle.build_pyramids(imgs[0], p)
    for i in range(1, nframes):
        cur = oracle.build_pyramids(imgs[i], p)
        x, y, v = oracle.track(prev, cur, p, x, y, v)
        table["x"][:, i - 1], table["y"][:, i - 1], table["val"][:, i - 1] = x, y, v
        prev = cur
    return table


def test_oracle_reproduces_golden_feature_table(oracle, oracle_mod, provided, golden_ft):
    raw, gold = golden_ft
    tab = _v1_flow_oracle(oracle, oracle_mod, provided)
    # column 9 of the golden file was never written by the driver (SURVEY 4)
    assert tab[:, :9].tobytes() == gold[:, :9].tobytes()
    # the whole file, header included, with the unwritten column taken as zeros
    tab[:, 9] = (0.0, 0.0, 0)
    blob = b"KLTFT1" + np.array([10, 150], np.int32).tobytes() + tab.tobytes()
    assert blob == raw


def test_oracle_call_counts_match_gprof(oracle, provided):
    # src/V1/example3_analysis.txt: 52 224 _minEigenvalue calls = (320-48)*(240-48)
    p = oracle.default_params()
    f = oracle.smooth(oracle.to_float(provided[0]), 0.7)
    gx, gy = oracle.gradients(f, 1.0)
    pts = oracle.mineig_points(gx, gy, 7, 7, p.borderx, p.bordery)
    assert len(pts) == 52224


@pytest.mark.parametrize("sigma,wg,wd", [(0.7, 5, 5), (1.0, 7, 7), (1.8, 11, 13),
                                         (3.6, 21, 25), (7.2, 43, 51)])
def test_tap_widths(oracle, sigma, wg, wd):
    # (wg, wd): the reference's _KLTGetKernelWidths at these sigmas
    g, d = oracle.taps(sigma)
    assert (len(g), len(d)) == (wg, wd)
    assert abs(g.sum() - 1.0) < 1e-6
    assert d[len(d) // 2] == 0.0


def test_params_match_reference(oracle):
    # the reference's KLTCreateTrackingContext defaults and, per search range, what its
    # KLTChangeTCPyramid + KLTUpdateTCBorder leave: (nPyramidLevels, subsampling, borderx, bordery)
    defaults = {"mindist": 10, "window_width": 7, "window_height": 7, "min_eigenvalue": 1,
                "max_iterations": 10, "nSkippedPixels": 0, "borderx": 24, "bordery": 24,
                "nPyramidLevels": 2, "subsampling": 4}
    per_search_range = {1: (1, 4, 5, 5), 3: (1, 4, 5, 5), 5: (2, 2, 14, 14), 10: (2, 2, 14, 14),
                        15: (2, 4, 24, 24), 17: (2, 4, 24, 24), 20: (2, 8, 48, 48), 31: (2, 8, 48, 48),
                        32: (2, 8, 48, 48), 60: (3, 8, 384, 384), 100: (3, 8, 384, 384),
                        400: (4, 8, 3072, 3072)}
    p = oracle.default_params()
    for f, want in defaults.items():
        assert getattr(p, f) == want, f
    for sr, want in per_search_range.items():
        oracle.change_pyramid(p, sr)
        oracle.update_border(p)
        assert (p.nPyramidLevels, p.subsampling, p.borderx, p.bordery) == want, sr
    # config 4 of BASELINE.json: L=4, ss=2 set directly, then the border update
    p.nPyramidLevels, p.subsampling = 4, 2
    oracle.update_border(p)
    assert p.borderx == 64


@pytest.mark.parametrize("shape", [(243, 321), (64, 80), (31, 47)])
@pytest.mark.parametrize("sigma", [0.7, 1.0, 1.8, 3.6])
def test_stages_bit_exact_vs_reference(oracle, shape, sigma):
    h, w = shape
    f = synth_image(w, h, seed=w * 7 + h).astype(np.float32)
    key = "stages/%dx%d/sigma%r" % (h, w, sigma)
    _pin(key + "/smooth", oracle.smooth(f, sigma))
    _pin(key + "/gradients", *oracle.gradients(f, sigma))


@pytest.mark.parametrize("ss,levels", [(2, 4), (4, 2), (4, 3), (8, 2)])
def test_pyramid_bit_exact_vs_reference(oracle, ss, levels):
    f = synth_image(352, 288, seed=ss * 10 + levels).astype(np.float32)
    cur = f
    for l in range(1, levels):
        cur = oracle.pyr_down(cur, ss, np.float32(ss * np.float32(0.9)))
        _pin("pyramid/ss%d/levels%d/level%d" % (ss, levels, l), cur)


def test_select_and_track_bit_exact_vs_reference(oracle, oracle_mod, provided):
    """the reference's default build (_quicksort) and its -DKLT_USE_QSORT build (stable ties)"""
    imgs = provided[:4]
    for lib, kind in (("ref", oracle_mod.SORT_QUICK), ("ref_qsort", oracle_mod.SORT_STABLE)):
        p = oracle.default_params()
        x, y, v = oracle.select(imgs[0], p, 150, sort_kind=kind)
        _pin("select_and_track/%s/frame0" % lib, x, y, v)
        prev = oracle.build_pyramids(imgs[0], p)
        for i in range(1, len(imgs)):
            cur = oracle.build_pyramids(imgs[i], p)
            x, y, v = oracle.track(prev, cur, p, x, y, v)
            _pin("select_and_track/%s/frame%d" % (lib, i), x, y, v)
            prev = cur


def test_four_level_config_and_replace_vs_reference(oracle, oracle_mod):
    """config-4 shaped parameters (L=4, ss=2) on a small synthetic pair, plus the
    KLTReplaceLostFeatures path that reuses pyramid_last (sequentialMode)."""
    imgs = [synth_image(480, 360, seed=5, shift=(1.7 * t, -0.9 * t)) for t in range(3)]
    n = 300
    p = oracle.default_params()
    p.nPyramidLevels, p.subsampling = 4, 2
    oracle.update_border(p)
    assert p.borderx == 64

    x, y, v = oracle.select(imgs[0], p, n, sort_kind=oracle_mod.SORT_STABLE)
    _pin("four_level/select", x, y, v)
    prev = oracle.build_pyramids(imgs[0], p)
    for i in (1, 2):
        cur = oracle.build_pyramids(imgs[i], p)
        x, y, v = oracle.track(prev, cur, p, x, y, v)
        _pin("four_level/frame%d/track" % i, x, y, v)
        # knock out some features so that the replacement has work to do
        v[::7] = -3; x[::7] = -1; y[::7] = -1
        x, y, v = oracle.select(imgs[i], p, n, sort_kind=oracle_mod.SORT_STABLE,
                                replace=True, last=cur, x=x, y=y, val=v)
        _pin("four_level/frame%d/replace" % i, x, y, v)
        prev = cur
    # the pyramids the reference keeps in sequential mode (tc->pyramid_last*)
    for l in range(4):
        _pin("four_level/pyramid_last/level%d" % l, prev.level(0, l), prev.level(1, l), prev.level(2, l))


def test_quicksort_permutation_matches_reference(oracle):
    rng = np.random.default_rng(3)
    for n in (1, 2, 3, 17, 1000, 52224):
        pts = np.zeros((n, 3), np.int32)
        pts[:, 0] = np.arange(n)
        pts[:, 1] = rng.integers(0, 1000, n)
        pts[:, 2] = rng.integers(0, 40, n)          # many ties
        a = pts.copy()
        oracle.lib.klto_sort_points(a, n, 1)
        _pin("quicksort/n%d" % n, a)                # the reference's _quicksort on the same points
        c = pts.copy()
        oracle.lib.klto_sort_points(c, n, 0)
        order = np.argsort(-pts[:, 2], kind="stable")
        assert np.array_equal(c, pts[order])


def test_lighting_insensitive_tracking_bit_exact_vs_reference(oracle, oracle_mod, provided):
    """tc->lighting_insensitive = TRUE (trackFeatures.c:125-220): gain / bias normalised windows,
    including the reference's quirk that the gradient sum's gain is sqrt(mean(g1) / mean(g2)).
    A brightness ramp is added to the later frames so that the normalisation matters."""
    imgs = [provided[0]]
    for k in range(1, 4):
        f = provided[k].astype(np.float32) * (1.0 + 0.08 * k) + 6.0 * k
        imgs.append(np.clip(f, 0, 255).astype(np.uint8))
    flows = {}
    for li in (1, 0):
        p = oracle.default_params()
        p.lighting_insensitive = li
        x, y, v = oracle.select(imgs[0], p, 150, sort_kind=oracle_mod.SORT_STABLE)
        prev = oracle.build_pyramids(imgs[0], p)
        flows[li] = []
        for i in range(1, len(imgs)):
            cur = oracle.build_pyramids(imgs[i], p)
            x, y, v = oracle.track(prev, cur, p, x, y, v)
            flows[li].append(x)
            if li:
                _pin("lighting_insensitive/frame%d" % i, x, y, v)
            prev = cur
    assert any(not np.array_equal(a, b) for a, b in zip(flows[1], flows[0]))   # the flag matters


def _ramped(provided, n):
    """the provided frames with a brightness gain / offset growing from frame to frame"""
    imgs = [provided[0]]
    for k in range(1, n):
        f = provided[k].astype(np.float32) * (1.0 + 0.01 * k) + 0.5 * k
        imgs.append(np.clip(f, 0, 255).astype(np.uint8))
    return imgs


def _pin_affine(key, x, y, v, st):
    """positions, status, and the affine members (aff_x, aff_y, A) of the features that hold a template"""
    live = st["has"] == 1
    _pin(key, x, y, v, st["has"], *[st[k][live] for k in ("aff_x", "aff_y", "Axx", "Ayx", "Axy", "Ayy")])


def test_affine_check_0_with_lighting_insensitive_bit_exact_vs_reference(oracle, oracle_mod, provided):
    """tc->affineConsistencyCheck = 0 together with tc->lighting_insensitive (trackFeatures.c:1024-1028):
    the translation refinement against the template runs on the gain / bias normalised windows, the
    final residue on the plain difference (:1196-1199)."""
    imgs = _ramped(provided, 7)
    n = 120
    p = oracle.default_params()
    p.lighting_insensitive = 1
    ap = oracle_mod.affine_params(check=0)
    x, y, v = oracle.select(imgs[0], p, n, sort_kind=oracle_mod.SORT_STABLE)
    st, tmpl = oracle_mod.affine_state(n)
    prev = oracle.build_pyramids(imgs[0], p)
    p_plain = oracle.default_params()
    differs = 0
    for i in range(1, len(imgs)):
        cur = oracle.build_pyramids(imgs[i], p)
        st2, tmpl2 = st.copy(), tmpl.copy()
        plain = oracle.track_affine(prev, cur, p_plain, ap, x.copy(), y.copy(), v.copy(), st2, tmpl2)
        x, y, v = oracle.track_affine(prev, cur, p, ap, x, y, v, st, tmpl)
        differs += int((plain[2] != v).sum()) + int((plain[0] != x).sum())
        _pin_affine("affine_check0_lighting_insensitive/frame%d" % i, x, y, v, st)
        prev = cur
    assert differs > 0                                  # the flag matters on these frames
    assert (st["has"] == 1).sum() > 20


def _warped(img, k):
    """frame k of a slowly rotating / zooming / shifting copy of img (bilinear, numpy)"""
    h, w = img.shape
    a, sc = np.deg2rad(0.6 * k), 1.0 + 0.004 * k
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float64)
    cx, cy = w / 2.0, h / 2.0
    xs = (np.cos(a) * (xx - cx) - np.sin(a) * (yy - cy)) / sc + cx + 0.9 * k
    ys = (np.sin(a) * (xx - cx) + np.cos(a) * (yy - cy)) / sc + cy - 0.6 * k
    x0 = np.clip(np.floor(xs).astype(int), 0, w - 2); y0 = np.clip(np.floor(ys).astype(int), 0, h - 2)
    ax = np.clip(xs - x0, 0, 1); ay = np.clip(ys - y0, 0, 1)
    f = img.astype(np.float64)
    v = (f[y0, x0] * (1 - ax) * (1 - ay) + f[y0, x0 + 1] * ax * (1 - ay)
         + f[y0 + 1, x0] * (1 - ax) * ay + f[y0 + 1, x0 + 1] * ax * ay)
    return np.clip(np.rint(v), 0, 255).astype(np.uint8)


@pytest.mark.parametrize("check", [0, 1, 2])
@pytest.mark.parametrize("seq", ["provided", "warped"])
def test_affine_consistency_check_bit_exact_vs_reference(oracle, oracle_mod, provided, check, seq):
    """tc->affineConsistencyCheck = 0 / 1 / 2 (trackFeatures.c:506-1224, :1438-1497): template
    creation after the first successful track, translation / similarity / affine refinement against
    the template, status changes, and the persistent aff_* members of every feature."""
    imgs = provided[:7] if seq == "provided" else [_warped(provided[0], k) for k in range(7)]
    n = 120
    p = oracle.default_params()
    ap = oracle_mod.affine_params(check=check)
    x, y, v = oracle.select(imgs[0], p, n, sort_kind=oracle_mod.SORT_STABLE)
    st, tmpl = oracle_mod.affine_state(n)
    prev = oracle.build_pyramids(imgs[0], p)
    changed = 0
    for i in range(1, len(imgs)):
        cur = oracle.build_pyramids(imgs[i], p)
        plain = oracle.track(prev, cur, p, x, y, v)
        x, y, v = oracle.track_affine(prev, cur, p, ap, x, y, v, st, tmpl)
        changed += int((plain[2] != v).sum())
        _pin_affine("affine_check%d/%s/frame%d" % (check, seq, i), x, y, v, st)
        prev = cur
    print("affine check %d on %s: %d status changes" % (check, seq, changed))
