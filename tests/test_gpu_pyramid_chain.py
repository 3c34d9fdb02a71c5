"""The chained pyramid (subsampling 2, radius 5, more than one level): l0_fused_kernel also makes L1 from
the L0 tile it holds, and level_chain_kernel makes gx_l, gy_l and L_{l+1} from L_l.  Compared with the
oracle (bit for bit in exact mode, within the image tolerance in fma mode) on a guarded arena, on shapes
that stress its index math: odd sizes, heights that are no multiple of the 40-row level-0 tile, a last
level-0 tile row that makes a partial L1 block, levels smaller than one tile, five levels, band sizes
around tile-row boundaries and one 4K frame.  In fma mode the chain must also give the same bits as the
unchained kernels (level-0 variant 0 + level_fused_kernel), which compute every sample with the same
operation sequence."""
import numpy as np
import pytest

from tests.conftest import synth_image
from tests.gpu_common import device_pyramids
from tests.test_gpu_guards import _guards_intact
from tests.test_gpu_stages import _check_build

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def L(pkg):
    from importlib import import_module
    lib = import_module(pkg.__name__ + ".runtime").load()
    lib.require_gpu()
    lib.KLTSetVerbosity(0)
    return lib


def _tc(L, levels):
    tc = L.KLTCreateTrackingContext()
    tc.contents.nPyramidLevels, tc.contents.subsampling = levels, 2
    L.KLTUpdateTCBorder(tc)
    return tc


# (h, w), levels
CASES = [
    ((323, 241), 4),      # odd W0 and H0
    ((203, 517), 4),      # H0 not a multiple of 40
    ((83, 300), 3),       # last level-0 tile row (y0 = 80) makes one L1 row of its block
    ((121, 259), 4),      # level 1 (129 x 60) short of a 64 x 32 tile row pair, level 3 under one tile
    ((130, 70), 4),       # levels 2 and 3 narrower than one tile
    ((30, 62), 2),        # level 1 (31 x 15) smaller than one tile
    ((500, 900), 5),      # five levels
    ((1080, 1920), 4),
]


@pytest.mark.parametrize("shape,levels", CASES)
def test_chained_pyramid_matches_oracle_on_a_guarded_arena(L, oracle, shape, levels):
    h, w = shape
    img = synth_image(w, h, seed=5 * h + w)
    for exact in (1, 0):
        tc = _tc(L, levels)
        dev = L.KLTB200Device(tc)
        L.klt_dev_set_guard(dev, 1)
        _check_build(L, oracle, img, tc, exact, 0, expect_tiled=True, expect_fused=True)
        assert L.klt_dev_last_build_fused(dev) == levels
        _guards_intact(L, dev, "%dx%d, %d levels, exact %d" % (w, h, levels, exact))
        L.KLTFreeTrackingContext(tc)


def test_chained_pyramid_4k(L, oracle):
    img = synth_image(3840, 2160, seed=11)
    for exact in (1, 0):
        tc = _tc(L, 4)
        dev = L.KLTB200Device(tc)
        L.klt_dev_set_guard(dev, 1)
        _check_build(L, oracle, img, tc, exact, 0, expect_tiled=True, expect_fused=True)
        _guards_intact(L, dev, "4K, exact %d" % exact)
        L.KLTFreeTrackingContext(tc)


# bands are rounded up to 64 rows: 64 / 128 / 192 end inside a 40-row level-0 tile row, 320 on one
@pytest.mark.parametrize("band_rows", [64, 128, 192, 320])
def test_banded_chained_build(L, oracle, band_rows):
    h, w = 653, 777
    img = synth_image(w, h, seed=band_rows)
    for exact in (1, 0):
        tc = _tc(L, 4)
        dev = L.KLTB200Device(tc)
        L.klt_dev_set_guard(dev, 1)
        L.klt_dev_set_band_rows(dev, band_rows)
        _check_build(L, oracle, img, tc, exact, 0, expect_tiled=True, expect_fused=True)
        assert L.klt_dev_last_build_bands(dev) == -(-h // band_rows)
        _guards_intact(L, dev, "band rows %d, exact %d" % (band_rows, exact))
        L.KLTFreeTrackingContext(tc)


@pytest.mark.parametrize("shape,levels", [((323, 241), 4), ((500, 900), 5), ((2160, 3840), 4)])
def test_fma_chain_equals_unchained_kernels(L, shape, levels):
    h, w = shape
    img = synth_image(w, h, seed=h + w)
    got = {}
    before = L.klt_dev_l0_kernel()
    try:
        for variant in (1, 0):             # 1: chained (default); 0: 64-row level 0 + level_fused_kernel
            L.klt_dev_set_l0_kernel(variant)
            tc = _tc(L, levels)
            dev = L.KLTB200Device(tc)
            L.dev_build(dev, 0, img, L.build_desc(tc, w, h, exact=0))
            assert L.klt_dev_last_build_fused(dev) == levels
            got[variant] = device_pyramids(L, dev, 0, levels)
            L.KLTFreeTrackingContext(tc)
    finally:
        L.klt_dev_set_l0_kernel(before)
    for which in range(3):
        for lv in range(levels):
            a, b = got[1][which][lv], got[0][which][lv]
            assert a.tobytes() == b.tobytes(), "plane %d level %d: %d samples differ" % (
                which, lv, int(np.count_nonzero(a != b)))
