"""Guard mode over every buffer a tracking context grows (klt_dev_set_guard, include/klt_cuda.h).

In guard mode each device buffer the context grows -- feature arrays, record mirror, positions before
tracking, affine states and templates, forward-backward and prediction records, guesses, motion check
buffers, selection buffers, frame staging -- sits between two canary bands.  One context runs every
feature of the library on lists of 7, 1025 and 5000 features and on frames of growing size, so that
each of those buffers is re-allocated at least once, and no canary word may change."""
import numpy as np
import pytest

from tests.conftest import synth_image
from tests.test_gpu_guards import _guards_intact

pytestmark = pytest.mark.gpu

EXPLICIT = 2   # KLTB200PredictionResult source of an explicit guess


@pytest.fixture(scope="module")
def L(pkg):
    from importlib import import_module
    lib = import_module(pkg.__name__ + ".runtime").load()
    lib.require_gpu()
    lib.KLTSetVerbosity(0)
    return lib


def test_every_grown_buffer_stays_inside_its_allocation(L, capi):
    tc = L.KLTCreateTrackingContext()
    tc.contents.sequentialMode = 1
    tc.contents.mindist = 5
    dev = L.KLTB200Device(tc)
    L.klt_dev_set_guard(dev, 1)
    L.KLTB200SetForwardBackward(tc, 0.5)
    L.KLTB200SetPrediction(tc, 1)                           # velocity
    for n, (w, h), hyps in ((7, (320, 240), 100), (1025, (640, 480), 1500), (5000, (1280, 960), 5000)):
        frames = [synth_image(w, h, n, shift=(1.5 * k, -1.0 * k)) for k in range(7)]
        fl = L.KLTCreateFeatureList(n)
        ft = L.KLTCreateFeatureTable(len(frames) - 3, n)
        L.select(tc, frames[0], fl)
        # per call: affine check, forward-backward check, velocity and explicit guesses, motion check
        tc.contents.affineConsistencyCheck = 1
        L.KLTB200SetMotionCheck(tc, 1.0, hyps)
        L.track(tc, frames[0], frames[1], fl)
        x, y, _ = capi.featurelist_to_arrays(fl)
        L.set_guesses(tc, x + np.float32(1.5), y - np.float32(1.0))
        L.track(tc, frames[1], frames[2], fl)
        assert (L.prediction(tc, n)[2] == EXPLICIT).any()
        L.forward_backward(tc, n)
        L.motion_result(tc, n)
        L.replace(tc, frames[2], fl)
        # record mode: the tracker reads a device mirror of the pinned list (no affine or motion check)
        tc.contents.affineConsistencyCheck = -1
        L.KLTB200SetMotionCheck(tc, 0.0, 0)
        L.track(tc, frames[2], frames[3], fl)
        L.replace(tc, frames[3], fl)
        # sequence call with every check on
        tc.contents.affineConsistencyCheck = 1
        L.KLTB200SetMotionCheck(tc, 1.0, hyps)
        L.track_sequence(tc, frames[3:], fl, ft, 0, True)
        assert (capi.featurelist_to_arrays(fl)[2] >= 0).any()
        _guards_intact(L, dev, "%d features, %dx%d" % (n, w, h))
        L.KLTFreeFeatureTable(ft)
        L.KLTFreeFeatureList(fl)
    L.KLTFreeTrackingContext(tc)
