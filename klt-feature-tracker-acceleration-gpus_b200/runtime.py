"""Loader and ctypes mirror of the native library (lib/libklt_b200.so).

There is no Python/CPU implementation behind this module: if the native
library is missing, or no CUDA device is present when the hot path is entered,
it raises -- loudly -- instead of falling back.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import capi

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("KLT_B200_LIB") or os.path.join(HERE, "lib", "libklt_b200.so")   # (env: A/B builds)
MAX_TAPS = 71


class DevTaps(C.Structure):           # include/klt_cuda.h: klt_dev_taps
    _fields_ = [("gauss_width", C.c_int), ("deriv_width", C.c_int),
                ("gauss", C.c_float * MAX_TAPS), ("deriv", C.c_float * MAX_TAPS)]


class BuildDesc(C.Structure):         # klt_dev_build_desc
    _fields_ = [("ncols", C.c_int), ("nrows", C.c_int), ("nlevels", C.c_int),
                ("subsampling", C.c_int), ("nlevels_built", C.c_int), ("smooth", C.c_int),
                ("exact", C.c_int), ("smooth_taps", DevTaps), ("pyramid_taps", DevTaps),
                ("grad_taps", DevTaps)]


class TrackParams(C.Structure):       # klt_dev_track_params
    _fields_ = [("window_width", C.c_int), ("window_height", C.c_int),
                ("step_factor", C.c_float), ("max_iterations", C.c_int),
                ("min_determinant", C.c_float), ("min_displacement", C.c_float),
                ("max_residue", C.c_float), ("borderx", C.c_int), ("bordery", C.c_int),
                ("exact", C.c_int), ("lighting_insensitive", C.c_int), ("fb_max_error", C.c_float),
                ("predict", C.c_int), ("motion_max_error", C.c_float), ("motion_hypotheses", C.c_int)]


class MotionModel(C.Structure):       # klt_dev_motion_model / KLT_B200_MotionModel
    _fields_ = [("H", C.c_float * 9), ("valid", C.c_int), ("tracked", C.c_int), ("inliers", C.c_int),
                ("hypothesis", C.c_int)]


class SelectParams(C.Structure):      # klt_dev_select_params
    _fields_ = [("window_width", C.c_int), ("window_height", C.c_int), ("borderx", C.c_int),
                ("bordery", C.c_int), ("nSkippedPixels", C.c_int), ("mindist", C.c_int),
                ("min_eigenvalue", C.c_int), ("overwrite_all", C.c_int)]


_f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
_TC = capi.KLT_TrackingContext
_FL = capi.KLT_FeatureList

# every symbol include/klt_cuda.h and include/klt_b200.h declare
DEV_API = {
    "klt_dev_count": (C.c_int, []),
    "klt_dev_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "klt_dev_destroy": (None, [C.c_void_p]),
    "klt_dev_error": (C.c_char_p, [C.c_void_p]),
    "klt_dev_create_error": (C.c_char_p, []),
    "klt_dev_device": (C.c_int, [C.c_void_p]),
    "klt_dev_stream": (C.c_void_p, [C.c_void_p]),
    "klt_dev_build": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_size_t, C.POINTER(BuildDesc)]),
    "klt_dev_slot_valid": (C.c_int, [C.c_void_p, C.c_int]),
    "klt_dev_exact_level0": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int)]),
    "klt_dev_invalidate": (None, [C.c_void_p, C.c_int]),
    "klt_dev_geometry": (C.c_int, [C.c_void_p] + [C.POINTER(C.c_int)] * 4),
    "klt_dev_track": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(TrackParams), C.c_int, _f32p, _f32p, _i32p]),
    "klt_dev_features_upload": (C.c_int, [C.c_void_p, C.c_int, _f32p, _f32p, _i32p]),
    "klt_dev_track_resident": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(TrackParams)]),
    "klt_dev_disable_track7w": (None, [C.c_void_p, C.c_int]),
    "klt_dev_features_download": (C.c_int, [C.c_void_p, C.c_int, _f32p, _f32p, _i32p]),
    "klt_dev_features_staging": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.POINTER(C.c_float)),
                                           C.POINTER(C.POINTER(C.c_float)), C.POINTER(C.POINTER(C.c_int))]),
    "klt_dev_features_commit": (C.c_int, [C.c_void_p, C.c_int]),
    "klt_dev_features_fetch": (C.c_int, [C.c_void_p, C.c_int]),
    "klt_dev_features_commit_records": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]),
    "klt_dev_host_alloc": (C.c_void_p, [C.c_size_t]),
    "klt_dev_host_free": (None, [C.c_void_p]),
    "klt_dev_select": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(SelectParams), C.c_int, _f32p, _f32p, _i32p]),
    "klt_dev_read_level": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, _f32p]),
    "klt_dev_level_dims": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "klt_dev_eigen_map": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(SelectParams), C.c_void_p, C.POINTER(C.c_int)]),
    "klt_dev_sync": (C.c_int, [C.c_void_p]),
    "klt_dev_set_overlap": (C.c_int, [C.c_void_p, C.c_int]),
    "klt_dev_slots": (C.c_int, []),
    "klt_dev_launch_count": (C.c_ulonglong, [C.c_void_p]),
    "klt_dev_last_build_path": (C.c_int, [C.c_void_p]),
    "klt_dev_force_generic": (None, [C.c_void_p, C.c_int]),
    "klt_dev_disable_fused": (None, [C.c_void_p, C.c_int]),
    "klt_dev_set_l0_kernel": (None, [C.c_int]),
    "klt_dev_set_guard": (None, [C.c_void_p, C.c_int]),
    "klt_dev_plane_address": (C.c_void_p, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "klt_dev_poke": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "klt_dev_check_guards": (C.c_int, [C.c_void_p, C.POINTER(C.c_longlong), C.POINTER(C.c_int)]),
    "klt_dev_l0_kernel": (C.c_int, []),
    "klt_dev_last_build_fused": (C.c_int, [C.c_void_p]),
    "klt_dev_set_band_rows": (None, [C.c_void_p, C.c_int]),
    "klt_dev_last_build_bands": (C.c_int, [C.c_void_p]),
    "klt_dev_forget_host_frames": (C.c_int, [C.c_void_p]),
    "klt_dev_registered_host_frames": (C.c_int, [C.c_void_p]),
    "klt_dev_set_register_frames": (None, [C.c_void_p, C.c_int]),
    "klt_dev_set_stage_threads": (None, [C.c_void_p, C.c_int]),
    "klt_dev_last_build_staged": (C.c_int, [C.c_void_p]),
    "klt_dev_timer_start": (C.c_int, [C.c_void_p]),
    "klt_dev_timer_stop": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "klt_dev_profile_begin": (C.c_int, [C.c_void_p]),
    "klt_dev_profile_end": (C.c_int, [C.c_void_p]),
    "klt_dev_profile_kernels": (C.c_int, []),
    "klt_dev_profile_get": (C.c_char_p, [C.c_void_p, C.c_int, C.POINTER(C.c_ulonglong), C.POINTER(C.c_double)]),
    "klt_dev_trace_count": (C.c_int, [C.c_void_p]),
    "klt_dev_trace_get": (C.c_char_p, [C.c_void_p, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "klt_dev_live_total": (C.c_int, [C.c_void_p, C.POINTER(C.c_ulonglong), C.c_int]),
    "klt_dev_fb_results": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "klt_dev_set_guesses": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "klt_dev_guesses_pending": (C.c_int, [C.c_void_p]),
    "klt_dev_prediction_results": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "klt_dev_motion_results": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "klt_dev_motion_models": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "klt_dev_motion_counts": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    # include/klt_b200.h
    "KLTB200SetDevice": (None, [_TC, C.c_int]),
    "KLTB200SetExact": (None, [_TC, C.c_int]),
    "KLTB200GetExact": (C.c_int, [_TC]),
    "KLTB200SetForwardBackward": (None, [_TC, C.c_float]),
    "KLTB200GetForwardBackward": (C.c_float, [_TC]),
    "KLTB200ForwardBackwardResult": (None, [_TC, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "KLTB200SetPrediction": (None, [_TC, C.c_int]),
    "KLTB200GetPrediction": (C.c_int, [_TC]),
    "KLTB200SetGuesses": (None, [_TC, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "KLTB200PredictionResult": (None, [_TC, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "KLTB200SetMotionCheck": (None, [_TC, C.c_float, C.c_int]),
    "KLTB200GetMotionCheck": (C.c_float, [_TC, C.POINTER(C.c_int)]),
    "KLTB200MotionResult": (None, [_TC, C.c_int, C.c_void_p]),
    "KLTB200MotionModels": (None, [_TC, C.c_int, C.c_void_p]),
    "KLTB200Device": (C.c_void_p, [_TC]),
    "KLTB200LastSlot": (C.c_int, [_TC]),
    "KLTTrackFeaturesDevice": (None, [_TC, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, _FL]),
    "KLTB200ResidentBegin": (None, [_TC, C.c_void_p, C.c_int, C.c_size_t, C.c_int, C.c_int, _FL]),
    "KLTB200ResidentStep": (None, [_TC, C.c_void_p, C.c_int, C.c_size_t, C.c_int, C.c_int]),
    "KLTB200ResidentEnd": (None, [_TC, _FL]),
    "KLTTrackFeaturesSequence": (None, [_TC, C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, _FL,
                                        capi.KLT_FeatureTable, C.c_int, C.c_int]),
    "klt_dev_features_capacity": (C.c_int, [C.c_void_p]),
    "klt_dev_snapshot_ring": (C.c_int, [C.c_void_p, C.c_int]),
    "klt_dev_snapshot_push": (C.c_int, [C.c_void_p, C.c_int]),
    "klt_dev_snapshot_wait": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                        C.POINTER(C.c_void_p)]),
    "klt_dev_select_resident": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(SelectParams)]),
    # host helpers shared with the tests
    "klt_fill_build_desc": (None, [_TC, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(BuildDesc)]),
    "_KLTGetKernelWidths": (None, [C.c_float, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
}


class NativeLibraryMissing(ImportError):
    pass


class B200Library(capi.KLTLibrary):
    """libklt_b200.so: the KLT C API plus the device C-ABI."""

    def __init__(self, path: str = LIB_PATH):
        if not os.path.exists(path):
            raise NativeLibraryMissing(
                "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(make -C klt-feature-tracker-acceleration-gpus_b200/csrc). "
                "There is no CPU fallback for the KLT hot path." % path)
        super().__init__(path)
        for name, (res, args) in DEV_API.items():
            fn = getattr(self.lib, name)
            fn.restype = res
            fn.argtypes = args

    def device_count(self) -> int:
        return self.lib.klt_dev_count()

    def require_gpu(self) -> None:
        if self.device_count() < 1:
            raise RuntimeError("no CUDA device visible: the KLT hot path runs only on the GPU "
                               "(no CPU fallback)")

    def track_sequence(self, tc, frames, fl, ft=None, first_frame=0, replace=False):
        """KLTTrackFeaturesSequence over a list of uint8 arrays / raw host addresses of one size
        (include/klt_b200.h): the batched form of the reference's driver loop."""
        keep, ptrs = [], (C.c_void_p * len(frames))()
        nrows = ncols = None
        for i, f in enumerate(frames):
            if isinstance(f, tuple):                       # (address, nrows, ncols)
                ptrs[i], nrows, ncols = f[0], f[1], f[2]
                continue
            a = np.ascontiguousarray(f, np.uint8)
            keep.append(a)
            ptrs[i] = a.ctypes.data
            nrows, ncols = a.shape
        self.lib.KLTTrackFeaturesSequence(tc, ptrs, len(frames), ncols, nrows, fl, ft, first_frame,
                                          1 if replace else 0)

    # -- device-level helpers used by stage parity tests --------------------
    def dev_check(self, dev, rc):
        if rc != 0:
            raise RuntimeError("klt_dev: " + (self.lib.klt_dev_error(dev) or b"?").decode())

    def build_desc(self, tc, ncols, nrows, nlevels_built=None, smooth=1, exact=0) -> BuildDesc:
        q = BuildDesc()
        if nlevels_built is None:
            nlevels_built = tc.contents.nPyramidLevels
        self.lib.klt_fill_build_desc(tc, ncols, nrows, nlevels_built, smooth, exact, C.byref(q))
        return q

    def dev_build(self, dev, slot, img, desc, device_ptr=None, pitch=None):
        if device_ptr is not None:
            rc = self.lib.klt_dev_build(dev, slot, C.c_void_p(device_ptr), 1, pitch, C.byref(desc))
        else:
            a = np.ascontiguousarray(img, np.uint8)
            rc = self.lib.klt_dev_build(dev, slot, a.ctypes.data_as(C.c_void_p), 0, a.shape[1], C.byref(desc))
            self.dev_check(dev, self.lib.klt_dev_sync(dev))     # `a` must outlive the copy
        self.dev_check(dev, rc)

    def dev_level(self, dev, slot, which, level) -> np.ndarray:
        w, h = C.c_int(0), C.c_int(0)
        if self.lib.klt_dev_level_dims(dev, level, C.byref(w), C.byref(h)) != 0:
            raise RuntimeError("bad level %d" % level)
        out = np.empty((h.value, w.value), np.float32)
        self.dev_check(dev, self.lib.klt_dev_read_level(dev, slot, which, level, out))
        return out

    def track_params(self, tc, exact=0, fb_max_error=0.0, predict=0, motion_max_error=0.0,
                     motion_hypotheses=0) -> TrackParams:
        t = tc.contents
        return TrackParams(t.window_width, t.window_height, t.step_factor, t.max_iterations,
                           t.min_determinant, t.min_displacement, t.max_residue,
                           t.borderx, t.bordery, exact, t.lighting_insensitive, fb_max_error, predict,
                           motion_max_error, motion_hypotheses)

    @staticmethod
    def _models(models) -> dict:
        """{H: (count, 3, 3) float32, valid, tracked, inliers, hypothesis: (count,) int32}"""
        raw = np.frombuffer(models, np.uint8).reshape(len(models), C.sizeof(MotionModel))
        return {"H": raw[:, :36].copy().view(np.float32).reshape(-1, 3, 3),
                **{k: raw[:, 36 + 4 * i:40 + 4 * i].copy().view(np.int32).ravel()
                   for i, k in enumerate(("valid", "tracked", "inliers", "hypothesis"))}}

    def motion_result(self, tc, n):
        """KLTB200MotionResult: per-feature reprojection distance of the last tracking call on tc"""
        err = np.empty(n, np.float32)
        self.lib.KLTB200MotionResult(tc, n, err.ctypes.data)
        return err

    def motion_models(self, tc, count):
        """KLTB200MotionModels: the models of the last `count` checked calls on tc, oldest first"""
        out = (MotionModel * count)()
        self.lib.KLTB200MotionModels(tc, count, C.cast(out, C.c_void_p))
        return self._models(out)

    def dev_motion_results(self, dev, n):
        """klt_dev_motion_results: per-feature reprojection distance of the last klt_dev_track* call"""
        err = np.empty(n, np.float32)
        self.dev_check(dev, self.lib.klt_dev_motion_results(dev, n, err.ctypes.data))
        return err

    def dev_motion_models(self, dev, count):
        """klt_dev_motion_models: the models of the last `count` checked klt_dev_track* calls"""
        out = (MotionModel * count)()
        self.dev_check(dev, self.lib.klt_dev_motion_models(dev, count, C.cast(out, C.c_void_p)))
        return self._models(out)

    def dev_motion_counts(self, dev, hyps):
        """klt_dev_motion_counts: (m, per-hypothesis inlier counts, -1: no model) of the last checked call"""
        m, counts = C.c_int(0), np.empty(hyps, np.int32)
        self.dev_check(dev, self.lib.klt_dev_motion_counts(dev, hyps, C.byref(m), counts.ctypes.data))
        return m.value, counts

    def set_guesses(self, tc, gx, gy, on_device=False):
        """KLTB200SetGuesses for the next tracking call on tc: float32 host arrays, or with on_device
        contiguous float32 CUDA tensors (complete: synchronise their stream first)"""
        if on_device:
            if gx.numel() != gy.numel():
                raise ValueError("gx and gy differ in size")
            self.lib.KLTB200SetGuesses(tc, gx.numel(), C.c_void_p(gx.data_ptr()), C.c_void_p(gy.data_ptr()), 1)
            return
        gx = np.ascontiguousarray(gx, np.float32)
        gy = np.ascontiguousarray(gy, np.float32)
        if gx.shape != gy.shape:
            raise ValueError("gx and gy differ in shape")
        self.lib.KLTB200SetGuesses(tc, gx.size, gx.ctypes.data, gy.ctypes.data, 0)

    def prediction(self, tc, n):
        """KLTB200PredictionResult: (gx, gy, source) of the last tracking call on tc"""
        gx, gy, src = np.empty(n, np.float32), np.empty(n, np.float32), np.empty(n, np.int32)
        self.lib.KLTB200PredictionResult(tc, n, gx.ctypes.data, gy.ctypes.data, src.ctypes.data)
        return gx, gy, src

    def dev_prediction(self, dev, n):
        """klt_dev_prediction_results: (gx, gy, source) of the last klt_dev_track* call on dev"""
        gx, gy, src = np.empty(n, np.float32), np.empty(n, np.float32), np.empty(n, np.int32)
        self.dev_check(dev, self.lib.klt_dev_prediction_results(dev, n, gx.ctypes.data, gy.ctypes.data,
                                                                src.ctypes.data))
        return gx, gy, src

    def forward_backward(self, tc, n):
        """KLTB200ForwardBackwardResult: (xb, yb, err, back_val) of the last tracking call on tc"""
        xb, yb, err = np.empty(n, np.float32), np.empty(n, np.float32), np.empty(n, np.float32)
        bv = np.empty(n, np.int32)
        self.lib.KLTB200ForwardBackwardResult(tc, n, xb.ctypes.data, yb.ctypes.data, err.ctypes.data, bv.ctypes.data)
        return xb, yb, err, bv

    def dev_forward_backward(self, dev, n):
        """klt_dev_fb_results: (xb, yb, err, back_val) of the last klt_dev_track* call on dev"""
        xb, yb, err = np.empty(n, np.float32), np.empty(n, np.float32), np.empty(n, np.float32)
        bv = np.empty(n, np.int32)
        self.dev_check(dev, self.lib.klt_dev_fb_results(dev, n, xb.ctypes.data, yb.ctypes.data, err.ctypes.data,
                                                        bv.ctypes.data))
        return xb, yb, err, bv

    def select_params(self, tc, overwrite_all=1) -> SelectParams:
        t = tc.contents
        return SelectParams(t.window_width, t.window_height, t.borderx, t.bordery,
                            t.nSkippedPixels, t.mindist, t.min_eigenvalue, overwrite_all)

    def dev_eigen_map(self, dev, slot, sp) -> np.ndarray:
        n = C.c_int(0)
        self.dev_check(dev, self.lib.klt_dev_eigen_map(dev, slot, C.byref(sp), None, C.byref(n)))
        out = np.empty(n.value, np.int32)
        if n.value:
            self.dev_check(dev, self.lib.klt_dev_eigen_map(dev, slot, C.byref(sp),
                                                           out.ctypes.data_as(C.c_void_p), C.byref(n)))
        return out


    def profile(self, dev) -> dict:
        """{kernel class: (launches, total ms)} accumulated since klt_dev_profile_begin"""
        out = {}
        for k in range(self.lib.klt_dev_profile_kernels()):
            n, ms = C.c_ulonglong(0), C.c_double(0.0)
            name = self.lib.klt_dev_profile_get(dev, k, C.byref(n), C.byref(ms))
            if name and n.value:
                out[name.decode()] = (int(n.value), float(ms.value))
        return out


    def trace(self, dev) -> list:
        """[(class name, start ms, end ms)] of the last profiling session, launch order"""
        out = []
        for i in range(self.lib.klt_dev_trace_count(dev)):
            t0, t1 = C.c_float(0), C.c_float(0)
            name = self.lib.klt_dev_trace_get(dev, i, C.byref(t0), C.byref(t1))
            out.append((name.decode(), float(t0.value), float(t1.value)))
        return out


_cached = None


def load() -> B200Library:
    global _cached
    if _cached is None:
        _cached = B200Library()
    return _cached
