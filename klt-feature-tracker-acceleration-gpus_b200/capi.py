"""ctypes mirror of the KLT C API (include/klt.h, include/pnmio.h).

This is the Python-side host binding of the *reference's own interface* for the
hot path: the same struct layouts (reference src/V4/klt.h:41-122) and the same
function names / argument meaning (src/V4/klt.h:131-233, src/V4/pnmio.h:13-49).
It binds ANY shared library that exports that API, so the parity tests drive the
B200 library and the compiled reference oracle through identical code.

Nothing in here computes anything: it is plumbing around `ctypes.CDLL`.
"""
from __future__ import annotations

import ctypes as C
import numpy as np

KLT_TRACKED = 0
KLT_NOT_FOUND = -1
KLT_SMALL_DET = -2
KLT_MAX_ITERATIONS = -3
KLT_OOB = -4
KLT_LARGE_RESIDUE = -5
KLT_B200_FB_INCONSISTENT = -6      # include/klt_b200.h: rejected by the forward-backward check
KLT_B200_MOTION_OUTLIER = -7       # include/klt_b200.h: rejected by the global motion check

STATUS_NAMES = {
    0: "TRACKED", -1: "NOT_FOUND", -2: "SMALL_DET", -3: "MAX_ITERATIONS",
    -4: "OOB", -5: "LARGE_RESIDUE",
}


class KLT_TrackingContextRec(C.Structure):
    """reference src/V4/klt.h:41-89 (136 bytes on LP64)."""
    _fields_ = [
        ("mindist", C.c_int),
        ("window_width", C.c_int),
        ("window_height", C.c_int),
        ("sequentialMode", C.c_int),
        ("smoothBeforeSelecting", C.c_int),
        ("writeInternalImages", C.c_int),
        ("lighting_insensitive", C.c_int),
        ("min_eigenvalue", C.c_int),
        ("min_determinant", C.c_float),
        ("min_displacement", C.c_float),
        ("max_iterations", C.c_int),
        ("max_residue", C.c_float),
        ("grad_sigma", C.c_float),
        ("smooth_sigma_fact", C.c_float),
        ("pyramid_sigma_fact", C.c_float),
        ("step_factor", C.c_float),
        ("nSkippedPixels", C.c_int),
        ("borderx", C.c_int),
        ("bordery", C.c_int),
        ("nPyramidLevels", C.c_int),
        ("subsampling", C.c_int),
        ("affine_window_width", C.c_int),
        ("affine_window_height", C.c_int),
        ("affineConsistencyCheck", C.c_int),
        ("affine_max_iterations", C.c_int),
        ("affine_max_residue", C.c_float),
        ("affine_min_displacement", C.c_float),
        ("affine_max_displacement_differ", C.c_float),
        ("pyramid_last", C.c_void_p),
        ("pyramid_last_gradx", C.c_void_p),
        ("pyramid_last_grady", C.c_void_p),
    ]


class KLT_FeatureRec(C.Structure):
    """reference src/V4/klt.h:92-106 (64 bytes on LP64)."""
    _fields_ = [
        ("x", C.c_float),
        ("y", C.c_float),
        ("val", C.c_int),
        ("aff_img", C.c_void_p),
        ("aff_img_gradx", C.c_void_p),
        ("aff_img_grady", C.c_void_p),
        ("aff_x", C.c_float),
        ("aff_y", C.c_float),
        ("aff_Axx", C.c_float),
        ("aff_Ayx", C.c_float),
        ("aff_Axy", C.c_float),
        ("aff_Ayy", C.c_float),
    ]


KLT_Feature = C.POINTER(KLT_FeatureRec)


class KLT_FeatureListRec(C.Structure):
    _fields_ = [("nFeatures", C.c_int), ("feature", C.POINTER(KLT_Feature))]


class KLT_FeatureHistoryRec(C.Structure):
    _fields_ = [("nFrames", C.c_int), ("feature", C.POINTER(KLT_Feature))]


class KLT_FeatureTableRec(C.Structure):
    _fields_ = [("nFrames", C.c_int), ("nFeatures", C.c_int),
                ("feature", C.POINTER(C.POINTER(KLT_Feature)))]


KLT_TrackingContext = C.POINTER(KLT_TrackingContextRec)
KLT_FeatureList = C.POINTER(KLT_FeatureListRec)
KLT_FeatureHistory = C.POINTER(KLT_FeatureHistoryRec)
KLT_FeatureTable = C.POINTER(KLT_FeatureTableRec)

_u8p = C.POINTER(C.c_ubyte)

# name -> (restype, argtypes); the 29 prototypes of klt.h + 6 of pnmio.h
PUBLIC_API = {
    "KLTCreateTrackingContext": (KLT_TrackingContext, []),
    "KLTCreateFeatureList": (KLT_FeatureList, [C.c_int]),
    "KLTCreateFeatureHistory": (KLT_FeatureHistory, [C.c_int]),
    "KLTCreateFeatureTable": (KLT_FeatureTable, [C.c_int, C.c_int]),
    "KLTFreeTrackingContext": (None, [KLT_TrackingContext]),
    "KLTFreeFeatureList": (None, [KLT_FeatureList]),
    "KLTFreeFeatureHistory": (None, [KLT_FeatureHistory]),
    "KLTFreeFeatureTable": (None, [KLT_FeatureTable]),
    "KLTSelectGoodFeatures": (None, [KLT_TrackingContext, C.c_void_p, C.c_int, C.c_int, KLT_FeatureList]),
    "KLTTrackFeatures": (None, [KLT_TrackingContext, C.c_void_p, C.c_void_p, C.c_int, C.c_int, KLT_FeatureList]),
    "KLTReplaceLostFeatures": (None, [KLT_TrackingContext, C.c_void_p, C.c_int, C.c_int, KLT_FeatureList]),
    "KLTCountRemainingFeatures": (C.c_int, [KLT_FeatureList]),
    "KLTPrintTrackingContext": (None, [KLT_TrackingContext]),
    "KLTChangeTCPyramid": (None, [KLT_TrackingContext, C.c_int]),
    "KLTUpdateTCBorder": (None, [KLT_TrackingContext]),
    "KLTStopSequentialMode": (None, [KLT_TrackingContext]),
    "KLTSetVerbosity": (None, [C.c_int]),
    "_KLTComputeSmoothSigma": (C.c_float, [KLT_TrackingContext]),
    "KLTStoreFeatureList": (None, [KLT_FeatureList, KLT_FeatureTable, C.c_int]),
    "KLTExtractFeatureList": (None, [KLT_FeatureList, KLT_FeatureTable, C.c_int]),
    "KLTStoreFeatureHistory": (None, [KLT_FeatureHistory, KLT_FeatureTable, C.c_int]),
    "KLTExtractFeatureHistory": (None, [KLT_FeatureHistory, KLT_FeatureTable, C.c_int]),
    "KLTWriteFeatureListToPPM": (None, [KLT_FeatureList, C.c_void_p, C.c_int, C.c_int, C.c_char_p]),
    "KLTWriteFeatureList": (None, [KLT_FeatureList, C.c_char_p, C.c_char_p]),
    "KLTWriteFeatureHistory": (None, [KLT_FeatureHistory, C.c_char_p, C.c_char_p]),
    "KLTWriteFeatureTable": (None, [KLT_FeatureTable, C.c_char_p, C.c_char_p]),
    "KLTReadFeatureList": (KLT_FeatureList, [KLT_FeatureList, C.c_char_p]),
    "KLTReadFeatureHistory": (KLT_FeatureHistory, [KLT_FeatureHistory, C.c_char_p]),
    "KLTReadFeatureTable": (KLT_FeatureTable, [KLT_FeatureTable, C.c_char_p]),
    # pnmio.h
    "pgmReadFile": (C.c_void_p, [C.c_char_p, C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "pgmWriteFile": (None, [C.c_char_p, C.c_void_p, C.c_int, C.c_int]),
    "ppmWriteFileRGB": (None, [C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    "pgmRead": (C.c_void_p, [C.c_void_p, C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "pgmWrite": (None, [C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    "ppmWrite": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
}


def _as_u8_ptr(img):
    """Accept a C-contiguous uint8 numpy array, a raw int address, or None."""
    if img is None:
        return None
    if isinstance(img, int):
        return C.c_void_p(img)
    a = np.ascontiguousarray(img)
    if a.dtype != np.uint8:
        raise TypeError("KLT images are unsigned char (uint8)")
    return a.ctypes.data_as(C.c_void_p)


class KLTLibrary:
    """A loaded shared library exporting the KLT C API."""

    def __init__(self, path: str):
        self.path = path
        self.lib = C.CDLL(path, mode=C.RTLD_LOCAL)
        for name, (res, args) in PUBLIC_API.items():
            fn = getattr(self.lib, name)
            fn.restype = res
            fn.argtypes = args

    def __getattr__(self, name):
        # anything not wrapped below is forwarded to the raw C function
        return getattr(self.lib, name)

    # -- thin conveniences (no computation) ---------------------------------
    def create_context(self, **fields):
        tc = self.lib.KLTCreateTrackingContext()
        for k, v in fields.items():
            setattr(tc.contents, k, v)
        return tc

    def select(self, tc, img, fl):
        a = np.ascontiguousarray(img)
        self.lib.KLTSelectGoodFeatures(tc, _as_u8_ptr(a), a.shape[1], a.shape[0], fl)

    def track(self, tc, img1, img2, fl):
        a = np.ascontiguousarray(img1)
        b = np.ascontiguousarray(img2)
        self.lib.KLTTrackFeatures(tc, _as_u8_ptr(a), _as_u8_ptr(b), b.shape[1], b.shape[0], fl)

    def replace(self, tc, img, fl):
        a = np.ascontiguousarray(img)
        self.lib.KLTReplaceLostFeatures(tc, _as_u8_ptr(a), a.shape[1], a.shape[0], fl)

    def read_pgm(self, fname: str) -> np.ndarray:
        nc, nr = C.c_int(0), C.c_int(0)
        hdr = self.lib.pgmReadFile(fname.encode(), None, C.byref(nc), C.byref(nr))
        buf = (C.c_ubyte * (nc.value * nr.value)).from_address(hdr)
        out = np.frombuffer(buf, dtype=np.uint8).reshape(nr.value, nc.value).copy()
        _libc_free(hdr)
        return out


_libc = C.CDLL(None)
_libc.free.argtypes = [C.c_void_p]
_libc.free.restype = None


def _libc_free(p):
    _libc.free(C.c_void_p(p))


# -- feature-list <-> numpy ---------------------------------------------------
_REC_DTYPE = np.dtype({"names": ["x", "y", "val"], "formats": ["f4", "f4", "i4"], "offsets": [0, 4, 8],
                       "itemsize": C.sizeof(KLT_FeatureRec)})


def _records_view(fl):
    """numpy view of the KLT_FeatureRec array when the list is the one block KLTCreateFeatureList
    makes (header, pointer array, records back to back: reference klt.c:148-167); None otherwise"""
    n = fl.contents.nFeatures
    if n < 1:
        return None
    f = fl.contents.feature
    a0 = C.addressof(f[0].contents)
    if C.addressof(f[n - 1].contents) != a0 + (n - 1) * C.sizeof(KLT_FeatureRec):
        return None
    buf = (C.c_char * (n * C.sizeof(KLT_FeatureRec))).from_address(a0)
    return np.frombuffer(buf, dtype=_REC_DTYPE, count=n)


def featurelist_to_arrays(fl):
    n = fl.contents.nFeatures
    rec = _records_view(fl)
    if rec is not None:
        return rec["x"].copy(), rec["y"].copy(), rec["val"].copy()
    x = np.empty(n, np.float32)
    y = np.empty(n, np.float32)
    v = np.empty(n, np.int32)
    f = fl.contents.feature
    for i in range(n):
        r = f[i].contents
        x[i], y[i], v[i] = r.x, r.y, r.val
    return x, y, v


def featurelist_affine(fl):
    """the affine-consistency members of every feature (klt.h:97-105): has = aff_img != NULL"""
    n = fl.contents.nFeatures
    out = np.zeros(n, dtype=[("has", "i4"), ("aff_x", "f4"), ("aff_y", "f4"), ("Axx", "f4"), ("Ayx", "f4"),
                             ("Axy", "f4"), ("Ayy", "f4")])
    f = fl.contents.feature
    for i in range(n):
        r = f[i].contents
        out[i] = (1 if r.aff_img else 0, r.aff_x, r.aff_y, r.aff_Axx, r.aff_Ayx, r.aff_Axy, r.aff_Ayy)
    return out


def arrays_to_featurelist(fl, x, y, v):
    n = fl.contents.nFeatures
    rec = _records_view(fl)
    if rec is not None:
        rec["x"][:] = np.asarray(x, np.float32)[:n]
        rec["y"][:] = np.asarray(y, np.float32)[:n]
        rec["val"][:] = np.asarray(v, np.int32)[:n]
        return
    f = fl.contents.feature
    for i in range(n):
        r = f[i].contents
        r.x, r.y, r.val = float(x[i]), float(y[i]), int(v[i])


def featuretable_to_array(ft):
    """-> structured array [nFeatures, nFrames] of (x, y, val)."""
    nf, nfr = ft.contents.nFeatures, ft.contents.nFrames
    out = np.zeros((nf, nfr), dtype=[("x", "f4"), ("y", "f4"), ("val", "i4")])
    if nf > 0 and nfr > 0:
        # a table made by KLTCreateFeatureTable keeps its records in one [feature][frame] block
        # (reference klt.c:210-236)
        rows = ft.contents.feature
        a0 = C.addressof(rows[0][0].contents)
        if C.addressof(rows[nf - 1][nfr - 1].contents) == a0 + (nf * nfr - 1) * C.sizeof(KLT_FeatureRec):
            buf = (C.c_char * (nf * nfr * C.sizeof(KLT_FeatureRec))).from_address(a0)
            rec = np.frombuffer(buf, dtype=_REC_DTYPE, count=nf * nfr).reshape(nf, nfr)
            out["x"], out["y"], out["val"] = rec["x"], rec["y"], rec["val"]
            return out
    for j in range(nf):
        row = ft.contents.feature[j]
        for i in range(nfr):
            r = row[i].contents
            out[j, i] = (r.x, r.y, r.val)
    return out


def read_pgm_numpy(fname: str) -> np.ndarray:
    """Pure-numpy P5 reader (handles '#' comments) for tests and benches."""
    with open(fname, "rb") as fh:
        data = fh.read()
    pos = 0
    toks = []
    while len(toks) < 4:
        while data[pos:pos + 1].isspace():
            pos += 1
        if data[pos:pos + 1] == b"#":
            while data[pos:pos + 1] != b"\n":
                pos += 1
            continue
        s = pos
        while not data[pos:pos + 1].isspace():
            pos += 1
        toks.append(data[s:pos])
    pos += 1  # single whitespace after maxval
    assert toks[0] == b"P5", toks
    w, h = int(toks[1]), int(toks[2])
    return np.frombuffer(data, dtype=np.uint8, count=w * h, offset=pos).reshape(h, w).copy()
