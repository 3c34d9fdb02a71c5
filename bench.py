#!/usr/bin/env python
"""bench.py -- KLT hot-path throughput on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W          (this repo's CUDA path)
  python bench.py --impl reference --gpus N --steps K --warmup W   (the reference's CPU path)

Workload (BASELINE.json configs[3], the configuration the metric is quoted on):
synthetic 3840x2160 translated sequence, 4096 features, 4 pyramid levels
(subsampling 2), 7x7 window.  One step = one KLTTrackFeatures call: build the
three pyramids of one new frame, then track every live feature into it.
Metric: tracked features/s = features with val >= 0 entering the calls / time.
At N > 1 every rank runs its own independent sequence on its own GPU (no
collective on the data path); value is the sum over ranks / max time over ranks.

The same line also carries, at every N, BASELINE.json configs[4] -- the multi-sequence workload
north_star names for 2/4/8 GPUs -- under "config5": 64 independent synthetic 1080p sequences,
1024 features each, sequence s on GPU s mod N, STRONG scaling (total work fixed), one
KLTTrackFeaturesSequence pipeline per sequence over pinned host frames, results checksummed and
gathered on the host; and "h2d_probe": what this box's host->device path delivers per GPU when
all N GPUs copy at once (the ceiling of every end-to-end number).

One JSON line on stdout (rank 0).  Keys are described in DESIGN.md section 6.
"""
from __future__ import annotations

import argparse
import ctypes as C
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
PKG = "klt-feature-tracker-acceleration-gpus_b200"

WORKLOADS = {
    # name: (ncols, nrows, nfeatures, nlevels, subsampling, window, distinct frames)
    "4k": (3840, 2160, 4096, 4, 2, 7, 20),
    "1080p": (1920, 1080, 1024, 2, 4, 7, 64),
    "vga": (640, 480, 1000, 2, 4, 7, 64),
}
METRIC = "tracked_features_per_s"
UNIT = "features/s"


_JSON_FD = None          # the real stdout when fd 1 has been pointed at stderr (multi-rank runs)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def emit_json(obj):
    line = json.dumps(obj) + "\n"
    if _JSON_FD is None:
        sys.stdout.write(line)
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, line.encode())


def workload_config(name):
    """the `config` object, identical in both arms (the driver compares them)"""
    ncols, nrows, nfeat, nlevels, ss, window, nframes = WORKLOADS[name]
    px, w, h = 0, ncols, nrows
    for _ in range(nlevels):
        px += w * h
        w //= ss
        h //= ss
    return {"workload": "synthetic %dx%d translated sequence (2.3,-1.4 px/frame), %d features, %d pyramid levels "
                        "(subsampling %d), window %dx%d, one independent sequence per GPU"
                        % (ncols, nrows, nfeat, nlevels, ss, window, window),
            "l2": "%s: %d distinct frames (%.0f MB) cycled ping-pong; every step also writes "
                  "%.0f MB of new pyramids" % ("inputs larger than L2" if nframes * ncols * nrows > 126e6 else
                                               "inputs SMALLER than the 126 MB L2 (not a valid bench workload)",
                                               nframes, nframes * ncols * nrows / 1e6, 12 * px / 1e6)}


def algorithmic_bytes(ncols, nrows, nlevels, ss):
    """SURVEY 8(d): per new frame, read the u8 frame once + write the three f32
    pyramids: W*H + 12 * sum_l W_l*H_l (integer division per level)."""
    px, w, h = [], ncols, nrows
    for _ in range(nlevels):
        px.append(w * h)
        w //= ss
        h //= ss
    per_kernel = {
        "smooth_u8_tile": 5 * px[0],                                   # read u8, write L0
        "grad_tile": 12 * sum(px),                                     # read L_l, write gx_l, gy_l
        "pyrdown_tile": sum(4 * px[l - 1] + 4 * px[l] for l in range(1, nlevels)),
        "l0_fused_kernel": 13 * px[0],                                 # read u8, write L0, gx0, gy0
        # one pyramid step + that level's gradients: read L_{l-1}, write L_l, gx_l, gy_l
        "level_fused_kernel[level 1]": (4 * px[0] + 12 * px[1]) if nlevels > 1 else 0,
        "level_fused_kernel[level 2]": (4 * px[1] + 12 * px[2]) if nlevels > 2 else 0,
        "level_fused_kernel[level 3+]": sum(4 * px[l - 1] + 12 * px[l] for l in range(3, nlevels)),
        "frame_pipeline": ncols * nrows + 12 * sum(px),                # fully fused floor
    }
    # when level 0 is fused, the stand-alone gradient kernel only sees the coarser levels
    per_kernel["grad_tile_coarse"] = 12 * sum(px[1:])
    return per_kernel, px


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._pump, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r for (t, r) in self.rows if t0 - 0.05 <= t <= t1 + 0.15] or [r for (_, r) in self.rows]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except Exception:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_frames(synth, ncols, nrows, nframes, seed, out):
    for t in range(nframes):
        synth.frame(ncols, nrows, seed=seed, t=float(t), out=out[t])


def setup_tc(L, nlevels, ss, window, device=None):
    tc = L.KLTCreateTrackingContext()
    t = tc.contents
    t.sequentialMode = 1
    t.window_width = t.window_height = window
    t.nPyramidLevels, t.subsampling = nlevels, ss
    if os.environ.get("KLT_BENCH_MAXIT"):          # diagnostic: how much of the tracker is its slowest features
        t.max_iterations = int(os.environ["KLT_BENCH_MAXIT"])
    L.KLTUpdateTCBorder(tc)
    if device is not None:
        L.KLTB200SetDevice(tc, device)
    return tc


# --------------------------------------------------------------------------- config 5
def run_config5(args, L, capi, synth, torch, dist, rank, local_rank, world, barrier):
    """BASELINE.json configs[4] / SURVEY 8(d) config 5: 64 independent synthetic 1920x1080 sequences
    (seed 1000 + s, velocity in [-3, 3]^2 px/frame), 1024 features each, tc defaults (2 levels,
    subsampling 4, 7x7), sequence s -> GPU s mod N.  Strong scaling: the total work is the same at
    every N.  Each sequence is a chain of KLTTrackFeaturesSequence calls (one per segment of frames,
    pinned host frames, per-frame results into a KLT_FeatureTable that the host thread folds into a
    checksum and a compact table); `inflight` sequences per GPU are driven at once from host threads
    so that one sequence's PCIe transfer overlaps another's kernels.  No collective on the data
    path; the per-sequence checksums are gathered on rank 0 afterwards (they must not depend on N)."""
    import queue
    import zlib
    from concurrent.futures import ThreadPoolExecutor
    multiseq = importlib.import_module(PKG + ".multiseq")
    NSEQ, W, H, NF, T = 64, 1920, 1080, 1024, 17
    SEG, NSEG, INFLIGHT = args.c5_segment, args.c5_segments, args.c5_inflight
    mine = multiseq.my_sequences(NSEQ, rank, world)
    vel = np.random.default_rng(2024).uniform(-3.0, 3.0, size=(NSEQ, 2))
    t0 = time.time()
    frames = torch.empty((max(len(mine), 1), T, H, W), dtype=torch.uint8, pin_memory=True)
    fh = frames.numpy()
    for k, s in enumerate(mine):
        for t in range(T):
            synth.frame(W, H, seed=1000 + s, t=float(t), velocity=tuple(vel[s]), out=fh[k, t])
    log("[rank %d] config 5: %d sequences x %d frames generated in %.1fs" % (rank, len(mine), T, time.time() - t0))
    rec = C.sizeof(capi.KLT_FeatureRec)
    ctx = []
    for k, s in enumerate(mine):
        tc = L.KLTCreateTrackingContext()
        tc.contents.sequentialMode = 1
        L.KLTB200SetDevice(tc, local_rank)
        fl = L.KLTCreateFeatureList(NF)
        L.KLTSelectGoodFeatures(tc, C.c_void_p(frames[k, 0].data_ptr()), W, H, fl)
        sel = capi.featurelist_to_arrays(fl)
        segs = []
        for j in range(NSEG):                  # segment j: steps j*SEG .. (j+1)*SEG; its frame 0 = the held pyramid
            segs.append((C.c_void_p * (SEG + 1))(*[frames[k, synth.pingpong_index(j * SEG + i, T)].data_ptr()
                                                   for i in range(SEG + 1)]))
        # warm-up (>= 3 steps per context: pinned rings, kernel attributes), then back to the selection
        L.KLTTrackFeaturesSequence(tc, segs[0], 4, W, H, fl, None, 0, 0)
        L.KLTStopSequentialMode(tc)
        tc.contents.sequentialMode = 1
        capi.arrays_to_featurelist(fl, *sel)
        ctx.append((tc, fl, segs))
    tables = queue.Queue()
    made = []
    for _ in range(max(1, INFLIGHT)):
        ft = L.KLTCreateFeatureTable(SEG + 1, NF)
        C.memset(C.cast(ft.contents.feature[0][0], C.c_void_p), 0, (SEG + 1) * NF * rec)
        made.append(ft)
        tables.put(ft)
    for tc, fl, _ in ctx:
        live = C.c_ulonglong(0)
        L.klt_dev_live_total(L.KLTB200Device(tc), C.byref(live), 1)

    def run_one(k):
        tc, fl, segs = ctx[k]
        ft = tables.get()
        base = C.cast(ft.contents.feature[0][0], C.c_void_p).value
        view = np.frombuffer((C.c_char * ((SEG + 1) * NF * rec)).from_address(base), dtype=capi._REC_DTYPE,
                             count=(SEG + 1) * NF).reshape(NF, SEG + 1)
        crc = 0
        for j in range(NSEG):
            L.KLTTrackFeaturesSequence(tc, segs[j], SEG + 1, W, H, fl, ft, 0, 0)
            for f in ("x", "y", "val"):         # the host gather: columns 1..SEG -> compact, checksummed
                crc = zlib.crc32(np.ascontiguousarray(view[f][:, 1:]).tobytes(), crc)
        tables.put(ft)
        return crc

    barrier()
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=max(1, INFLIGHT)) as pool:
        crcs = list(pool.map(run_one, range(len(ctx))))
    torch.cuda.synchronize()
    secs = time.perf_counter() - t0
    barrier()
    feats = 0
    for tc, fl, _ in ctx:
        live = C.c_ulonglong(0)
        L.klt_dev_live_total(L.KLTB200Device(tc), C.byref(live), 1)
        feats += int(live.value)
    alive = [int(L.KLTCountRemainingFeatures(fl)) for _, fl, _ in ctx]
    local = {int(s): int(c) for s, c in zip(mine, crcs)}
    local_alive = {int(s): a for s, a in zip(mine, alive)}
    if world > 1:
        bucket = [None] * world if rank == 0 else None
        dist.gather_object((local, local_alive), bucket, dst=0)
        t = torch.tensor([secs], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        c = torch.tensor([float(feats)], dtype=torch.float64, device="cuda")
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
        secs, feats = float(t[0]), int(c[0])
        if rank == 0:
            local, local_alive = {}, {}
            for a, b in bucket:
                local.update(a)
                local_alive.update(b)
    for ft in made:
        L.KLTFreeFeatureTable(ft)
    for tc, fl, _ in ctx:
        L.KLTFreeFeatureList(fl)
        L.KLTFreeTrackingContext(tc)
    del frames
    if rank != 0:
        return None
    assert len(local) == NSEQ
    all_crc = 0
    for s in sorted(local):
        all_crc = zlib.crc32(int(local[s]).to_bytes(4, "little"), all_crc)
    nframes_total = NSEQ * SEG * NSEG
    h2d = (SEG * NSEG + 1) * W * H                       # per sequence: every tracked frame + the first one
    return {"metric": METRIC, "value": round(feats / secs, 1), "unit": UNIT, "scaling": "strong",
            "frames_per_s": round(nframes_total / secs, 1), "seconds": round(secs, 4), "n_gpus": world,
            "e2e": {"value": round(feats / secs, 1), "unit": UNIT,
                    "h2d_bytes_per_step": W * H, "d2h_bytes_per_step": 12 * NF,
                    "per_gpu_h2d_gbs": round(NSEQ * h2d / world / secs / 1e9, 1)},
            "config": {"workload": "BASELINE config 5: %d independent synthetic %dx%d sequences, %d features each, "
                                   "%d tracked frames each (%d distinct frames per sequence cycled ping-pong), tc "
                                   "defaults (2 levels, subsampling 4, 7x7), sequence s on GPU s mod N"
                                   % (NSEQ, W, H, NF, SEG * NSEG, T),
                       "api": "KLTTrackFeaturesSequence, %d calls of %d frames per sequence, pinned host frames, "
                              "%d sequences in flight per GPU; value == e2e (there is no resident variant: "
                              "every frame crosses PCIe inside the timed region)" % (NSEG, SEG, INFLIGHT)},
            "tables_crc32": "%08x" % all_crc,
            "features_alive_at_end_min_max": [min(local_alive.values()), max(local_alive.values())]}


# --------------------------------------------------------------------------- configs 2 / 3 at their own size
def small_frame_legs(L, capi, synth, torch):
    """BASELINE configs 2 and 3 are 640x480 sequences (1000 features; 2000 features with
    KLTReplaceLostFeatures after every frame).  The real frames do not travel with the repo (their
    full-length parity report is profiles/r2_full_sequences*.json); this times the same driver loops
    on a synthetic 640x480 sequence of 240 frames (translation + 0.2 deg/frame rotation + 0.1 % zoom)
    through the per-call API and through KLTTrackFeaturesSequence, host frames, wall clock."""
    W, H, NFR = 640, 480, 241
    frames = torch.empty((NFR, H, W), dtype=torch.uint8, pin_memory=True)
    fh = frames.numpy()
    for t in range(NFR):
        synth.frame(W, H, seed=2024, t=float(t), velocity=(1.7, -1.1), rot_deg=0.2, scale=1.001, out=fh[t])
    ptr = lambda i: C.c_void_p(frames.data_ptr() + i * W * H)
    out = {}
    for name, n, replace in (("config2_like", 1000, False), ("config3_like", 2000, True)):
        res = {}
        for api in ("per_call", "sequence"):
            tc = L.KLTCreateTrackingContext()
            tc.contents.sequentialMode = 1
            L.KLTB200SetDevice(tc, torch.cuda.current_device())
            fl = L.KLTCreateFeatureList(n)
            ft = L.KLTCreateFeatureTable(NFR, n)
            C.memset(C.cast(ft.contents.feature[0][0], C.c_void_p), 0, NFR * n * C.sizeof(capi.KLT_FeatureRec))
            L.KLTSelectGoodFeatures(tc, ptr(0), W, H, fl)
            dev = L.KLTB200Device(tc)
            for k in range(1, 9):                         # warm-up on the first frames
                L.KLTTrackFeatures(tc, ptr(k - 1), ptr(k), W, H, fl)
                if replace:
                    L.KLTReplaceLostFeatures(tc, ptr(k), W, H, fl)
            live = C.c_ulonglong(0)
            L.klt_dev_live_total(dev, C.byref(live), 1)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            if api == "per_call":
                for k in range(9, NFR):
                    L.KLTTrackFeatures(tc, ptr(k - 1), ptr(k), W, H, fl)
                    if replace:
                        L.KLTReplaceLostFeatures(tc, ptr(k), W, H, fl)
                    L.KLTStoreFeatureList(fl, ft, k)
            else:
                seq = (C.c_void_p * (NFR - 8))(*[ptr(k).value for k in range(8, NFR)])
                L.KLTTrackFeaturesSequence(tc, seq, NFR - 8, W, H, fl, ft, 8, 1 if replace else 0)
            secs = time.perf_counter() - t0
            L.klt_dev_live_total(dev, C.byref(live), 1)
            res[api] = {"frames_per_s": round((NFR - 9) / secs, 1), "features_per_s": round(int(live.value) / secs, 1),
                        "us_per_frame": round(secs / (NFR - 9) * 1e6, 1),
                        "alive_at_end": int(L.KLTCountRemainingFeatures(fl))}
            L.KLTFreeFeatureTable(ft)
            L.KLTFreeFeatureList(fl)
            L.KLTFreeTrackingContext(tc)
        out[name] = dict(res, features=n, replace=replace)
    out["frames"] = "synthetic %dx%d, %d tracked frames, tc defaults (2 levels, subsampling 4, 7x7)" % (W, H, NFR - 9)
    return out


# --------------------------------------------------------------------------- what a store-heavy kernel can get
def write_ceiling():
    """tools/write_probe.bin (built by __graft_entry__.build): a kernel that does nothing but read the
    u8 frame and write three float planes in the level-0 kernel's own tile pattern, back to back on
    buffers larger than L2.  The roofline denominator (a copy: half reads, half writes) is not
    reachable for traffic that is 92 % stores; this is."""
    exe = os.path.join(ROOT, "tools", "write_probe.bin")
    if not os.path.exists(exe):
        return None
    try:
        txt = subprocess.run([exe], capture_output=True, text=True, timeout=120).stdout
    except Exception:
        return None
    out = {}
    for line in txt.splitlines():
        f = line.split()
        if line.startswith("tiled  64x48  4 CTAs/SM +u8"):
            out["tiled_fill_plus_u8_us"] = float(f[f.index("us") - 1])
        elif line.startswith("fill     grid 2368"):
            out["fill_only_us"] = float(f[f.index("us") - 1])
        elif line.startswith("cudaMemcpy D2D"):
            out["memcpy_d2d_gbs"] = float(f[f.index("GB/s") - 1])
    return out or None


# --------------------------------------------------------------------------- host I/O (SURVEY 8f N4)
def io_throughput(L, capi, fh):
    """Feature-table / PPM writers and the PGM reader: this library vs the reference's own C code
    (oracle/_ref), same inputs, byte-identical outputs (tests/test_host.py), wall clock per call."""
    import tempfile
    ref, _ = _ref_library(capi)
    W, H, NF, NFR = 640, 480, 1000, 200
    img = np.ascontiguousarray(fh[0][:H, :W])
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        for name, lib in (("b200", L), ("reference", ref)):
            if lib is None:
                continue
            fl = lib.KLTCreateFeatureList(NF)
            ft = lib.KLTCreateFeatureTable(NFR, NF)
            rng = np.random.default_rng(5)
            x = rng.uniform(10, W - 10, NF).astype(np.float32)
            y = rng.uniform(10, H - 10, NF).astype(np.float32)
            v = np.zeros(NF, np.int32)
            capi.arrays_to_featurelist(fl, x, y, v)
            for k in range(NFR):
                lib.KLTStoreFeatureList(fl, ft, k)
            ppm = os.path.join(tmp, name + ".ppm").encode()
            txt = os.path.join(tmp, name + ".txt").encode()
            bin_ = os.path.join(tmp, name + ".ft").encode()
            pgm = os.path.join(tmp, name + ".pgm").encode()
            lib.pgmWriteFile(pgm, img.ctypes.data_as(C.c_void_p), W, H)
            buf = np.empty((H, W), np.uint8)
            nc, nr = C.c_int(0), C.c_int(0)

            def timeit(fn, reps):
                fn()
                t0 = time.perf_counter()
                for _ in range(reps):
                    fn()
                return (time.perf_counter() - t0) / reps
            e = {}
            e["KLTWriteFeatureListToPPM_ms"] = round(1e3 * timeit(
                lambda: lib.KLTWriteFeatureListToPPM(fl, img.ctypes.data_as(C.c_void_p), W, H, ppm), 20), 3)
            e["pgmReadFile_ms"] = round(1e3 * timeit(
                lambda: lib.pgmReadFile(pgm, buf.ctypes.data_as(C.c_void_p), C.byref(nc), C.byref(nr)), 50), 3)
            e["KLTWriteFeatureTable_text_ms"] = round(1e3 * timeit(
                lambda: lib.KLTWriteFeatureTable(ft, txt, b"%5.1f"), 3), 2)
            e["KLTWriteFeatureTable_binary_ms"] = round(1e3 * timeit(
                lambda: lib.KLTWriteFeatureTable(ft, bin_, None), 5), 3)
            lib.KLTFreeFeatureTable(ft)
            lib.KLTFreeFeatureList(fl)
            out[name] = e
    out["case"] = "640x480 frame, %d features, %d-frame table; files on the box's tmpfs/disk" % (NF, NFR)
    return out


def dump_features(L, dev, n, out_dir):
    """The resident features as a caller of KLTB200ResidentEnd would receive them, written as
    out_dir/x.npy, y.npy (float32) and val.npy (the int32 status / eigenvalue, exact in float64), so
    that two builds can be compared output for output.  Synchronises; changes no device state."""
    x, y, val = np.empty(n, np.float32), np.empty(n, np.float32), np.empty(n, np.int32)
    L.dev_check(dev, L.klt_dev_features_download(dev, n, x, y, val))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("x", x), ("y", y), ("val", val.astype(np.float64))):
        np.save(os.path.join(out_dir, name + ".npy"), a)


# --------------------------------------------------------------------------- B200 arm
def run_b200(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist

    pkg = importlib.import_module(PKG)
    rt = importlib.import_module(PKG + ".runtime")
    synth = importlib.import_module(PKG + ".synth")
    capi = pkg.capi
    L = rt.load()
    L.require_gpu()
    L.KLTSetVerbosity(0)
    torch.cuda.set_device(local_rank)
    if world > 1:
        # NCCL prints its version banner / debug lines on the process's stdout (fd 1, from C): point
        # fd 1 at stderr for the whole run and keep the real stdout for the one JSON line
        global _JSON_FD
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ncols, nrows, nfeat, nlevels, ss, window, nframes = WORKLOADS[args.workload]
    K, W = args.steps, args.warmup
    tc = setup_tc(L, nlevels, ss, window, device=local_rank)
    dev = L.KLTB200Device(tc)

    # ---- synthetic sequence: pinned host copy + HBM-resident copy -------------------
    t0 = time.time()
    # (KLT_BENCH_PAGEABLE=1: ordinary host memory, what a driver that mallocs its frames gets)
    frames_h = torch.empty((nframes, nrows, ncols), dtype=torch.uint8,
                           pin_memory=not os.environ.get("KLT_BENCH_PAGEABLE"))
    fh = frames_h.numpy()
    make_frames(synth, ncols, nrows, nframes, 12345 + rank, fh)
    frames_d = frames_h.cuda(non_blocking=False)
    torch.cuda.synchronize()
    fbytes = ncols * nrows
    d_ptr = lambda i: frames_d.data_ptr() + i * fbytes
    h_ptr = lambda i: frames_h.data_ptr() + i * fbytes
    log("[rank %d] %d frames %dx%d generated in %.1fs" % (rank, nframes, ncols, nrows, time.time() - t0))

    # ---- select on frame 0 (not part of the metric) ----------------------------------
    fl = L.KLTCreateFeatureList(nfeat)
    t0 = time.time()
    L.KLTSelectGoodFeatures(tc, C.c_void_p(h_ptr(0)), ncols, nrows, fl)
    t_select = time.time() - t0
    t0 = time.time()
    L.KLTSelectGoodFeatures(tc, C.c_void_p(h_ptr(0)), ncols, nrows, fl)
    t_select2 = time.time() - t0
    sel = capi.featurelist_to_arrays(fl)
    nsel = int((sel[2] > 0).sum())
    log("[rank %d] selected %d/%d features (first call %.1f ms, second %.1f ms)"
        % (rank, nsel, nfeat, t_select * 1e3, t_select2 * 1e3))

    def restart():
        L.KLTStopSequentialMode(tc)
        tc.contents.sequentialMode = 1
        capi.arrays_to_featurelist(fl, *sel)

    idx = lambda s: synth.pingpong_index(s, nframes)

    # ---- (1) value: frames resident in HBM, features resident, no host sync ----------
    # (nvidia-smi is sampled every 100 ms from here to the end of the e2e legs; the rows taken are
    # those between the start of the first timed region and the end of the last)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    restart()
    L.KLTB200ResidentBegin(tc, C.c_void_p(d_ptr(0)), 1, ncols, ncols, nrows, fl)
    step = 1
    for _ in range(W):
        L.KLTB200ResidentStep(tc, C.c_void_p(d_ptr(idx(step))), 1, ncols, ncols, nrows)
        step += 1
    live = C.c_ulonglong(0)
    L.klt_dev_live_total(dev, C.byref(live), 1)
    launches0 = L.klt_dev_launch_count(dev)
    barrier()
    wall0 = time.time()
    L.klt_dev_timer_start(dev)
    for _ in range(K):
        L.KLTB200ResidentStep(tc, C.c_void_p(d_ptr(idx(step))), 1, ncols, ncols, nrows)
        step += 1
    ms = C.c_float(0)
    L.klt_dev_timer_stop(dev, C.byref(ms))
    barrier()
    launches = int(L.klt_dev_launch_count(dev) - launches0)
    L.klt_dev_live_total(dev, C.byref(live), 1)
    dev_ms, dev_feats = float(ms.value), int(live.value)
    if args.dump_outputs and rank == 0:
        dump_features(L, dev, nfeat, args.dump_outputs)
    # ---- (1b) the same loop for max(K, 2000) more steps: a timed region of >= 0.1 s (K = 20 is 1.5 ms)
    KS = max(K, 2000)
    barrier()
    L.klt_dev_timer_start(dev)
    for _ in range(KS):
        L.KLTB200ResidentStep(tc, C.c_void_p(d_ptr(idx(step))), 1, ncols, ncols, nrows)
        step += 1
    L.klt_dev_timer_stop(dev, C.byref(ms))
    barrier()
    L.klt_dev_live_total(dev, C.byref(live), 1)
    sus_ms, sus_feats = float(ms.value), int(live.value)
    L.KLTB200ResidentEnd(tc, fl)
    alive_end = int(L.KLTCountRemainingFeatures(fl))

    # ---- (2) e2e: the public KLTTrackFeatures call, pinned HOST frames ---------------
    restart()
    step = 1
    for _ in range(W):
        L.KLTTrackFeatures(tc, C.c_void_p(h_ptr(idx(step - 1))), C.c_void_p(h_ptr(idx(step))), ncols, nrows, fl)
        step += 1
    L.klt_dev_live_total(dev, C.byref(live), 1)          # numerator counted on the device, as in (1)
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        L.KLTTrackFeatures(tc, C.c_void_p(h_ptr(idx(step - 1))), C.c_void_p(h_ptr(idx(step))), ncols, nrows, fl)
        step += 1
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()
    L.klt_dev_live_total(dev, C.byref(live), 1)
    e2e_feats = int(live.value)

    # ---- (2b) e2e, batched: KLTTrackFeaturesSequence over the same pinned HOST frames -----
    # (one call for K frames, per-frame results into a feature table; frame k+1 crosses PCIe while
    # frame k is processed; the call returns after its single synchronisation)
    restart()
    ft = L.KLTCreateFeatureTable(K + 1, nfeat)
    C.memset(C.cast(ft.contents.feature[0][0], C.c_void_p), 0,          # map the table's pages now
             (K + 1) * nfeat * C.sizeof(capi.KLT_FeatureRec))
    warm = (C.c_void_p * (W + 1))(*[h_ptr(idx(s)) for s in range(W + 1)])
    # (with a table, so that the pinned snapshot ring exists before the timed call)
    L.KLTTrackFeaturesSequence(tc, warm, W + 1, ncols, nrows, fl, ft if W <= K else None, 0, 0)
    seq = (C.c_void_p * (K + 1))(*[h_ptr(idx(W + s)) for s in range(K + 1)])
    L.klt_dev_live_total(dev, C.byref(live), 1)
    barrier()
    t0 = time.perf_counter()
    L.KLTTrackFeaturesSequence(tc, seq, K + 1, ncols, nrows, fl, ft, 0, 0)
    seq_s = time.perf_counter() - t0
    barrier()
    L.klt_dev_live_total(dev, C.byref(live), 1)
    seq_feats = int(live.value)
    L.KLTFreeFeatureTable(ft)
    wall1 = time.time()
    clocks = sampler.stop(wall0, wall1) if sampler else None

    # ---- (2c) e2e with PAGEABLE frames: what the reference's own driver passes (it mallocs its two
    # images and refills them, src/V3/example3.c:45-46,75).  Two ordinary numpy buffers are refilled
    # from the sequence before every call (outside the timed sum).  Default: staged through pinned
    # memory by the staging team; "registered": the buffers are page-locked in place on second sight
    # (opt-in, KLT_B200_REGISTER_FRAMES=1).  N = 1 only (torchrun pins every rank to one host thread).
    pageable = None
    if world == 1:
        pageable = {}
        bufs = [np.empty((nrows, ncols), np.uint8) for _ in range(2)]
        for mode in ("staged", "registered"):
            L.klt_dev_set_register_frames(dev, 1 if mode == "registered" else 0)
            restart()
            np.copyto(bufs[0], fh[idx(0)])
            step, secs, feats_p = 1, 0.0, 0
            KP = max(K, 50)
            for it in range(W + KP):
                cur, prv = bufs[step & 1], bufs[(step - 1) & 1]
                np.copyto(cur, fh[idx(step)])                     # the driver's pgmReadFile into its buffer
                if it == W:
                    L.klt_dev_live_total(dev, C.byref(live), 1)
                t0 = time.perf_counter()
                L.KLTTrackFeatures(tc, C.c_void_p(prv.ctypes.data), C.c_void_p(cur.ctypes.data), ncols, nrows, fl)
                if it >= W:
                    secs += time.perf_counter() - t0
                step += 1
            L.klt_dev_live_total(dev, C.byref(live), 1)
            pageable[mode] = {"value": round(int(live.value) / secs, 1), "unit": UNIT,
                              "ms_per_step": round(secs / KP * 1e3, 4), "steps": KP,
                              "host_buffers_page_locked_in_place": int(L.klt_dev_registered_host_frames(dev))}
            L.KLTStopSequentialMode(tc)                            # drops the registrations
            tc.contents.sequentialMode = 1
        L.klt_dev_set_register_frames(dev, 0)

    # ---- (2d) what the box's host->device path gives each GPU when all N copy at once ----------
    probe_src = frames_h[:4]
    probe_dst = torch.empty_like(frames_d[:4])
    st = torch.cuda.Stream()
    ncopies = 64
    with torch.cuda.stream(st):
        for i in range(8):
            probe_dst[i % 4].copy_(probe_src[i % 4], non_blocking=True)
        st.synchronize()
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(st)
        for i in range(ncopies):
            probe_dst[i % 4].copy_(probe_src[i % 4], non_blocking=True)
        ev1.record(st)
        st.synchronize()
    barrier()
    h2d_gbs = ncopies * fbytes / (ev0.elapsed_time(ev1) * 1e-3) / 1e9
    del probe_dst

    # ---- (5) BASELINE config 5: 64 independent 1080p sequences over the N GPUs (strong scaling) ----
    c5 = None if args.only_4k else run_config5(args, L, capi, synth, torch, dist, rank, local_rank, world, barrier)

    # ---- (3) per-kernel device time (CUDA events on the launching stream) ------------
    restart()
    L.KLTB200ResidentBegin(tc, C.c_void_p(d_ptr(0)), 1, ncols, ncols, nrows, fl)
    step = 1
    for _ in range(min(W, 5)):
        L.KLTB200ResidentStep(tc, C.c_void_p(d_ptr(idx(step))), 1, ncols, ncols, nrows)
        step += 1
    L.klt_dev_profile_begin(dev)
    for _ in range(K):
        L.KLTB200ResidentStep(tc, C.c_void_p(d_ptr(idx(step))), 1, ncols, ncols, nrows)
        step += 1
    L.klt_dev_profile_end(dev)
    prof = L.profile(dev)
    L.KLTB200ResidentEnd(tc, fl)

    # ---- (4) the level-0 kernel alone, launched back to back (no event pair per launch: the
    # brackets of pass (3) add the launch latency that the frame chain hides) ----------------
    l0_b2b_ms = None
    if "l0_fused_kernel" in prof:
        q0 = L.build_desc(tc, ncols, nrows, nlevels_built=1, exact=0)
        nb2b = max(10, min(K, 200))
        for i in range(5):
            L.klt_dev_build(dev, i % 3, C.c_void_p(d_ptr(idx(i))), 1, ncols, C.byref(q0))
        L.klt_dev_timer_start(dev)
        for i in range(nb2b):
            L.klt_dev_build(dev, i % 3, C.c_void_p(d_ptr(idx(i))), 1, ncols, C.byref(q0))
        ms0 = C.c_float(0)
        L.klt_dev_timer_stop(dev, C.byref(ms0))
        l0_b2b_ms = float(ms0.value) / nb2b

    # ---- reduce over ranks: sum of features, max of time -------------------------------
    h2d_min = h2d_sum = h2d_gbs
    if world > 1:
        t = torch.tensor([dev_ms, e2e_s, seq_s, sus_ms, -h2d_gbs], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        c = torch.tensor([dev_feats, e2e_feats, seq_feats, sus_feats, h2d_gbs], dtype=torch.float64, device="cuda")
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
        dev_ms, e2e_s, seq_s, sus_ms, h2d_min = float(t[0]), float(t[1]), float(t[2]), float(t[3]), -float(t[4])
        dev_feats, e2e_feats, seq_feats, sus_feats, h2d_sum = int(c[0]), int(c[1]), int(c[2]), int(c[3]), float(c[4])

    if rank == 0:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy)"
        else:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        bytes_tab, px = algorithmic_bytes(ncols, nrows, nlevels, ss)
        kernels = {}
        for name, (n, tot) in prof.items():
            per_step = tot / K
            ent = {"launches_per_step": n / K, "ms_per_step": round(per_step, 5)}
            key = name
            if name == "grad_tile" and "l0_fused_kernel" in prof:
                key = "grad_tile_coarse"
            if key in bytes_tab:
                ent["algorithmic_bytes_per_step"] = bytes_tab[key]
                ent["gbs"] = round(bytes_tab[key] / (per_step * 1e-3) / 1e9, 1)
            kernels[name] = ent
        pipe = ["smooth_u8_tile", "grad_tile", "pyrdown_tile", "l0_fused_kernel", "level_fused_kernel[level 1]",
                "level_fused_kernel[level 2]", "level_fused_kernel[level 3+]"]
        hbm_kernels = {k: v for k, v in kernels.items() if "gbs" in v}
        dom = max(hbm_kernels, key=lambda k: hbm_kernels[k]["ms_per_step"]) if hbm_kernels else None
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if dom and os.path.exists(tpath):
            traffic = json.load(open(tpath)).get(dom)
        roofline = None
        if dom:
            d = kernels[dom]
            roofline = {"kernel": dom, "bound": "hbm", "achieved": d["gbs"], "peak": peak, "unit": "GB/s",
                        "frac": round(d["gbs"] / peak, 4), "traffic": traffic, "peak_source": peak_src,
                        "bytes_per_step": d["algorithmic_bytes_per_step"],
                        "launches_per_step": d["launches_per_step"], "ms_per_step": d["ms_per_step"]}
            if dom == "l0_fused_kernel" and l0_b2b_ms:
                g = d["algorithmic_bytes_per_step"] / (l0_b2b_ms * 1e-3) / 1e9
                roofline["back_to_back"] = {
                    "ms_per_launch": round(l0_b2b_ms, 5), "gbs": round(g, 1), "frac": round(g / peak, 4),
                    "how": "the same kernel launched back to back on distinct frames between ONE pair of "
                           "events (level-0-only builds): its steady-state rate without the per-launch "
                           "event brackets of `kernels`"}
            wc = write_ceiling() if dom == "l0_fused_kernel" else None
            if wc and "tiled_fill_plus_u8_us" in wc:
                t_att = wc["tiled_fill_plus_u8_us"] * 1e-6
                roofline["attainable"] = dict(
                    wc, gbs=round(d["algorithmic_bytes_per_step"] / t_att / 1e9, 1),
                    frac_of_peak=round(d["algorithmic_bytes_per_step"] / t_att / 1e9 / peak, 4),
                    kernel_vs_attainable=round(t_att / (l0_b2b_ms * 1e-3), 4) if l0_b2b_ms else None,
                    how="tools/write_probe.cu on the same GPU in the same run: the time of a kernel that only "
                        "moves this kernel's bytes (1 B read + 12 B written per pixel, same 64x48 tile store "
                        "pattern, 4 CTAs per SM, back to back); kernel_vs_attainable = that time / the "
                        "kernel's back-to-back time")
            pipe_ms = sum(v["ms_per_step"] for k, v in kernels.items() if k in pipe)
            if pipe_ms > 0:
                roofline["frame_pipeline"] = {
                    "algorithmic_bytes_per_step": bytes_tab["frame_pipeline"], "ms_per_step": round(pipe_ms, 5),
                    "gbs": round(bytes_tab["frame_pipeline"] / (pipe_ms * 1e-3) / 1e9, 1),
                    "frac": round(bytes_tab["frame_pipeline"] / (pipe_ms * 1e-3) / 1e9 / peak, 4)}
        value = dev_feats / (dev_ms * 1e-3)
        out = {
            "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": round(dev_ms / K, 5), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "frames_per_s": round(K * world / (dev_ms * 1e-3), 1),
            "config": workload_config(args.workload),
            "details": {"features_selected": nsel, "features_alive_at_end": alive_end,
                        "arithmetic": "fma (default mode); exact mode is the parity-test mode",
                        "select_ms": round(t_select2 * 1e3, 2)},
            "sustained": {"steps": KS, "ms_per_step": round(sus_ms / KS, 5),
                          "value": round(sus_feats / (sus_ms * 1e-3), 1), "unit": UNIT,
                          "how": "the loop of `value` continued for max(K, 2000) steps between one pair of events"},
            "e2e": {"value": round(e2e_feats / e2e_s, 1), "unit": UNIT,
                    "frames_per_s": round(K * world / e2e_s, 1), "ms_per_step": round(e2e_s / K * 1e3, 4),
                    "h2d_bytes_per_step": fbytes + 64 * nfeat, "d2h_bytes_per_step": 12 * nfeat,
                    "api": "KLTTrackFeatures(tc, img1, img2, ncols, nrows, fl) with pinned host frames; the frame "
                           "goes up in 2 bands behind which the pyramid kernels run, the feature records "
                           "(64 B each) are mirrored in one copy and the tracker writes x|y|val (12 B) of "
                           "every feature straight into the caller's pinned feature list"},
            "e2e_sequence": {"value": round(seq_feats / seq_s, 1), "unit": UNIT,
                             "frames_per_s": round(K * world / seq_s, 1), "ms_per_step": round(seq_s / K * 1e3, 4),
                             "h2d_bytes_per_step": fbytes, "d2h_bytes_per_step": 12 * nfeat,
                             "api": "KLTTrackFeaturesSequence(tc, frames[K+1], ..., fl, ft, 0, 0): one call for K "
                                    "pinned host frames, per-frame x|y|val snapshots into a KLT_FeatureTable; the "
                                    "upload of frame k+1 overlaps the kernels of frame k (PCIe-bound), one "
                                    "synchronisation at the end; wall clock around the call"},
            "gpu_launches": launches, "kernels": kernels, "roofline": roofline, "clocks": clocks,
            "h2d_probe": {"per_gpu_gbs_min": round(h2d_min, 1), "aggregate_gbs": round(h2d_sum, 1),
                          "e2e_per_gpu_gbs": round((fbytes + 64 * nfeat) * K / e2e_s / 1e9, 1),
                          "e2e_sequence_per_gpu_gbs": round(fbytes * K / seq_s / 1e9, 1),
                          "how": "every rank copies 64 pinned %.1f MB frames to its GPU back to back, all ranks "
                                 "at once, CUDA events; e2e_*: bytes the end-to-end legs move per second per GPU"
                                 % (fbytes / 1e6)},
            "config5": c5,
        }
        if pageable is not None:
            out["e2e_pageable"] = dict(pageable["staged"], api="KLTTrackFeatures with two ordinary (pageable) frame "
                                       "buffers refilled by the driver every frame, as the reference's example3 does; "
                                       "staged through pinned memory by the library")
            out["e2e_pageable_registered"] = dict(pageable["registered"], api="same buffers, page-locked in place by "
                                                  "the library on second sight (KLT_B200_REGISTER_FRAMES=1, opt-in)")
        if world == 1 and not args.no_cpu_baseline and not args.only_4k:
            out["cpu_baseline"] = cpu_baseline(capi, fh, ncols, nrows, nfeat, nlevels, ss, window,
                                               budget_s=args.cpu_budget)
            try:
                out["small_frames"] = small_frame_legs(L, capi, synth, torch)
            except Exception as e:
                out["small_frames"] = {"error": repr(e)}
            try:
                out["host_io"] = io_throughput(L, capi, fh)
            except Exception as e:                      # never lose the bench line over the I/O side show
                out["host_io"] = {"error": repr(e)}
        emit_json(out)
    barrier()
    L.KLTFreeFeatureList(fl)
    L.KLTFreeTrackingContext(tc)
    if world > 1:
        dist.destroy_process_group()


# --------------------------------------------------------------------------- CPU legs
def _ref_library(capi):
    from oracle import oracle_py
    if os.path.exists(oracle_py.REF_PATH):
        return capi.KLTLibrary(oracle_py.REF_PATH), "reference"
    return None, "port"


def _cpu_sequence(capi, frames, ncols, nrows, nfeat, nlevels, ss, window, warmup, steps, budget_s,
                  start_evt=None):
    """select + track on the CPU reference; returns (features, seconds in KLTTrackFeatures, steps)."""
    lib, kind = _ref_library(capi)
    nframes = len(frames)
    idx = lambda s: s % (2 * (nframes - 1)) if s % (2 * (nframes - 1)) < nframes else 2 * (nframes - 1) - s % (2 * (nframes - 1))
    if lib is not None:
        lib.KLTSetVerbosity(0)
        tc = setup_tc(lib, nlevels, ss, window)
        fl = lib.KLTCreateFeatureList(nfeat)
        ptr = lambda i: C.c_void_p(frames[i].ctypes.data)
        lib.KLTSelectGoodFeatures(tc, ptr(0), ncols, nrows, fl)
        track = lambda a, b: lib.KLTTrackFeatures(tc, ptr(a), ptr(b), ncols, nrows, fl)
        count = lambda: lib.KLTCountRemainingFeatures(fl)
    else:                                           # plain-C port (oracle/klt_oracle.c)
        from oracle import oracle_py
        o = oracle_py.Oracle()
        p = o.default_params()
        p.window_width = p.window_height = window
        p.nPyramidLevels, p.subsampling = nlevels, ss
        o.update_border(p)
        state = {"xyv": o.select(frames[0], p, nfeat), "prev": o.build_pyramids(frames[0], p)}

        def track(a, b):
            cur = o.build_pyramids(frames[b], p)
            state["xyv"] = o.track(state["prev"], cur, p, *state["xyv"])
            state["prev"] = cur
        count = lambda: int((state["xyv"][2] >= 0).sum())
    step = 1
    for _ in range(warmup):
        track(idx(step - 1), idx(step))
        step += 1
    if start_evt is not None:
        start_evt()
    feats, secs, done = 0, 0.0, 0
    for _ in range(steps):
        feats += count()
        t0 = time.perf_counter()
        track(idx(step - 1), idx(step))
        secs += time.perf_counter() - t0
        step += 1
        done += 1
        if secs > budget_s:
            break
    return feats, secs, done, kind


def cpu_baseline(capi, frames, ncols, nrows, nfeat, nlevels, ss, window, budget_s=20.0):
    feats, secs, done, kind = _cpu_sequence(capi, frames[:6], ncols, nrows, nfeat, nlevels, ss, window,
                                            warmup=1, steps=1000, budget_s=budget_s)
    return {"value": round(feats / secs, 1), "unit": UNIT, "cores": 1, "kind": kind,
            "frames_per_s": round(done / secs, 3),
            "sample": "1 sequence on 1 host core: KLTSelectGoodFeatures + 1 warm-up + %d timed "
                      "KLTTrackFeatures calls on the same %dx%d frames / %d features (wall clock around "
                      "KLTTrackFeatures only, as the reference driver times it)" % (done, ncols, nrows, nfeat)}


_REF_FRAMES = None          # the synthetic frames, generated once in the parent and inherited by the forked workers


def _ref_worker(args):
    (widx, workload, warmup, steps, budget_s) = args
    pkg = importlib.import_module(PKG)
    ncols, nrows, nfeat, nlevels, ss, window, _ = WORKLOADS[workload]
    t_begin = [0.0]
    feats, secs, done, kind = _cpu_sequence(pkg.capi, _REF_FRAMES, ncols, nrows, nfeat, nlevels, ss, window,
                                            warmup, steps, budget_s,
                                            start_evt=lambda: t_begin.__setitem__(0, time.time()))
    return feats, secs, done, kind, t_begin[0], time.time()


def run_reference(args, rank, world):
    """The reference's own CPU implementation (oracle/_ref = its unmodified sources compiled in
    place), on all host cores: the library is single-threaded, so one independent sequence per core
    (every worker runs the same synthetic sequence; nothing is shared but the read-only frames)."""
    if rank != 0:
        return
    import multiprocessing as mp
    global _REF_FRAMES
    pkg = importlib.import_module(PKG)
    synth = importlib.import_module(PKG + ".synth")
    ncols, nrows, nfeat, nlevels, ss, window, nframes = WORKLOADS[args.workload]
    # load the library in THIS process too (the forked workers inherit the mapping): the driver
    # records the native libraries of the process it launched
    lib, kind0 = _ref_library(pkg.capi)
    cores = os.cpu_count() or 1
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        pass
    per_proc_gb = 0.75 * (ncols * nrows) / (3840 * 2160)
    try:
        avail_gb = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE") / 2 ** 30
    except Exception:
        avail_gb = 16.0
    procs = max(1, min(cores, 64, int(avail_gb * 0.6 / max(per_proc_gb, 1e-3))))
    _REF_FRAMES = np.empty((nframes, nrows, ncols), np.uint8)
    make_frames(synth, ncols, nrows, nframes, 12345, _REF_FRAMES)
    # a reference step at 4K costs about half a second: the timed loop is bounded by --ref-budget
    jobs = [(w, args.workload, args.warmup, args.steps, args.ref_budget) for w in range(procs)]
    t0 = time.time()
    with mp.get_context("fork").Pool(procs) as pool:
        res = pool.map(_ref_worker, jobs)
    feats = sum(r[0] for r in res)
    frames_done = sum(r[2] for r in res)
    span = max(r[5] for r in res) - min(r[4] for r in res)     # wall time of the timed phase
    busy = max(r[1] for r in res)                               # slowest worker's time inside the calls
    secs = max(busy, 1e-9)
    kind = res[0][3]
    steps_done = min(r[2] for r in res)
    value = feats / secs
    sample = ("%d copies of the sequence in parallel (one per host core, the library is single-threaded), "
              "each: select + %d warm-up + %d timed KLTTrackFeatures calls at %dx%d / %d features; "
              "timed-phase wall %.1fs" % (procs, args.warmup, steps_done, ncols, nrows, nfeat, span))
    out = {
        "impl": "reference", "metric": METRIC, "value": round(value, 1), "unit": UNIT,
        "n_gpus": args.gpus, "steps": steps_done, "warmup": args.warmup,
        "ms_per_step": round(secs / max(steps_done, 1) * 1e3, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "frames_per_s": round(frames_done / secs, 3),
        "config": workload_config(args.workload),
        "cpu_baseline": {"value": round(value, 1), "unit": UNIT, "cores": procs, "kind": kind, "sample": sample},
        "e2e": {"value": round(value, 1), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "total_wall_s": round(time.time() - t0, 1),
    }
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="4k", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-budget", type=float, default=15.0, help="seconds of CPU work for cpu_baseline")
    ap.add_argument("--ref-budget", type=float, default=90.0,
                    help="--impl reference: stop a worker's timed loop after this many seconds")
    ap.add_argument("--only-4k", action="store_true", help="development: skip config 5 and the CPU legs")
    ap.add_argument("--c5-segment", type=int, default=128, help="config 5: frames per KLTTrackFeaturesSequence call")
    ap.add_argument("--c5-segments", type=int, default=8, help="config 5: calls per sequence")
    ap.add_argument("--c5-inflight", type=int, default=4, help="config 5: sequences in flight per GPU")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the features the timed loop of `value` holds after its last step (rank 0) "
                         "to DIR/x.npy, y.npy, val.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.warmup < 3:
        log("warmup raised to 3 (timing rules)")
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_b200(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
