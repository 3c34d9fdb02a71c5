"""Cost and effect of the motion prior (KLTB200SetPrediction / KLTB200SetGuesses): prediction off,
velocity, and explicit guesses, alternated in one process.

  * 4K: 3840x2160, 4096 features, 4 levels (subsampling 2), 7x7 -- the resident pipeline of bench.py's
    `value` leg over 20 distinct HBM-resident frames (166 MB, larger than the 126 MB L2), device
    events around the steps; every round restarts from the same selection.  "explicit" hands the
    step all-NaN host guesses (a guess per feature that is no guess): the copy and the per-feature
    read are paid, the tracking is that of prediction off.
  * the tracker kernel alone, from the klt_dev_profile_* event brackets (a separate profiled run).
  * 640x480 accelerating pan (3 px/frame^2, up to 48 px/frame; tests/predict_oracle.py pan_frames),
    300 features, tc defaults (2 levels, subsampling 4, 7x7), KLTTrackFeatures per call without
    replacement: tracked results and their error against the exact pan, prediction off / velocity.

Prints one JSON object (also written to --out); the card and its power limit are read in the same run.
"""
import argparse
import ctypes as C
import importlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PKG = "klt-feature-tracker-acceleration-gpus_b200"
MODES = (("off", 0, False), ("velocity", 1, False), ("explicit", 0, True))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                     # (the measurement itself does not depend on it)
        return {"error": str(e)}


def run_4k(L, capi, synth, torch, rounds, steps):
    W, H, N, LV, SS, NF = 3840, 2160, 4096, 4, 2, 20
    tc = L.KLTCreateTrackingContext()
    t = tc.contents
    t.sequentialMode = 1
    t.nPyramidLevels, t.subsampling = LV, SS
    L.KLTUpdateTCBorder(tc)
    L.KLTB200SetDevice(tc, torch.cuda.current_device())
    dev = L.KLTB200Device(tc)
    fh = torch.empty((NF, H, W), dtype=torch.uint8, pin_memory=True)
    for k in range(NF):
        synth.frame(W, H, seed=12345, t=float(k), out=fh[k].numpy())
    fd = fh.cuda()
    torch.cuda.synchronize()
    ptr = lambda i: C.c_void_p(fd.data_ptr() + synth.pingpong_index(i, NF) * W * H)
    fl = L.KLTCreateFeatureList(N)
    L.KLTSelectGoodFeatures(tc, C.c_void_p(fh.data_ptr()), W, H, fl)
    sel = capi.featurelist_to_arrays(fl)
    nan = np.full(N, np.nan, np.float32)

    def step(s, explicit):
        if explicit:
            L.set_guesses(tc, nan, nan)
        L.KLTB200ResidentStep(tc, ptr(s), 1, W, W, H)

    def leg(mode, explicit, k, profile=False):
        L.KLTStopSequentialMode(tc)
        tc.contents.sequentialMode = 1
        capi.arrays_to_featurelist(fl, *sel)
        L.KLTB200SetPrediction(tc, mode)
        L.KLTB200ResidentBegin(tc, ptr(0), 1, W, W, H, fl)
        for s in range(1, 21):
            step(s, explicit)
        L.klt_dev_sync(dev)
        ms = C.c_float(0)
        if profile:
            L.klt_dev_profile_begin(dev)
        else:
            L.klt_dev_timer_start(dev)
        for s in range(21, 21 + k):
            step(s, explicit)
        if profile:
            L.klt_dev_profile_end(dev)
            prof = L.profile(dev)
        else:
            L.klt_dev_timer_stop(dev, C.byref(ms))
        L.KLTB200ResidentEnd(tc, fl)
        src = np.bincount(L.prediction(tc, N)[2], minlength=3).tolist() if mode or explicit else None
        if profile:
            return prof
        return ms.value * 1e3 / k, src

    times = {m[0]: [] for m in MODES}
    sources = {}
    for _ in range(rounds):
        for name, mode, explicit in MODES:
            us, src = leg(mode, explicit, steps)
            times[name].append(round(us, 3))
            sources[name] = src
    kern = {}
    for name, mode, explicit in MODES:
        prof = leg(mode, explicit, steps, profile=True)
        tr = {k: v for k, v in prof.items() if k.startswith("track")}
        kern[name] = {k: {"launches": v[0], "us_per_launch": round(v[1] * 1e3 / v[0], 3)} for k, v in tr.items()}
    L.KLTFreeFeatureList(fl)
    L.KLTFreeTrackingContext(tc)
    del fd
    med = {k: statistics.median(v) for k, v in times.items()}
    return {"workload": "3840x2160, 4096 features, 4 levels (subsampling 2), 7x7; resident pipeline "
                        "(KLTB200ResidentStep) over 20 distinct HBM-resident frames (166 MB) ping-pong; "
                        "%d steps per round after 20 warm-up steps, each round from the same selection" % steps,
            "step_us": times, "step_us_median": med,
            "step_overhead_us": {k: round(med[k] - med["off"], 3) for k in med},
            "tracker_kernel": kern,
            "last_step_sources_none_velocity_explicit": sources}


def run_pan(L, capi, torch):
    from tests.predict_oracle import pan_frames
    frames, motion = pan_frames(accel=3, frames=17)
    n = 300
    out = {"workload": "640x480 accelerating pan, 3 px/frame^2 up to 48 px/frame, 16 frame pairs, %d "
                       "features, tc defaults (2 levels, subsampling 4, 7x7), fma mode, KLTTrackFeatures per "
                       "call, no replacement; error = distance from the exact pan motion" % n}
    for name, mode in (("off", 0), ("velocity", 1)):
        tc = L.KLTCreateTrackingContext()
        tc.contents.sequentialMode = 1
        L.KLTB200SetDevice(tc, torch.cuda.current_device())
        L.KLTB200SetPrediction(tc, mode)
        fl = L.KLTCreateFeatureList(n)
        L.select(tc, frames[0], fl)
        tracked, errs, per_frame = 0, [], []
        for k in range(1, len(frames)):
            x0, y0, v0 = capi.featurelist_to_arrays(fl)
            L.track(tc, frames[k - 1], frames[k], fl)
            x, y, v = capi.featurelist_to_arrays(fl)
            ok = (v0 >= 0) & (v == 0)
            tracked += int(ok.sum())
            per_frame.append(int(ok.sum()))
            errs.extend(np.hypot(x[ok] - (x0[ok] + motion[k]), y[ok] - y0[ok]).tolist())
        e = np.array(errs) if errs else np.zeros(1)
        out[name] = {"tracked_results": tracked, "per_frame": per_frame,
                     "error_px_median": round(float(np.median(e)), 4), "error_px_p99": round(float(np.percentile(e, 99)), 4),
                     "error_px_max": round(float(e.max()), 4), "over_1px": int((e > 1.0).sum())}
        L.KLTFreeFeatureList(fl)
        L.KLTFreeTrackingContext(tc)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    rt = importlib.import_module(PKG + ".runtime")
    synth = importlib.import_module(PKG + ".synth")
    capi = importlib.import_module(PKG).capi
    L = rt.load()
    L.require_gpu()
    L.KLTSetVerbosity(0)
    res = {"card": card(), "rounds": args.rounds,
           "4k": run_4k(L, capi, synth, torch, args.rounds, args.steps),
           "640x480_pan": run_pan(L, capi, torch)}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
