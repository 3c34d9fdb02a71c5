"""Cost and effect of the global motion check (KLTB200SetMotionCheck): check off vs on at 1 px and
1024 hypotheses, alternated in one process, on the workloads of bench.py.

  * 4K: 3840x2160, 4096 features, 4 levels (subsampling 2), 7x7 -- the resident pipeline of bench.py's
    `value` leg over 20 distinct HBM-resident frames (166 MB, larger than the 126 MB L2), device
    events around the steps; every round restarts from the same selection.
  * the tracker and the check's three kernels, from the klt_dev_profile_* event brackets (a separate
    profiled run).
  * 640x480, 1000 features: KLTTrackFeatures per call and KLTTrackFeaturesSequence, pinned host
    frames, wall clock.
    A profiled per-call pass gives the D2H copy the per-call API pays with the check on (the tracker
    writes the device arrays instead of posting its results into pinned host memory).
  * the effect scenario of tests/motion_oracle.py (640x480, 300 features, a moving rectangle against a
    homography): tracked results more than 1 px from the true motion, and rectangle features kept.
  * with --parent DIR (a checkout of the parent commit, built): `bench.py --only-4k` of this tree and of
    DIR, alternated, with the check off; ms per step and whether the features after the timed loop are
    identical.

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
MAX_ERROR = 1.0
HYPS = 1024


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                     # (the measurement itself does not depend on it)
        return {"error": str(e)}


def rejected(L, tc, val):
    """(features the last call's check dropped, features that entered it)"""
    return int((val == -7).sum()), int(L.motion_models(tc, 1)["tracked"][0])


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

    def leg(max_error, k, profile=False):
        L.KLTStopSequentialMode(tc)
        tc.contents.sequentialMode = 1
        capi.arrays_to_featurelist(fl, *sel)
        L.KLTB200SetMotionCheck(tc, max_error, HYPS)
        L.KLTB200ResidentBegin(tc, ptr(0), 1, W, W, H, fl)
        for s in range(1, 21):
            L.KLTB200ResidentStep(tc, ptr(s), 1, W, W, H)
        L.klt_dev_sync(dev)
        ms = C.c_float(0)
        if profile:
            L.klt_dev_profile_begin(dev)
        else:
            L.klt_dev_timer_start(dev)
        for s in range(21, 21 + k):
            L.KLTB200ResidentStep(tc, ptr(s), 1, W, W, H)
        if profile:
            L.klt_dev_profile_end(dev)
            prof = L.profile(dev)
        else:
            L.klt_dev_timer_stop(dev, C.byref(ms))
        L.KLTB200ResidentEnd(tc, fl)
        rej = rejected(L, tc, capi.featurelist_to_arrays(fl)[2]) if max_error > 0 else None
        if profile:
            return prof
        return ms.value * 1e3 / k, rej

    times = {"off": [], "on": []}
    rej = None
    for _ in range(rounds):
        for name, e in (("off", 0.0), ("on", MAX_ERROR)):
            us, r = leg(e, steps)
            times[name].append(round(us, 3))
            rej = r if r else rej
    kern = {}
    for name, e in (("off", 0.0), ("on", MAX_ERROR)):
        prof = leg(e, steps, profile=True)
        tr = {k: v for k, v in prof.items() if k.startswith("track") or k.startswith("motion")}
        kern[name] = {k: {"launches": v[0], "us_per_launch": round(v[1] * 1e3 / v[0], 3)} for k, v in tr.items()}
    L.KLTFreeFeatureList(fl)
    L.KLTFreeTrackingContext(tc)
    del fd
    med = {k: statistics.median(v) for k, v in times.items()}
    return {"workload": "3840x2160, 4096 features, 4 levels (subsampling 2), 7x7; resident pipeline "
                        "(KLTB200ResidentStep) over 20 distinct HBM-resident frames (166 MB) ping-pong; "
                        "%d steps per round after 20 warm-up steps, each round from the same selection" % steps,
            "step_us": times, "step_us_median": med,
            "step_overhead_pct": round(100.0 * (med["on"] / med["off"] - 1.0), 2),
            "kernels": kern,
            "last_step_rejected_of_checked": rej}


def run_small(L, capi, synth, torch, rounds):
    W, H, NFR, N = 640, 480, 241, 1000
    frames = torch.empty((NFR, H, W), dtype=torch.uint8, pin_memory=True)
    fh = frames.numpy()
    for t in range(NFR):
        synth.frame(W, H, seed=2024, t=float(t), velocity=(1.7, -1.1), rot_deg=0.2, scale=1.001, out=fh[t])
    ptr = lambda i: C.c_void_p(frames.data_ptr() + i * W * H)
    res = {"per_call": {"off": [], "on": []}, "sequence": {"off": [], "on": []}}
    rej = [0, 0]
    for _ in range(rounds):
        for api in ("per_call", "sequence"):
            for name, e in (("off", 0.0), ("on", MAX_ERROR)):
                tc = L.KLTCreateTrackingContext()
                tc.contents.sequentialMode = 1
                L.KLTB200SetDevice(tc, torch.cuda.current_device())
                L.KLTB200SetMotionCheck(tc, e, HYPS)
                fl = L.KLTCreateFeatureList(N)
                ft = L.KLTCreateFeatureTable(NFR, N)
                L.KLTSelectGoodFeatures(tc, ptr(0), W, H, fl)
                for k in range(1, 9):
                    L.KLTTrackFeatures(tc, ptr(k - 1), ptr(k), W, H, fl)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                if api == "per_call":
                    for k in range(9, NFR):
                        L.KLTTrackFeatures(tc, ptr(k - 1), ptr(k), W, H, fl)
                        L.KLTStoreFeatureList(fl, ft, k)
                else:
                    seq = (C.c_void_p * (NFR - 8))(*[ptr(k).value for k in range(8, NFR)])
                    L.KLTTrackFeaturesSequence(tc, seq, NFR - 8, W, H, fl, ft, 8, 0)
                secs = time.perf_counter() - t0
                res[api][name].append(round(secs / (NFR - 9) * 1e6, 2))
                if e > 0 and api == "per_call":
                    tab = capi.featuretable_to_array(ft)
                    # rejections per step over the timed frames: val -7 first appears in that frame's column
                    for k in range(10, NFR):
                        prev, cur = tab["val"][:, k - 1], tab["val"][:, k]
                        rej[0] += int(((prev == 0) & (cur == -7)).sum())
                        rej[1] += int((prev == 0).sum())
                L.KLTFreeFeatureTable(ft)
                L.KLTFreeFeatureList(fl)
                L.KLTFreeTrackingContext(tc)
    out = {"workload": "synthetic 640x480, 240 frames (translation + 0.2 deg/frame rotation + 0.1 %% zoom), %d "
                       "features, tc defaults (2 levels, subsampling 4, 7x7), pinned host frames, no replacement; "
                       "us per frame, wall clock" % N}
    for api, v in res.items():
        med = {k: statistics.median(x) for k, x in v.items()}
        out[api] = {"us_per_frame": v, "median": med, "overhead_pct": round(100.0 * (med["on"] / med["off"] - 1.0), 2)}
    out["rejected_per_step"] = {"rejected": rej[0], "entering_tracked": rej[1],
                                "fraction": round(rej[0] / max(rej[1], 1), 5)}
    # per call, from the profile brackets: the feature copies and the check's kernels
    prof = {}
    for name, e in (("off", 0.0), ("on", MAX_ERROR)):
        tc = L.KLTCreateTrackingContext()
        tc.contents.sequentialMode = 1
        L.KLTB200SetDevice(tc, torch.cuda.current_device())
        L.KLTB200SetMotionCheck(tc, e, HYPS)
        dev = L.KLTB200Device(tc)
        fl = L.KLTCreateFeatureList(N)
        L.KLTSelectGoodFeatures(tc, ptr(0), W, H, fl)
        for k in range(1, 9):
            L.KLTTrackFeatures(tc, ptr(k - 1), ptr(k), W, H, fl)
        L.klt_dev_profile_begin(dev)
        for k in range(9, 109):
            L.KLTTrackFeatures(tc, ptr(k - 1), ptr(k), W, H, fl)
        L.klt_dev_profile_end(dev)
        prof[name] = {k: round(v[1] * 1e3 / 100, 3) for k, v in L.profile(dev).items()
                      if k.startswith("copy") or k.startswith("motion") or k.startswith("track")}
        L.KLTFreeFeatureList(fl)
        L.KLTFreeTrackingContext(tc)
    out["per_call_profile_us_per_call"] = prof
    return out


def run_parent(parent, rounds, steps):
    """bench.py --only-4k of this tree and of `parent`, alternated, check off"""
    import tempfile
    res = {"this": [], "parent": []}
    dumps = {}
    for r in range(rounds):
        for name, root in (("this", ROOT), ("parent", os.path.abspath(parent))):
            with tempfile.TemporaryDirectory() as tmp:
                cmd = [sys.executable, "bench.py", "--gpus", "1", "--only-4k", "--steps", str(steps), "--warmup", "50"]
                if r == 0:
                    cmd += ["--dump-outputs", tmp]
                env = dict(os.environ)
                env.pop("KLT_B200_LIB", None)
                env.pop("KLT_B200_MOTION_MAX_ERROR", None)
                q = subprocess.run(cmd, cwd=root, capture_output=True, text=True, env=env, timeout=900)
                if q.returncode != 0:
                    raise RuntimeError("bench.py in %s: %s" % (root, q.stderr[-2000:]))
                res[name].append(json.loads(q.stdout.strip().splitlines()[-1])["ms_per_step"] * 1e3)
                if r == 0:
                    dumps[name] = b"".join(np.load(os.path.join(tmp, k + ".npy")).tobytes() for k in ("x", "y", "val"))
    return {"workload": "bench.py --gpus 1 --only-4k --steps %d --warmup 50, alternated, check off" % steps,
            "us_per_step": res, "median": {k: statistics.median(v) for k, v in res.items()},
            "features_identical": dumps["this"] == dumps["parent"]}


def run_effect(L, capi):
    from tests import motion_oracle as mo
    from oracle import oracle_py
    o = oracle_py.Oracle()
    a, b = mo.scene()
    out = {"workload": "tests/motion_oracle.py scene(): 640x480, 300 features, tc defaults; background warped "
                       "by a 0.8 deg / 1.01 zoom / (3, -2) px homography, a 200x160 rectangle moving by (6, 4) px"}
    for name, e in (("off", 0.0), ("on", MAX_ERROR)):
        tc = L.KLTCreateTrackingContext()
        L.KLTB200SetMotionCheck(tc, e, HYPS)
        p = o.default_params()
        x0, y0, v0 = o.select(a, p, 300)
        fl = L.KLTCreateFeatureList(300)
        capi.arrays_to_featurelist(fl, x0, y0, v0)
        L.track(tc, a, b, fl)
        x1, y1, v1 = capi.featurelist_to_arrays(fl)
        truth = mo.project(mo.scene_homography(), np.c_[x0, y0])
        ok = v1 == 0
        off = np.hypot(x1 - truth[:, 0], y1 - truth[:, 1]) > 1.0
        rect, _ = mo.scene_groups(x0, y0, x1, y1, ok, p.window_width // 2)
        out[name] = {"tracked": int(ok.sum()), "tracked_more_than_1px_off": int((ok & off).sum()),
                     "rectangle_features_kept": int(rect.sum())}
        L.KLTFreeFeatureList(fl)
        L.KLTFreeTrackingContext(tc)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--out", default=None)
    ap.add_argument("--parent", default=None, help="a built checkout of the parent commit: compare bench.py --only-4k")
    args = ap.parse_args()
    import torch
    rt = importlib.import_module(PKG + ".runtime")
    synth = importlib.import_module(PKG + ".synth")
    capi = importlib.import_module(PKG).capi
    L = rt.load()
    L.require_gpu()
    L.KLTSetVerbosity(0)
    res = {"card": card(), "max_error_px": MAX_ERROR, "hypotheses": HYPS, "rounds": args.rounds,
           "4k": run_4k(L, capi, synth, torch, args.rounds, args.steps),
           "640x480": run_small(L, capi, synth, torch, args.rounds),
           "effect": run_effect(L, capi)}
    if args.parent:
        res["bench_vs_parent"] = run_parent(args.parent, args.rounds, args.steps)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
