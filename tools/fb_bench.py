"""Cost of the forward-backward check (KLTB200SetForwardBackward): check off vs on at 0.5 px,
alternated in one process, on the workloads of bench.py.

  * 4K: 3840x2160, 4096 features, 4 levels (subsampling 2), 7x7 -- the resident pipeline of bench.py's
    `value` leg over 20 distinct HBM-resident frames (166 MB, larger than the 126 MB L2), device
    events around the steps; every round restarts from the same selection.
  * the tracker kernel alone, from the klt_dev_profile_* event brackets (a separate profiled run).
  * 640x480, 1000 features: KLTTrackFeatures per call and KLTTrackFeaturesSequence, pinned host
    frames, wall clock.
  * the fraction of the features the check examines that it rejects, per step, at 0.5 px.

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

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PKG = "klt-feature-tracker-acceleration-gpus_b200"
FB = 0.5


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                     # (the measurement itself does not depend on it)
        return {"error": str(e)}


def rejected_fraction(L, tc, n, val):
    xb, yb, err, bv = L.forward_backward(tc, n)
    checked = bv != 1
    return int((val[checked] == -6).sum()), int(checked.sum())


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

    def leg(fb, k, profile=False):
        L.KLTStopSequentialMode(tc)
        tc.contents.sequentialMode = 1
        capi.arrays_to_featurelist(fl, *sel)
        L.KLTB200SetForwardBackward(tc, fb)
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
        rej = rejected_fraction(L, tc, N, capi.featurelist_to_arrays(fl)[2]) if fb > 0 else None
        if profile:
            return prof
        return ms.value * 1e3 / k, rej

    times = {"off": [], "on": []}
    rej = None
    for _ in range(rounds):
        for name, fb in (("off", 0.0), ("on", FB)):
            us, r = leg(fb, steps)
            times[name].append(round(us, 3))
            rej = r if r else rej
    kern = {}
    for name, fb in (("off", 0.0), ("on", FB)):
        prof = leg(fb, steps, profile=True)
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
            "step_overhead_pct": round(100.0 * (med["on"] / med["off"] - 1.0), 2),
            "tracker_kernel": kern,
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
            for name, fb in (("off", 0.0), ("on", FB)):
                tc = L.KLTCreateTrackingContext()
                tc.contents.sequentialMode = 1
                L.KLTB200SetDevice(tc, torch.cuda.current_device())
                L.KLTB200SetForwardBackward(tc, fb)
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
                if fb > 0 and api == "per_call":
                    tab = capi.featuretable_to_array(ft)
                    # rejections per step over the timed frames: val -6 first appears in that frame's column
                    for k in range(10, NFR):
                        prev, cur = tab["val"][:, k - 1], tab["val"][:, k]
                        rej[0] += int(((prev == 0) & (cur == -6)).sum())
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
    res = {"card": card(), "max_error_px": FB, "rounds": args.rounds,
           "4k": run_4k(L, capi, synth, torch, args.rounds, args.steps),
           "640x480": run_small(L, capi, synth, torch, args.rounds)}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
