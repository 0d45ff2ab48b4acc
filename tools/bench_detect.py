"""Detect-stage device time of ORB (Kp/DetectorStrategy=2) and GFTT/ORB (8) on a B200, with single-thread cv2 per frame as context.

For each frame size (128 frames of 640x480 and of 1280x720, BGR with u16 depth, device-resident inputs) and detector: warm-up calls, then
CUDA events on the engine stream around each of --reps calls of lcd_orb_detect_describe_dev (gray + mask, detection, blur, descriptors,
3-D points); the median and the spread are reported.  The GPU name and power limit are read in the same run.
usage: python tools/bench_detect.py [--frames 128] [--reps 20] [--out profiles/r03_detect_gftt.json]
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from oracle import feature2d_py as f2d  # noqa: E402
from rtabmap_b200 import Engine, synth  # noqa: E402
from rtabmap_b200.capi import LCD_DETECTOR_GFTT_ORB, LCD_DETECTOR_ORB  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clk = [s.strip() for s in q.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clk}


def frames(n, h, w):
    base = [synth.make_image(h, w, 100 + i, bgr=True) for i in range(8)]
    deps = [synth.make_depth(h, w, 200 + i) for i in range(8)]
    return np.stack([base[i % 8] for i in range(n)]), np.stack([deps[i % 8] for i in range(n)])


def time_device(eng, imgs, deps, op, reps, warmup):
    import torch

    n, h, w = imgs.shape[:3]
    cap = op.n_features + 256
    d_img = torch.from_numpy(imgs).cuda()
    d_dep = torch.from_numpy(deps.view(np.int16)).cuda()
    d_kp = torch.zeros(n * cap * 6, dtype=torch.float32, device="cuda")
    d_desc = torch.zeros(n * cap * 32, dtype=torch.uint8, device="cuda")
    d_xyz = torch.zeros(n * cap * 3, dtype=torch.float32, device="cuda")
    d_n = torch.zeros(n, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    stream = torch.cuda.ExternalStream(eng.stream)
    lib = eng._lib
    import ctypes as C

    def call():
        eng._check(lib.lcd_orb_detect_describe_dev(eng.handle, n, C.c_void_p(d_img.data_ptr()), w, h, 3, C.c_void_p(d_dep.data_ptr()), 1, C.byref(op), cap,
                                                   C.c_void_p(d_kp.data_ptr()), C.c_void_p(d_desc.data_ptr()), C.c_void_p(d_xyz.data_ptr()), None,
                                                   C.c_void_p(d_n.data_ptr()), C.c_void_p(eng.stream)))

    for _ in range(warmup):
        call()
    torch.cuda.synchronize()
    assert not eng.orb_overflow()
    ms = []
    with torch.cuda.stream(stream):
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            call()
            b.record(stream)
            b.synchronize()
            ms.append(a.elapsed_time(b))
    nk = d_n.cpu().numpy()
    # where the time goes: device time per kernel name over 3 calls, in a profiled pass of its own (after the timed one)
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            call()
        torch.cuda.synchronize()
    kernels = {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA and "lcd::" in ev.name:
            k = ev.name.split("lcd::")[1].split("(")[0]
            us = getattr(ev, "device_time_total", None)
            kernels[k] = kernels.get(k, 0.0) + (us if us is not None else ev.cuda_time_total) / 3e3
    return {"kernels_ms_per_call": {k: round(v, 4) for k, v in sorted(kernels.items(), key=lambda kv: -kv[1])},
            "median_ms": float(np.median(ms)), "min_ms": float(np.min(ms)), "max_ms": float(np.max(ms)), "reps": reps,
            "mean_keypoints_per_frame": float(nk.mean())}


def time_cv2(imgs, deps, detector, n=16):
    import cv2

    cv2.setNumThreads(1)
    p = f2d.OrbParams()
    orb = f2d.make_orb(p)
    gftt = cv2.GFTTDetector_create(p.n_features, 0.001, 7, 3)
    t = []
    for i in range(n):
        gray = cv2.cvtColor(imgs[i], cv2.COLOR_BGR2GRAY)
        mask = f2d.depth_mask(deps[i], p)
        t0 = time.perf_counter()
        kps = orb.detect(gray, mask) if detector == "orb" else gftt.detect(gray, mask)
        orb.compute(gray, kps)
        t.append(time.perf_counter() - t0)
    return {"median_ms_per_frame": 1e3 * float(np.median(t)), "frames": n, "threads": 1}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=128)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r03_detect_gftt.json"))
    args = ap.parse_args()
    res = {"info": gpu_info(), "what": "device time of lcd_orb_detect_describe_dev per batch (CUDA events on the engine stream)", "runs": []}
    for h, w in ((480, 640), (720, 1280)):
        imgs, deps = frames(args.frames, h, w)
        k4 = (525.0 * w / 640, 525.0 * w / 640, w / 2, h / 2)
        op = Engine.orb_params(k4)
        for name, strategy in (("orb", LCD_DETECTOR_ORB), ("gftt_orb", LCD_DETECTOR_GFTT_ORB)):
            eng = Engine()
            eng.set_detector(strategy, Engine.gftt_params() if strategy == LCD_DETECTOR_GFTT_ORB else None)
            r = {"detector": name, "size": f"{w}x{h}", "frames": args.frames}
            r["device"] = time_device(eng, imgs, deps, op, args.reps, args.warmup)
            r["cv2_single_thread"] = time_cv2(imgs, deps, "orb" if name == "orb" else "gftt")
            res["runs"].append(r)
            print(json.dumps(r), flush=True)
            eng.close()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps(res["info"]))


if __name__ == "__main__":
    main()
