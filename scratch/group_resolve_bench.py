"""The multi-GPU group's resolves on the GPU, for every device count from 1 to the devices the run has (1, 2, 4, 8): host time of
the synchronising call (median of --calls, after 20 warm-up calls) of rt_group_resolve_rgba8, rt_group_denoise_rgba8 at 0 and 5
passes and rt_group_temporal_rgba8 with and without 5 filter passes, at 1920x1080 into an rt_host_alloc surface; the temporal
calls at a fixed pose (the prior is kept), and as device time of filter + pack (stats().last_resolve_ms, which leaves out the reduce)
with the pose alternating so that every call reprojects. Then the frame latency p50 / p99 of a turning camera (0.25 degrees per
frame; each frame restarts the accumulation, renders one sample per device and presents). Scene1, depth 8. Prints one JSON line
with the card's name and power limit, and writes it to --out.

    python scratch/group_resolve_bench.py [--calls 200] [--frames 200] [--out profiles/x.json]
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "software-raytracer_b200", "python"))
import rtb200  # noqa: E402

W, H = 1920, 1080


def setup(g):
    g.set_scene(np.load(os.path.join(ROOT, "tests", "golden", "bundled_scenes.npz"))["Scene1"])
    cam = rtb200.default_camera()
    g.set_camera(cam)
    g.set_params(rtb200.default_params(width=W, height=H, mode=rtb200.RT_MODE_PATH, max_bounces=8, seed_lo=7, seed_hi=9))
    g.reset_accumulation()
    return cam


def turn(cam, deg):
    rtb200.rotate_camera(cam, deg * math.pi / 180.0, [cam.up[0], cam.up[1], cam.up[2]])


def call_times(g, surf, calls):
    n = g.size()
    setup(g)
    g.render_spp(n)
    dn0, dn5 = rtb200.default_denoise_params(passes=0), rtb200.default_denoise_params(passes=5)
    kinds = {
        "resolve": lambda: g.resolve_rgba8(out=surf),
        "denoise0": lambda: g.denoise_rgba8(dn0, out=surf),
        "denoise5": lambda: g.denoise_rgba8(dn5, out=surf),
        "temporal": lambda: g.temporal_rgba8(out=surf),
        "temporal+denoise5": lambda: g.temporal_rgba8(dn=dn5, out=surf),
    }
    res = {}
    for name, fn in kinds.items():
        for _ in range(20):
            fn()
        ms = []
        for _ in range(calls):
            t0 = time.perf_counter()
            fn()
            ms.append((time.perf_counter() - t0) * 1e3)
        res[name] = {"median_ms": float(np.median(ms)), "p99_ms": float(np.percentile(ms, 99))}
    # device time of filter + pack with a reprojection on every call (the moved pose's primary-hit trace precedes the timed window)
    cams = [rtb200.default_camera(), rtb200.default_camera()]
    turn(cams[1], 0.25)
    for name, dn in (("temporal_reproject", None), ("temporal_reproject+denoise5", dn5)):
        ms = []
        for k in range(calls + 20):
            g.set_camera(cams[k & 1])
            g.temporal_rgba8(dn=dn, out=surf)
            if k >= 20:
                ms.append(g.stats().last_resolve_ms)
        res[name] = {"device_median_ms": float(np.median(ms))}
    return res


def frame_latency(g, surf, frames):
    n = g.size()
    dn5 = rtb200.default_denoise_params(passes=5)
    present = {
        "resolve": lambda: g.resolve_rgba8(out=surf),
        "denoise5": lambda: g.denoise_rgba8(dn5, out=surf),
        "temporal": lambda: g.temporal_rgba8(out=surf),
        "temporal+denoise5": lambda: g.temporal_rgba8(dn=dn5, out=surf),
    }
    res = {}
    for rep in range(2):                                    # alternate the loops; keep the second round
        for name, fn in present.items():
            cam = setup(g)
            ms = []
            for f in range(frames + 20):
                t0 = time.perf_counter()
                turn(cam, 0.25); g.set_camera(cam); g.reset_accumulation(); g.render_spp(n)
                fn()
                d = (time.perf_counter() - t0) * 1e3
                if f >= 20:
                    ms.append(d)
            res[name] = {"p50_ms": float(np.percentile(ms, 50)), "p99_ms": float(np.percentile(ms, 99))}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--frames", type=int, default=200)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    import torch
    n_dev = torch.cuda.device_count()
    res = {"gpu": smi[0] if smi else "unknown", "devices": n_dev, "size": [W, H], "calls": a.calls, "frames": a.frames,
           "gather_bytes_per_call": W * H * 16, "by_device_count": {}}
    surf, owner = rtb200.host_surface(W, H)
    for k in (1, 2, 4, 8):
        if k > n_dev:
            break
        g = rtb200.TracerGroup(list(range(k)))
        try:
            res["by_device_count"][str(k)] = {"call_ms": call_times(g, surf, a.calls), "frame_latency_ms": frame_latency(g, surf, a.frames)}
        finally:
            g.close()
    del owner
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
