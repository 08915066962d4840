"""Temporal resolve on the GPU: device time of the call (reprojection + blend + pack, with and without 5 filter passes; CUDA events
of the library, stats().last_resolve_ms) into an rt_host_alloc surface at 1280x720 and 1920x1080 next to the plain and denoised
resolves, per-frame latency of a turning camera (reset + render_spp(1) + temporal_rgba8, which includes the primary-hit cache
trace every moved frame costs) next to reset + render_frame, and the tonemapped PSNR of the last of 16 frames turning 0.25 degrees
each (160x120, depth 8, 1 spp per frame) against 4096 spp of another seed, with the cap / tau_depth sweep that chose the defaults.
Prints one JSON line (with the card's name and power limit).

    python scratch/temporal_bench.py [--calls 200] [--frames 300] [--out profiles/x.json]
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
sys.path.insert(0, os.path.join(ROOT, "tests"))
import rtb200  # noqa: E402
from denoise_reference import psnr  # noqa: E402


def scene(name):
    return np.load(os.path.join(ROOT, "tests", "golden", "bundled_scenes.npz"))[name]


def setup(t, name, w, h, seed=(7, 9)):
    t.set_scene(scene(name))
    cam = rtb200.default_camera()
    t.set_camera(cam)
    t.set_params(rtb200.default_params(width=w, height=h, mode=rtb200.RT_MODE_PATH, max_bounces=8, seed_lo=seed[0], seed_hi=seed[1]))
    t.reset_accumulation()
    return cam


def turn(cam, deg):
    rtb200.rotate_camera(cam, deg * math.pi / 180.0, [cam.up[0], cam.up[1], cam.up[2]])


def device_times(t, w, h, calls):
    """median / mean device ms per call kind into a page-locked surface; the temporal calls alternate two poses, so every call
    reprojects (the cache trace of the moved pose is enqueued before the timed window)."""
    cam = setup(t, "Scene1", w, h)
    t.render_spp(1)
    surf, owner = rtb200.host_surface(w, h)
    cams = [rtb200.default_camera(), rtb200.default_camera()]
    turn(cams[1], 0.25)
    dn5 = rtb200.default_denoise_params(passes=5)
    kinds = {
        "resolve": lambda k: t.resolve_rgba8(out=surf),
        "denoise5": lambda k: t.denoise_rgba8(dn5, out=surf),
        "temporal": lambda k: (t.set_camera(cams[k & 1]), t.temporal_rgba8(out=surf)),
        "temporal+denoise5": lambda k: (t.set_camera(cams[k & 1]), t.temporal_rgba8(dn=dn5, out=surf)),
        "temporal_same_pose": lambda k: t.temporal_rgba8(out=surf),
    }
    out = {}
    for name, fn in kinds.items():
        t.set_camera(cam)
        for k in range(20):
            fn(k)
        ms = []
        for k in range(calls):
            fn(k)
            ms.append(t.stats().last_resolve_ms)
        out[name] = {"median_ms": float(np.median(ms)), "mean_ms": float(np.mean(ms))}
    del owner
    return out


def frame_latency(t, w, h, frames):
    """host wall time per frame of a camera turning 0.25 degrees per frame (every frame restarts the accumulation)."""
    surf, owner = rtb200.host_surface(w, h)
    dn5 = rtb200.default_denoise_params(passes=5)
    res = {}
    for rep in range(2):                                    # alternate the loops; keep the second round
        for kind in ("render_frame", "render_spp+temporal", "render_spp+temporal+denoise5"):
            cam = setup(t, "Scene1", w, h)
            ms = []
            for f in range(frames + 20):
                t0 = time.perf_counter()
                turn(cam, 0.25); t.set_camera(cam); t.reset_accumulation()
                if kind == "render_frame":
                    t.render_frame(1, out=surf)
                else:
                    t.render_spp(1)
                    t.temporal_rgba8(dn=dn5 if "denoise" in kind else None, out=surf)
                d = (time.perf_counter() - t0) * 1e3
                if f >= 20:
                    ms.append(d)
            res[kind] = {"p50_ms": float(np.percentile(ms, 50)), "p99_ms": float(np.percentile(ms, 99))}
    del owner
    return res


def run_turning(t, name, w, h, frames, deg, tp, dn):
    cam = setup(t, name, w, h)
    for f in range(frames):
        if f:
            turn(cam, deg); t.set_camera(cam)
        t.reset_accumulation(); t.render_spp(1)
        tem = t.read_temporal(tp)[..., :3]
    raw = t.read_denoised(rtb200.default_denoise_params(passes=0))[..., :3]
    return raw, tem, t.read_denoised(dn)[..., :3], t.read_temporal(tp, dn)[..., :3], cam


def quality(t, caps, taus):
    w, h = 160, 120
    dn = rtb200.default_denoise_params()
    rows = {}
    for name in ("Scene1", "Scene2", "Scene_indirect", "Scene1_reflection"):
        raw, tem, den, both, cam = run_turning(t, name, w, h, 16, 0.25, rtb200.default_temporal_params(), dn)
        setup(t, name, w, h, seed=(0x5EED, 0xF00D))
        t.set_camera(cam)
        t.render_spp(4096)
        gt = t.read_denoised(rtb200.default_denoise_params(passes=0))[..., :3]
        r = {"raw_1spp_db": psnr(raw, gt), "filter_db": psnr(den, gt), "temporal_db": psnr(tem, gt), "temporal+filter_db": psnr(both, gt)}
        for cap in caps:
            for tz in taus:
                _, tem, _, both, _ = run_turning(t, name, w, h, 16, 0.25, rtb200.default_temporal_params(max_history=cap, tau_depth=tz), dn)
                r["cap%d_tz%g" % (cap, tz)] = [psnr(tem, gt), psnr(both, gt)]
        rows[name] = r
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--frames", type=int, default=300)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    t = rtb200.PathTracer(0)
    res = {"gpu": smi[0] if smi else "unknown", "calls": a.calls, "frames": a.frames}
    res["device_ms"] = {"720p": device_times(t, 1280, 720, a.calls), "1080p": device_times(t, 1920, 1080, a.calls)}
    res["frame_latency_720p"] = frame_latency(t, 1280, 720, a.frames)
    res["frame_latency_1080p"] = frame_latency(t, 1920, 1080, a.frames)
    res["quality_160x120_depth8_16frames_0.25deg"] = quality(t, (8, 16, 32, 64), (0.005, 0.01, 0.02, 0.05))
    t.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
