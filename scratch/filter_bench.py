"""Pixel filter on the GPU: Scene1 1080p 1024 spp render time with the box filter against none (device time of the render call,
CUDA events of the library, stats().last_render_ms), the 1280x720 rt_render_frame latency p50 / p99 with and without a filter
(host clock around the synchronising call, page-locked surface), and the tonemapped edge error of a 64-spp filtered frame against a
4096-spp filtered render with another seed (Scene1, 320x180: RMS of the Reinhard-mapped difference over edge pixels, those whose
primary-hit object id differs from a neighbour's, and over all pixels). Prints one JSON line with the card's name and power limit.

    python scratch/filter_bench.py [--out profiles/x.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "software-raytracer_b200", "python"))
import rtb200  # noqa: E402

O = rtb200


def setup(t, w, h, seed=(7, 9), bounces=8):
    t.set_scene(np.load(os.path.join(ROOT, "tests", "golden", "bundled_scenes.npz"))["Scene1"])
    t.set_camera(rtb200.default_camera())
    t.set_params(rtb200.default_params(width=w, height=h, mode=O.RT_MODE_PATH, max_bounces=bounces, seed_lo=seed[0], seed_hi=seed[1]))
    t.reset_accumulation()


def render_ms(t, f, spp, reps=5):
    t.set_pixel_filter(f)
    out = []
    for _ in range(reps + 1):
        t.reset_accumulation()
        t.render_spp(spp)
        t.sync()
        out.append(t.stats().last_render_ms)
    return float(np.median(out[1:]))


def frame_ms(t, f, frames=300):
    t.set_pixel_filter(f)
    surf, owner = rtb200.host_surface(1280, 720)
    t.reset_accumulation()
    ms = []
    for i in range(frames + 20):
        a = time.perf_counter()
        t.render_frame(1, out=surf)
        if i >= 20:
            ms.append((time.perf_counter() - a) * 1e3)
    del owner
    ms.sort()
    return ms[len(ms) // 2], ms[int(len(ms) * 0.99)]


def tonemap(acc, n):
    m = acc[..., :3].astype(np.float64) / n
    return m / (1 + m)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    a = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": smi[0] if smi else "unknown"}
    t = rtb200.PathTracer(0)
    box = rtb200.default_pixel_filter(type=O.RT_FILTER_BOX, radius=0.5)
    tent = rtb200.default_pixel_filter(type=O.RT_FILTER_TENT, radius=1.0)

    setup(t, 1920, 1080)
    render_ms(t, None, 64, 1)                                         # builds, tunes
    res["c2_1080p_1024spp_none_ms"] = render_ms(t, None, 1024)
    res["c2_1080p_1024spp_box_ms"] = render_ms(t, box, 1024)
    res["c2_1080p_1024spp_tent_ms"] = render_ms(t, tent, 1024)
    res["c2_box_over_none"] = res["c2_1080p_1024spp_box_ms"] / res["c2_1080p_1024spp_none_ms"]

    setup(t, 1280, 720)
    for name, f in (("none", None), ("box", box), ("tent", tent)):
        p50, p99 = frame_ms(t, f)
        res["frame_720p_%s_p50_ms" % name], res["frame_720p_%s_p99_ms" % name] = p50, p99

    w, h = 320, 180
    for name, f in (("box", box), ("tent", tent)):
        setup(t, w, h, seed=(1, 2))
        t.set_pixel_filter(f)
        t.render_spp(4096)
        ref_img = tonemap(*t.read_accum())
        ids = t.read_aov()[0]
        setup(t, w, h, seed=(7, 9))
        t.set_pixel_filter(f)
        t.render_spp(64)
        img = tonemap(*t.read_accum())
        edge = np.zeros_like(ids, bool)
        edge[:, 1:] |= ids[:, 1:] != ids[:, :-1]; edge[:, :-1] |= ids[:, 1:] != ids[:, :-1]
        edge[1:] |= ids[1:] != ids[:-1]; edge[:-1] |= ids[1:] != ids[:-1]
        d = (img - ref_img) ** 2
        res["edge_rms_64spp_%s" % name] = float(np.sqrt(d[edge].mean()))
        res["all_rms_64spp_%s" % name] = float(np.sqrt(d.mean()))
        res["edge_pixels"] = int(edge.sum())
    t.set_pixel_filter(None)
    t.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
