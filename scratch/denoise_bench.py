"""Denoised resolve on the GPU: device time of the filter + pack per number of passes (CUDA events of the library,
stats().last_resolve_ms) at 1280x720 and 1920x1080, the shared-memory staging cut-over (RTB200_DENOISE_STAGE, one child
process per setting), interactive frame latency (render_spp(1) + denoise_rgba8 into an rt_host_alloc surface next to
rt_render_frame alone, same process) and the tonemapped PSNR of the default and swept tolerances at 4 spp against 4096 spp
of another seed. Prints one JSON line (with the card's name and power limit).

    python scratch/denoise_bench.py [--calls 200] [--out profiles/x.json]
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
sys.path.insert(0, os.path.join(ROOT, "tests"))
import rtb200  # noqa: E402
import denoise_reference as ref  # noqa: E402


def scene(name):
    return np.load(os.path.join(ROOT, "tests", "golden", "bundled_scenes.npz"))[name]


def setup(t, name, w, h, seed=(7, 9)):
    t.set_scene(scene(name))
    t.set_camera(rtb200.default_camera())
    t.set_params(rtb200.default_params(width=w, height=h, mode=rtb200.RT_MODE_PATH, max_bounces=8, seed_lo=seed[0], seed_hi=seed[1]))
    t.reset_accumulation()


def device_times(t, w, h, calls, max_passes=5):
    """median / mean device ms of denoise_rgba8 (filter + pack) into a page-locked surface, for passes 0..max_passes."""
    setup(t, "Scene1", w, h)
    t.render_spp(1)
    surf, owner = rtb200.host_surface(w, h)
    out = {}
    for passes in range(0, max_passes + 1):
        p = rtb200.default_denoise_params(passes=passes)
        for _ in range(20):
            t.denoise_rgba8(p, out=surf)
        ms = []
        for _ in range(calls):
            t.denoise_rgba8(p, out=surf)
            ms.append(t.stats().last_resolve_ms)
        out[passes] = {"median_ms": float(np.median(ms)), "mean_ms": float(np.mean(ms))}
    del owner
    split = [out[k]["median_ms"] - out[k - 1]["median_ms"] for k in range(2, max_passes + 1)]
    return {"passes": out, "added_per_pass_ms": split}


def frame_latency(t, w, h, frames):
    setup(t, "Scene1", w, h)
    surf, owner = rtb200.host_surface(w, h)
    p = rtb200.default_denoise_params()
    res = {}
    for rep in range(2):                                    # alternate the two loops; keep the second round
        for kind in ("render_frame", "render_spp+denoise5"):
            t.reset_accumulation()
            ms = []
            for f in range(frames + 20):
                t0 = time.perf_counter()
                if kind == "render_frame":
                    t.render_frame(1, out=surf)
                else:
                    t.render_spp(1)
                    t.denoise_rgba8(p, out=surf)
                d = (time.perf_counter() - t0) * 1e3
                if f >= 20:
                    ms.append(d)
            res[kind] = {"p50_ms": float(np.percentile(ms, 50)), "p99_ms": float(np.percentile(ms, 99))}
    del owner
    return res


def quality(t, sweep):
    w, h = 160, 120
    rows = {}
    for name in ("Scene1", "Scene2", "Scene_indirect"):
        setup(t, name, w, h, seed=(0x5EED, 0xF00D))
        t.render_spp(4096)
        gt = t.read_denoised(rtb200.default_denoise_params(passes=0))[..., :3]
        setup(t, name, w, h)
        t.render_spp(4)
        raw = t.read_denoised(rtb200.default_denoise_params(passes=0))[..., :3]
        r = {"raw_4spp_db": ref.psnr(raw, gt)}
        for sc in sweep:
            for sz in sweep:
                d = t.read_denoised(rtb200.default_denoise_params(sigma_color=sc, sigma_depth=sz))[..., :3]
                r["sc%g_sz%g_db" % (sc, sz)] = ref.psnr(d, gt)
        t.render_spp(4092)
        raw_hi = t.read_denoised(rtb200.default_denoise_params(passes=0))[..., :3]
        den_hi = t.read_denoised()[..., :3]
        rmse = lambda x: float(np.sqrt(np.mean((ref.tonemap(x) - ref.tonemap(gt)) ** 2)))
        r["rmse_4096_raw"] = rmse(raw_hi); r["rmse_4096_denoised"] = rmse(den_hi)
        rows[name] = r
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--frames", type=int, default=500)
    ap.add_argument("--child", action="store_true", help="device times only (one staging setting, from the environment)")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    t = rtb200.PathTracer(0)
    if a.child:
        print(json.dumps({"stage": os.environ.get("RTB200_DENOISE_STAGE", "default"), "1080p": device_times(t, 1920, 1080, a.calls)}))
        return
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": smi[0] if smi else "unknown", "calls": a.calls}
    res["device_ms"] = {"720p": device_times(t, 1280, 720, a.calls), "1080p": device_times(t, 1920, 1080, a.calls)}
    res["frame_latency_720p"] = frame_latency(t, 1280, 720, a.frames)
    res["frame_latency_1080p"] = frame_latency(t, 1920, 1080, a.frames)
    res["quality_160x120_depth8"] = quality(t, (0.5, 1.0, 2.0, 4.0))
    t.close()
    ab = {}
    for stage in ("0", "1", "2", "4"):
        env = dict(os.environ, RTB200_DENOISE_STAGE=stage)
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "--calls", str(a.calls)], capture_output=True, text=True, env=env)
        ab[stage] = json.loads(r.stdout.strip().splitlines()[-1])["1080p"] if r.returncode == 0 else r.stderr[-400:]
    res["stage_ab_1080p"] = ab
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
