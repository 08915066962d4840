#!/usr/bin/env python
"""bench.py - headline benchmark of the B200 path tracer (BASELINE.json metric:
Mpaths*bounces/s = path SEGMENTS per second, one segment = one closest-hit query + its shading).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config c1..c5] [--scaling weak|strong] [--dump-outputs DIR]

Headline workload (BASELINE.json configs[1], "c2"): bundled Scene1 (67 spheres), 1920x1080, 1024 spp, depth 8,
default camera. One step = one rt_render_spp(1024) over the whole frame (2.12 G paths).

N > 1 (one process per GPU under torchrun): weak scaling by default - every rank renders its own 1024 samples of the
full frame (global spp = 1024 N) - and the ONE exchange of the path, the sum of the float4 accumulation buffers before
the resolve, runs inside the timed step as rt_exchange_resolve: a fused reduce + resolve kernel that reads every rank's
buffer over NVLink peer mappings and orders the ranks with flags in device memory (no NCCL call, no host barrier in the
step; `--reduce nccl` is the plain all-reduce for comparison). The line also carries a `strong` object: the same 1024
global samples split over the N GPUs with rt_set_shard(rank, N) and one shared seed. Outside the timed region rank 0
checks that the fused surface equals the resolve of the sum of all ranks' buffers (`multi_gpu_check`).

`value`  : segments/s with the scene resident on the device (CUDA events around the kernels).
`e2e`    : the same metric through the C-ABI with HOST buffers each step: rt_set_scene (H2D) + rt_set_camera +
           rt_reset_accumulation + rt_render_spp + rt_resolve_rgba8 (D2H ARGB8).
`configs`: (N = 1, default config only) short legs of the other BASELINE.json configs - c1 640x480x64 spp, c3 10 000
           spheres at 3840x2160 through the BVH / wavefront pipeline, c4 1 M-triangle mesh at 1080p, c5 interactive 1 spp
           frames at 720p - each with its own roofline object, so that every config is observed by whoever runs this file.
`frame_1080p_1spp`: the metric's "ms/frame at 1080p", measured: p50 / p99 of one rt_render_frame(1) per frame into a host surface.
`cpu_baseline`: the reference's own renderArea loop on the box's host cores (24 frames of 1 spp; also as Mpaths/s, ms per 1-spp
           frame, and with glibc's locked rand() instead of MSVC's per-thread one); the c3 leg carries the same for ITS scene.
`--impl reference`: the reference's own CPU code (oracle/_ref, else the validated C port) on the host cores, same
           metric, bounded sample per step.
`--dump-outputs DIR`: after the timed steps, what the last timed step handed its caller, as DIR/<name>.npy in float32, so that
           two builds can be compared output for output (the inputs are seeded: the same arguments give the same inputs):
           `accum` (height x width x 4, rt_read_accum: the step's sample sums), or at N > 1 with the fused exchange and for c5
           `surface_argb` (height x width x 4, the resolved ARGB8 frame, one channel per byte). Past 60 MiB in all, a fixed seeded
           sample of pixels is kept, with their flat indices in `pixel_index` (float64).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "software-raytracer_b200", "python"))

METRIC = "Mpaths*bounces/s (path segments per second), bundled Scene1 @1920x1080"
UNIT = "Msegments/s"
W, H, SPP, DEPTH = 1920, 1080, 1024, 8
L2_NOTE = "GPU arm: flushed between timed steps (256 MiB write); CPU arm: not applicable"


def load_scene(name="Scene1"):
    return np.load(os.path.join(ROOT, "tests", "golden", "bundled_scenes.npz"))[name]


def workload_config(scene="Scene1", n_obj=67, w=W, h=H, depth=DEPTH):
    """The part of `config` both arms share word for word (the driver compares them)."""
    return {"workload": "%s (%d objects) %dx%d, depth %d, path mode" % (scene, n_obj, w, h, depth), "scene": scene, "width": w, "height": h,
            "depth": depth, "mode": "path", "l2": L2_NOTE}


DUMP_BYTES = 60 << 20                 # stays under 64 MB with the .npy headers


def argb_channels(argb):
    """packed ARGB8 surface (h x w uint32) -> h x w x 4 float32 (A, R, G, B)."""
    return np.stack([(argb >> s) & 255 for s in (24, 16, 8, 0)], -1).astype(np.float32)


def write_outputs(out_dir, arrays):
    """--dump-outputs: every h x w x c array as out_dir/<name>.npy (float32). Over DUMP_BYTES in all, the same seeded sample of
    pixels is taken from each array and their flat indices are written as pixel_index.npy."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.ascontiguousarray(v, np.float32) for k, v in arrays.items()}
    h, w = next(iter(arrays.values())).shape[:2]
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        keep = DUMP_BYTES // (total // (h * w) + 8)          # + 8: the pixel's index
        idx = np.sort(np.random.default_rng(0).choice(h * w, keep, replace=False))
        arrays = {k: v.reshape(h * w, -1)[idx] for k, v in arrays.items()}
        arrays["pixel_index"] = idx.astype(np.float64)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def flops_per_segment(objs):
    """SURVEY.md 8d: 23 per sphere test + 30 per cube test + 110 shading/scatter."""
    return 23 * int((objs["type"] == 1).sum()) + 30 * int((objs["type"] == 2).sum()) + 110


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def sample_once(self):
        """One blocking query (the short legs sample before and after their steps instead of during them: a leg of 3 x 22 ms lies
        entirely inside the start-up of the first concurrent nvidia-smi, whose device queries were seen to double the step time of
        the 40-launch wavefront pipeline - profiles/r3a_bench_n1.json c4: 44 ms; the same leg alone or sampled outside: 22 ms)."""
        try:
            out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                 capture_output=True, text=True, timeout=5).stdout.strip()
            if out:
                self.rows.append([c.strip() for c in out.split(",")])
        except Exception:
            pass

    def summary(self):
        self.stop_flag = True
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for i, n in enumerate(names):
                if len(r) > 4 + i and r[4 + i].lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


# ---- the reference's CPU implementation (the only place that executes oracle/) -----------------------------------
def write_scene_json(path, objs):
    """Reference-format scene file (Scene.hpp:27-104) with json.dump: the reference arm must not map librt_b200.so."""
    out = []
    for i, o in enumerate(objs):
        r = {"Type": "None"}
        if o["type"] == 1:
            r = {"Type": "Sphere", "Radius": float(o["radius"])}
        elif o["type"] == 2:
            r = {"Type": "Cube", "Size": [float(v) for v in o["half"]]}
        out.append({"Name": "object%d" % i, "Position": [float(v) for v in o["pos"]],
                    "Material": {"Color": [float(v) for v in o["base"]], "Emissive": [float(v) for v in o["emissive"]],
                                 "SpecularColor": [float(v) for v in o["spec_color"]], "Smoothness": float(o["smoothness"]),
                                 "SpecularAmount": float(o["spec_amount"]), "Metalness": float(o["spec_amount"])},
                    "Renderer": r})
    with open(path, "w") as f:
        json.dump({"SceneName": "bench", "SceneObjects": out}, f)


def cpu_reference_run(objs, frames, w=W, h=H, want_ref=True, cam=None, fov=55, label="Scene1"):
    """Time the reference's CPU implementation of the path on all host cores: `frames` 1-spp frames at w x h.
    Returns (segments/s, info). oracle/_ref (the reference's own code, 16 strip threads, per-thread MSVC rand) when its .so
    is present, else the bit-for-bit validated C port."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from oracle_py import Oracle, Reference, OrcCamera, REF_SO
    cores = os.cpu_count() or 1
    tmp_scene = "/tmp/_bench_scene_%d.json" % os.getpid()
    if want_ref and os.path.exists(REF_SO):
        write_scene_json(tmp_scene, objs)
        ref = Reference()
        assert ref.load_scene(tmp_scene) == len(objs)
        ref.setup(w, h, fov, DEPTH, False, cam)
        sec, segs = ref.render_frames(frames, rng_mode=0, count_segments=True)
        info = {"kind": "reference", "cores": cores, "threads": 16, "seconds": sec, "segments": int(segs),
                "sample": "%d frames of 1 spp at %dx%d, depth %d, %s; reference's own renderArea loop, 16 threads, per-thread MSVC rand()" % (frames, w, h, DEPTH, label)}
        if frames >= 8:      # SURVEY.md 8d: both rand() variants. glibc's rand() is ONE locked global state: the 16 workers serialise on it
            n2 = max(2, frames // 12)
            sec2, segs2 = ref.render_frames(n2, rng_mode=2, count_segments=True)
            info["glibc_rand_variant"] = {"value": segs2 / sec2 / 1e6, "unit": UNIT, "sample": "%d frames, rand() = glibc's global locked generator" % n2}
        return segs / sec, info
    orc = Oracle()
    cam = OrcCamera(); cam.right[0] = 1; cam.up[1] = 1; cam.forward[2] = 1; cam.fov_deg = 55
    p = orc.default_params(width=w, height=h, max_bounces=DEPTH, mode=0)
    sec, segs = orc.time_render(objs, cam, p, frames, rng_mode=0, threads=cores)
    return segs / sec, {"kind": "port", "cores": cores, "threads": cores, "seconds": sec, "segments": int(segs),
                        "sample": "%d spp at %dx%d, depth %d, Scene1; validated C port, %d threads" % (frames, w, h, DEPTH, cores)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    objs = load_scene()
    frames_per_step = 2
    for _ in range(args.warmup):
        cpu_reference_run(objs, 1)
    times, segs = [], 0
    info = None
    for _ in range(args.steps):
        rate, info = cpu_reference_run(objs, frames_per_step)
        times.append(info["seconds"]); segs += info["segments"]
    total = sum(times)
    value = segs / total / 1e6
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic: bundled Scene1 fixture, default camera",
            "config": workload_config("Scene1", len(objs)),
            "step": "%d frames of 1 spp on the host CPU (rate metric: a bounded sample of the same workload)" % frames_per_step,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": info["cores"], "kind": info["kind"], "sample": info["sample"]},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "paths_per_s_M": (W * H * frames_per_step * args.steps) / total / 1e6}
    print(json.dumps(line), flush=True)


# ---- workloads ---------------------------------------------------------------------------------------------------
def make_workload(config, scene, spp_arg):
    """BASELINE.json configs[0..4] -> dict(objs, cam, mesh, w, h, spp, labels)."""
    import rtb200
    wl = {"objs": load_scene(scene), "cam": rtb200.default_camera(), "mesh": None, "w": W, "h": H, "spp": spp_arg or SPP, "scene": scene,
          "workload": "%s (%d objects)" % (scene, len(load_scene(scene))), "scene_label": "bundled %s" % scene,
          "data": "synthetic: bundled %s fixture (tests/golden/bundled_scenes.npz), default camera, Philox seeds" % scene}
    if config == "c3":                                   # configs[2]: 10k random spheres at 4K
        from rtb200.scenes import synthetic_spheres, config3_camera
        wl.update(objs=synthetic_spheres(10000), cam=config3_camera(rtb200.default_camera), w=3840, h=2160, spp=spp_arg or 16, scene="synthetic10k",
                  workload="config 3: 10 000 random spheres + ground + 8 lights", scene_label="synthetic 10k spheres",
                  data="synthetic: rtb200.scenes.synthetic_spheres(10000) (seeded), config3_camera, Philox seeds")
    elif config == "c4":                                 # configs[3]: ~1M-triangle mesh through the BVH
        from rtb200.scenes import heightfield_mesh, mesh_scene
        cam = rtb200.default_camera(); cam.pos[1] = 1.5; cam.pos[2] = -1.0
        wl.update(objs=mesh_scene(), mesh=heightfield_mesh(1024, 512), cam=cam, spp=spp_arg or 64, scene="mesh1M",
                  workload="config 4: 1 048 576-triangle heightfield mesh + 3 spheres", scene_label="synthetic 1M-triangle mesh",
                  data="synthetic: rtb200.scenes.heightfield_mesh(1024, 512) (seeded) + mesh_scene(), Philox seeds")
    elif config == "c5":                                 # configs[4]: interactive 1 spp frames at 720p
        wl.update(w=1280, h=720, spp=1)
    elif config == "c1":                                 # configs[0]: the reference's own CPU-runnable case
        wl.update(w=640, h=480, spp=spp_arg or 64)
    return wl


def make_tracer(args, device, stream_handle, wl, seed_hi=0):
    import rtb200
    tr = rtb200.PathTracer(device)
    if stream_handle is not None:
        tr.set_stream(stream_handle)
    tr.set_option(rtb200.RT_OPT_ACCEL, {"auto": rtb200.RT_ACCEL_AUTO, "brute": rtb200.RT_ACCEL_BRUTE, "bvh": rtb200.RT_ACCEL_BVH,
                                        "flat": rtb200.RT_ACCEL_FLAT}[args.accel])
    tr.set_option(rtb200.RT_OPT_PRIMARY_REUSE, 0 if args.no_primary_reuse else 1)
    tr.set_option(rtb200.RT_OPT_PIPELINE, {"auto": rtb200.RT_PIPELINE_AUTO, "regen": rtb200.RT_PIPELINE_REGEN, "wavefront": rtb200.RT_PIPELINE_WAVEFRONT,
                                           "stream": rtb200.RT_PIPELINE_STREAM}[args.pipeline])
    for opt, v in ((rtb200.RT_OPT_BVH_SCHED, args.bvh_sched), (rtb200.RT_OPT_BVH_WIDE, args.bvh_wide), (rtb200.RT_OPT_BVH_WAIT_K, args.wait_k),
                   (rtb200.RT_OPT_FLAT_COOP, args.flat_coop), (rtb200.RT_OPT_WF_REFILL, args.wf_refill), (rtb200.RT_OPT_WF_NODE_MIN, args.wf_node_min),
                   (rtb200.RT_OPT_WF_WAVE_MPATHS, args.wave_mpaths)):
        if v >= 0:
            tr.set_option(opt, v)
    tr.set_scene(wl["objs"])
    if wl["mesh"] is not None:
        tr.set_mesh(0, wl["mesh"][0], wl["mesh"][1])
    tr.set_camera(wl["cam"])
    tr.set_params(rtb200.default_params(width=wl["w"], height=wl["h"], mode=rtb200.RT_MODE_PATH, max_bounces=DEPTH, seed_lo=2026, seed_hi=seed_hi))
    tr.reset_accumulation()
    return tr


ACCEL_NAMES = {1: "brute-force object loop", 2: "host-built BVH candidates + strict tests",
               3: "flat two-level accelerator (conservative FMA culls, warp-uniform) + strict tests"}
PIPE_NAMES = {1: "regeneration megakernel", 2: "wavefront (raygen / persistent intersect / shade + ballot compaction)",
              3: "streaming (one persistent kernel: lanes claim paths, traverse with postponed leaves, shade and continue; no per-bounce state)"}


def fp32_roofline(objs, st, delivered_per_step, traced_per_step, kern_s, peaks, peaks_src, w, h):
    """Brute-force-equivalent FLOP roofline of the small-scene kernels (SURVEY.md 8d). `frac` is taken on the closest-hit
    queries the launch EXECUTES; the delivered-segment figure (primary-hit reuse credits the cached primary segments) is kept
    beside it."""
    fps = flops_per_segment(objs)
    sm_mhz = peaks.get("sm_max_mhz", 1965.0)
    peak_tf = st.sm_count * 128 * 2 * sm_mhz * 1e6 / 1e12
    ach_exec = traced_per_step * fps / kern_s / 1e12
    ach_deliv = delivered_per_step * fps / kern_s / 1e12
    return {"bound": "fp32", "achieved": ach_exec, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach_exec / peak_tf,
            "basis": "executed closest-hit queries x the reference's brute-force op count per segment (23/sphere + 30/cube + 110)",
            "achieved_delivered": ach_deliv, "frac_delivered": ach_deliv / peak_tf,
            "traffic": 86.2e6 * (w * h) / (1920 * 1080), "traffic_note": "dram read+write per launch, ncu --set full at 1080p (profiles/r2v_summary_regen_c2_1024spp.txt: 75.4 MB read + 10.8 MB written) scaled by pixel count: the primary-hit cache (20 B per pixel) and the float4 accumulation buffer once, the write mostly still in L2 when the launch ends; independent of spp",
            "kernel": "k_render_regen", "kernel_ms": kern_s * 1e3, "flop_per_segment": fps,
            "peak_source": "%d SMs x 128 lanes x 2 (FMA) x %.0f MHz (%s MEASURED_PEAKS.json sm_max_mhz)" % (st.sm_count, sm_mhz, peaks_src),
            "note": "path is FP32-CUDA-core issue bound, not HBM or tensor (SURVEY.md 8d). The strict-IEEE build (-fmad=false) issues multiply and add separately, "
                    "so the attainable rate on this arithmetic is half the FMA peak; the flat accelerator's conservative culls execute far fewer operations than the "
                    "brute-force count. ncu (profiles/): issue slots busy, active threads per instruction and warp instructions per executed query are the hardware-side figures",
            "hbm_peak_gbs": peaks.get("hbm_gbs"), "hbm_algorithmic_gbs": (w * h * 32 / kern_s) / 1e9}


# dram__bytes_read.sum + dram__bytes_write.sum of the dominant launch, from the committed ncu captures (profiles/r3a_summary_wavefront_*.txt)
NCU_BVH_TRAFFIC = {("synthetic10k", 2): 5.545e9, ("mesh1M", 2): 4.951e9}


def bvh_roofline(tr, wl, spp, traced_per_s, kern_share, peaks, peaks_src, pipeline):
    """SURVEY.md 8d for BVH scenes: bytes per segment = node bytes x <nodes visited> + primitive bytes x <primitives tested>,
    from the device's own traversal counters (one extra untimed step with RT_OPT_TRAVERSAL_STATS), times the executed query
    rate. BVH and primitives are L2-resident on these scenes, so the figure is compared with the measured HBM copy bandwidth
    only as a yardstick (it can exceed it); dram traffic per launch comes from ncu."""
    import rtb200
    tr.set_option(rtb200.RT_OPT_TRAVERSAL_STATS, 1)
    tr.reset_accumulation(); tr.render_spp(spp)
    ts = tr.traversal_stats()
    tr.set_option(rtb200.RT_OPT_TRAVERSAL_STATS, 0)
    q = max(ts.queries, 1)
    nodes, sph, cube, tri = ts.node_visits / q, ts.sphere_tests / q, ts.cube_tests / q, ts.tri_tests / q
    bytes_per_query = ts.node_bytes * nodes + 20 * sph + 36 * cube + 52 * tri
    flop_per_query = 40 * nodes + 23 * sph + 30 * cube + 40 * tri + 110      # two slab tests per node visit ~ 2 x 20
    ach = bytes_per_query * traced_per_s / 1e9
    peak = peaks.get("hbm_gbs", 6650.0)
    wf = pipeline == rtb200.RT_PIPELINE_WAVEFRONT
    kname = {rtb200.RT_PIPELINE_WAVEFRONT: "k_wf_intersect_bvh", rtb200.RT_PIPELINE_STREAM: "k_wf_stream"}.get(pipeline, "k_render_regen<3>")
    return {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
            "basis": "executed closest-hit queries/s x (%d B x %.1f node visits + 20 B x %.2f sphere + 36 B x %.2f cube + 52 B x %.2f triangle tests) per query, device counters of this run"
                     % (ts.node_bytes, nodes, sph, cube, tri),
            "bytes_per_query": bytes_per_query, "node_visits_per_query": nodes, "prim_tests_per_query": sph + cube + tri, "flop_per_query": flop_per_query,
            "achieved_tflops": flop_per_query * traced_per_s / 1e12,
            "traffic": NCU_BVH_TRAFFIC.get((wl["scene"], pipeline)),
            "traffic_note": "dram read+write of the dominant launch (first bounce round of a full wave: c3 133 M rays, c4 69 M rays), ncu --set full, profiles/r3a_summary_wavefront_c3.txt / "
                            "_c4.txt (3.43 + 2.11 GB and 3.87 + 1.08 GB): the rays read and the hits written; BVH + primitives are L2-resident (0.9 MB / 75 MB in a 126 MB L2). null = no capture of this pipeline",
            "kernel": kname, "kernel_share_of_step": kern_share,
            "peak_source": "%s MEASURED_PEAKS.json hbm_gbs" % peaks_src,
            "note": "node and primitive fetches are served by L1/L2, not HBM: frac is algorithmic bytes against the HBM copy peak as SURVEY.md 8d defines it; the kernel is bound by "
                    "instruction issue under divergence and dependent L2 round trips (ncu: issue slots busy, long-scoreboard stalls, L1 hit rate in profiles/)"}


# ---- one short leg of a non-headline config (N = 1) ----------------------------------------------------------------
def run_leg(args, config, torch, stream, steps=3, warmup=3):
    import rtb200
    wl = make_workload(config, "Scene1", 0)
    tr = make_tracer(args, 0, stream.cuda_stream, wl)
    w, h, spp = wl["w"], wl["h"], wl["spp"]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    peaks, peaks_src = measured_peaks()
    with torch.cuda.stream(stream):
        if config == "c5":
            line = interactive_line(tr, wl, frames=1000)     # SURVEY.md 8d: p50 / p99 over 1000 frames
            tr.close()
            return line
        for _ in range(warmup):
            tr.reset_accumulation(); tr.render_spp(spp)
        torch.cuda.synchronize()
        s0 = tr.stats()
        sampler = ClockSampler(0)
        sampler.sample_once()                            # before and after, not during: see sample_once()
        evs = []
        tr.reset_accumulation()
        for _ in range(steps):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream); tr.render_spp(spp); e1.record(stream)
            evs.append((e0, e1))
        torch.cuda.synchronize()
        sampler.sample_once()
        clocks = sampler.summary()
        clocks["sampling"] = "one query right before and one right after the leg's timed steps"
        ms = [a.elapsed_time(b) for a, b in evs]
        s1 = tr.stats()
    total_s = sum(ms) * 1e-3
    segs, traced = s1.total_segments - s0.total_segments, s1.total_traced_segments - s0.total_traced_segments
    paths = w * h * spp * steps
    out = {"config": config, "workload": "%s %dx%d, %d spp per step, depth %d" % (wl["workload"], w, h, spp, DEPTH), "data": wl["data"],
           "value": segs / total_s / 1e6, "unit": UNIT, "traced_segments_per_s_M": traced / total_s / 1e6, "paths_per_s_M": paths / total_s / 1e6,
           "ms_per_step": 1e3 * total_s / steps, "steps": steps, "warmup": warmup, "segments_per_path": segs / paths, "traced_segments_per_path": traced / paths,
           "accel": ACCEL_NAMES[s1.accel], "pipeline": PIPE_NAMES[s1.pipeline], "clocks": clocks}
    kern_s = statistics.mean(ms) * 1e-3
    if s1.accel == rtb200.RT_ACCEL_BVH:
        out["roofline"] = bvh_roofline(tr, wl, spp, traced / total_s, 0.8 if s1.pipeline == rtb200.RT_PIPELINE_WAVEFRONT else 0.98, peaks, peaks_src, s1.pipeline)
    else:
        out["roofline"] = fp32_roofline(wl["objs"], s1, segs / steps, traced / steps, kern_s, peaks, peaks_src, w, h)
    tr.close()
    del flush
    return out


def interactive_line(tr, wl, frames, outputs=None):
    """BASELINE.json configs[4]: progressive 1 spp frames at 1280x720, each frame = rt_render_frame(1) into a HOST surface
    (3.7 MB per frame over PCIe), what a viewer's frame loop does (Raytracer.cpp:572-595). Frame latency p50/p99 (host clock around
    the call, which synchronises), the same frame as rt_render_spp + rt_resolve_rgba8, and the device time of the render kernel alone.
    `outputs` (a dict) receives the last timed frame as "surface_argb"."""
    import rtb200
    w, h = wl["w"], wl["h"]
    out, _owner = rtb200.host_surface(w, h)              # page-locked surface (rt_host_alloc): one DMA per frame
    for _ in range(20):
        tr.render_frame(1, True, out)
    lat2 = []
    for _ in range(frames // 4):                         # the two-call form of the same frame, for comparison
        t0 = time.perf_counter()
        tr.render_spp(1)
        tr.resolve_rgba8(True, out)
        lat2.append((time.perf_counter() - t0) * 1e3)
    lat2.sort()
    tr.reset_accumulation(); tr.sync()
    st0 = tr.stats()
    lat, dev = [], []
    t_all = time.perf_counter()
    for _ in range(frames):
        t0 = time.perf_counter()
        tr.render_frame(1, True, out)                    # rt_render_frame: synchronises, the frame is on the host
        lat.append((time.perf_counter() - t0) * 1e3)
    total = time.perf_counter() - t_all
    if outputs is not None:
        outputs["surface_argb"] = argb_channels(out)
    for _ in range(50):                                  # device time of the render kernel (rt_get_stats synchronises: outside the latency loop)
        tr.render_spp(1)
        dev.append(tr.stats().last_render_ms)
    st1 = tr.stats()
    segs = st1.total_segments - st0.total_segments
    traced = st1.total_traced_segments - st0.total_traced_segments
    n_all = frames + 50
    lat.sort(); dev.sort()
    kern_s = dev[len(dev) // 2] * 1e-3
    peaks, peaks_src = measured_peaks()
    line = {"config": "c5", "metric": "frame latency, progressive 1 spp/frame (BASELINE.json configs[4])", "value": lat[len(lat) // 2], "unit": "ms (p50)",
            "p99_ms": lat[int(len(lat) * 0.99) - 1], "mean_ms": 1e3 * total / frames, "frames": frames, "fps": frames / total,
            "render_kernel_ms_p50": dev[len(dev) // 2], "two_call_frame_ms_p50": lat2[len(lat2) // 2], "higher_is_better": False,
            "workload": "Scene1 %dx%d, 1 spp per frame, depth %d, one rt_render_frame per frame: the render kernel resolves the pixels it finishes and streams them (%d bytes per frame) into a page-locked host surface while it traces; two_call_frame = rt_render_spp + rt_resolve_rgba8 (render, resolve, copy one after the other); static camera: primary hits come from the per-pixel cache"
                        % (w, h, DEPTH, w * h * 4),
            "data": wl["data"], "Msegments_per_s": segs / n_all / (total / frames) / 1e6, "segments_per_path": segs / (w * h * n_all), "traced_segments_per_path": traced / (w * h * n_all),
            "accel": ACCEL_NAMES[st1.accel], "pipeline": PIPE_NAMES[st1.pipeline],
            "roofline": fp32_roofline(wl["objs"], st1, segs / n_all, traced / n_all, kern_s, peaks, peaks_src, w, h)}
    line["roofline"]["kernel"] = "k_render_pool"
    return line


def run_b200(args):
    import torch
    import torch.distributed as dist
    import rtb200

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # keep stdout to the one JSON line: NCCL's version banner / debug output goes to stderr
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    strong = args.scaling == "strong"
    wl = make_workload(args.config, args.scene, args.spp)
    w, h, spp, objs, mesh, cam0 = wl["w"], wl["h"], wl["spp"], wl["objs"], wl["mesh"], wl["cam"]
    stream = torch.cuda.Stream()
    # weak scaling: every rank its own sample streams (seed_hi = rank); strong: ONE global sample sequence, sharded
    tr = make_tracer(args, local, stream.cuda_stream, wl, seed_hi=0 if strong else rank)
    if strong:
        tr.set_shard(rank, world)
    outputs = {}
    if args.config == "c5":
        with torch.cuda.stream(stream):
            line = interactive_line(tr, wl, frames=max(args.steps, 1) * 200, outputs=outputs)
        line.update({"n_gpus": 1, "dtype": "f32", "config": {"workload": line.pop("workload")}})
        print(json.dumps(line), flush=True)
        tr.close()
        if args.dump_outputs:
            write_outputs(args.dump_outputs, outputs)
        return

    class DevBuf:                                   # wrap the library's accumulation buffer for torch / NCCL
        def __init__(self, ptr, n):
            self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f4", "data": (ptr, False), "version": 2}
    accum = torch.as_tensor(DevBuf(tr.accum_device_ptr(), w * h * 4), device=torch.device("cuda", local))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")       # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # N > 1: map every rank's accumulation buffer and exchange flags (and rank 0's surface) through CUDA IPC once; after that
    # the exchange needs no collective and no host synchronisation (rt_exchange_resolve)
    fused = world > 1 and args.reduce == "fused"
    if fused:
        def gather_handles(which):
            mine = torch.tensor(list(tr.ipc_export(which)), dtype=torch.uint8, device="cuda")
            allh = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(allh, mine)
            return [bytes(x.cpu().tolist()) for x in allh]
        acc_h, srf_h, flg_h = gather_handles(0), gather_handles(1), gather_handles(2)
        tr.exchange_setup(rank, world, [None if r == rank else tr.ipc_open(acc_h[r]) for r in range(world)],
                          [None if r == rank else tr.ipc_open(flg_h[r]) for r in range(world)], None if rank == 0 else tr.ipc_open(srf_h[0]))
        barrier()
    total_spp = spp if strong else spp * world      # samples per pixel in the reduced image

    def exchange():
        """the path's one exchange step (N > 1), stream-ordered on every rank."""
        if fused:
            tr.exchange_resolve(total_spp)
        else:
            dist.all_reduce(accum)

    def step_resident():
        """device-resident step: samples into the accumulation buffer (+ the one exchange at N > 1)."""
        tr.reset_accumulation()                      # N > 1: every step is a whole frame (the exchange consumes the buffers)
        tr.render_spp(spp)
        if world > 1:
            exchange()

    def timed(n_steps):
        evs = []
        for _ in range(n_steps):
            flush.fill_(1)                                                  # L2 flush between timed steps
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream); step_resident(); e1.record(stream)
            evs.append((e0, e1))
        barrier()
        return [a.elapsed_time(b) for a, b in evs]

    # ---- device-timed: value ---------------------------------------------------------------
    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            step_resident()
        barrier()
        s0 = tr.stats()
        sampler = ClockSampler(local); sampler.start()
        barrier()
        step_ms = timed(args.steps)
        clocks = sampler.summary()
        if args.dump_outputs and rank == 0:                  # before anything else renders into the buffers
            if fused:
                outputs["surface_argb"] = argb_channels(tr.read_surface())
            else:
                outputs["accum"] = tr.read_accum()[0]
        s1 = tr.stats()
        segs_rank = s1.total_segments - s0.total_segments
        traced_rank = s1.total_traced_segments - s0.total_traced_segments
        paths_rank = (w * h * spp * args.steps) // (world if strong else 1)

        # ---- multi-GPU check, outside the timed region: fused surface == resolve of the sum of all ranks' buffers -----
        multi_check = None
        if world > 1 and fused:
            step_resident()
            barrier()
            parts = [torch.empty_like(accum) for _ in range(world)]
            dist.all_gather(parts, accum)
            if rank == 0:
                total = parts[0].clone()
                for p in parts[1:]:
                    total += p                       # rank order: the fused kernel's summation order
                ref_surface = torch.empty(w * h, dtype=torch.int32, device="cuda")
                tr.resolve_device(total.data_ptr(), total_spp, 0, w * h, ref_surface.data_ptr(), True)   # a slice resolve keeps the y-up pixel order
                tr.sync()
                got = torch.from_numpy(tr.read_surface().view(np.int32)).cuda()                        # the fused surface is y-down
                multi_check = "ok" if bool(torch.equal(got, ref_surface.view(h, w).flip(0))) else "MISMATCH"
            barrier()

        # ---- the exchange alone (N > 1): every rank's buffer already rendered ------------------------------------------
        exchange_ms = None
        if world > 1:
            ex = []
            for _ in range(5):
                barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream); exchange(); e1.record(stream)
                barrier()
                ex.append(e0.elapsed_time(e1))
            exchange_ms = statistics.median(ex)

        # ---- end to end through the C-ABI with host buffers: e2e ------------------------------
        out = np.zeros((h, w), np.uint32)

        def step_e2e():
            if mesh is None:
                tr.set_scene(objs)                   # host rt_object[] -> device SoA (H2D)
            tr.set_camera(cam0)
            tr.reset_accumulation()
            tr.render_spp(spp)
            if world > 1:
                exchange()
                if fused:
                    if rank == 0:
                        out[:] = tr.read_surface()   # D2H of the fused result
                    else:
                        tr.sync()
                    return
                tr.set_sample_count(total_spp)
            tr.resolve_rgba8(True, out)              # Reinhard + pack, D2H into the host surface; synchronises
        for _ in range(max(1, args.warmup - 1)):
            step_e2e()
        barrier()
        seg1 = tr.stats().total_segments
        t0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            step_e2e()
        e1.record(stream)
        barrier()
        e2e_wall = time.perf_counter() - t0
        e2e_dev_ms = e0.elapsed_time(e1)
        e2e_segs = tr.stats().total_segments - seg1

        # ---- strong scaling beside the weak headline (N > 1, headline config): the same 1024 global samples, sharded -----
        strong_obj = None
        if world > 1 and not strong and fused and args.config == "c2":
            tr.set_params(seed_hi=0)                 # one global sample sequence
            tr.set_shard(rank, world)
            total_spp_keep, total_spp = total_spp, spp
            for _ in range(3):
                step_resident()
            barrier()
            sg0 = tr.stats().total_segments
            k = max(args.steps, 5)
            sms = timed(k)
            sg = tr.stats().total_segments - sg0
            tt = torch.tensor([sum(sms), float(sg)], dtype=torch.float64, device="cuda")
            tmx = tt.clone(); dist.all_reduce(tmx, op=dist.ReduceOp.MAX)
            tsm = tt.clone(); dist.all_reduce(tsm, op=dist.ReduceOp.SUM)
            strong_obj = {"scaling": "strong", "spp_total_per_step": spp, "spp_per_gpu_per_step": spp / world, "steps": k,
                          "ms_per_step": tmx[0].item() / k, "value": tsm[1].item() / (tmx[0].item() * 1e-3) / 1e6, "unit": UNIT,
                          "note": "fixed total work: rt_set_shard(rank, %d), one shared seed, reset + render + exchange per step; compare ms_per_step with the N=1 line" % world}
            total_spp = total_spp_keep

    total_ms = sum(step_ms)
    t = torch.tensor([total_ms, e2e_wall * 1e3, float(segs_rank), float(e2e_segs), float(traced_rank)], dtype=torch.float64, device="cuda")
    if world > 1:
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        total_ms, e2e_ms = tmax[0].item(), tmax[1].item()
        segs_all, e2e_segs_all, traced_all = tsum[2].item(), tsum[3].item(), tsum[4].item()
    else:
        e2e_ms, segs_all, e2e_segs_all, traced_all = e2e_wall * 1e3, float(segs_rank), float(e2e_segs), float(traced_rank)

    if rank == 0:
        peaks, peaks_src = measured_peaks()
        st = tr.stats()
        value = segs_all / (total_ms * 1e-3) / 1e6
        kern_s = statistics.mean(step_ms) * 1e-3     # dominant kernel = one k_render_regen launch per step; its duration = the step (N = 1)
        wf = st.pipeline == rtb200.RT_PIPELINE_WAVEFRONT
        streamk = st.pipeline == rtb200.RT_PIPELINE_STREAM
        cfg = workload_config(wl["scene"], len(objs), w, h)
        par = "single GPU" if world == 1 else ("spp-sharded x%d (%s scaling), " % (world, args.scaling)) + \
            ("fused reduce+resolve kernel over NVLink peer memory, ranks ordered by device-side flags (rt_exchange_resolve)" if fused else "one NCCL all-reduce per step")
        line = {
            "metric": METRIC.replace("bundled Scene1", wl["scene_label"]).replace("1920x1080", "%dx%d" % (w, h)), "value": value, "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32", "data": wl["data"], "config": cfg,
            "step": "%d spp %s per step" % (spp, "in total, sharded over the GPUs" if strong else "per GPU"),
            "implementation": {"parallelism": par, "build": "strict IEEE, -fmad=false (bit-exact geometry vs the reference)", "accel": ACCEL_NAMES[st.accel], "pipeline": PIPE_NAMES[st.pipeline],
                               "primary_reuse": ("off: every sample re-traces its primary ray" if args.no_primary_reuse else
                                                 "on: the reference has no pixel jitter, so the primary closest-hit query of a pixel is identical for all samples of all frames; it is traced "
                                                 "once per camera/scene change into a per-pixel cache and every sample shades/scatters from it (bit-identical radiance; `value` counts path "
                                                 "segments delivered, traced_segments_per_s_M the queries executed)")},
            "paths_per_s_M": paths_rank * world / (total_ms * 1e-3) / 1e6,
            "ms_per_1spp_frame": total_ms / args.steps / (spp if strong else spp),
            "segments_per_path": segs_rank / paths_rank,
            "traced_segments_per_s_M": traced_all / (total_ms * 1e-3) / 1e6,
            "traced_segments_per_path": traced_rank / paths_rank,
            "e2e": {"value": e2e_segs_all / (e2e_ms * 1e-3) / 1e6, "unit": UNIT,
                    "h2d_bytes_per_step": int(objs.nbytes + 52), "d2h_bytes_per_step": int(w * h * 4),
                    "ms_per_step": e2e_ms / args.steps, "device_ms_per_step": e2e_dev_ms / args.steps,
                    "api": "rt_set_scene + rt_set_camera + rt_reset_accumulation + rt_render_spp + " + ("rt_resolve_rgba8(host)" if world == 1 else "rt_exchange_resolve + rt_read_surface(host)")},
            "clocks": clocks,
        }
        if wf:
            line["gpu_launches"] = int(args.steps * (3 + 2 * DEPTH) * 2)
            line["gpu_launches_detail"] = "per rank: the wavefront pipeline launches raygen + 2 kernels per bounce round per wave (about 20 per step) + accumulate/commit, in both timed regions"
        elif streamk:
            line["gpu_launches"] = int(args.steps * 3 * 2)
            line["gpu_launches_detail"] = "per rank and wave: k_wf_stream + k_wf_accumulate, + k_wf_commit per step, in both timed regions"
        else:
            per_step = 1 + (2 if world > 1 else 0)   # k_render_regen (+ k_resolve_fused_sync + k_exchange_wait)
            per_e2e = 2 + (1 if world == 1 else 2)   # k_primary_cache (the scene is re-submitted) + k_render_regen + k_resolve | the two exchange kernels
            line["gpu_launches"] = int(args.steps * (per_step + per_e2e))
            line["gpu_launches_detail"] = ("per rank. timed value region: 1 k_render_regen per step" + (" + k_resolve_fused_sync + k_exchange_wait" if world > 1 else "") +
                                           "; e2e region: k_primary_cache + k_render_regen + " + ("k_resolve" if world == 1 else "k_resolve_fused_sync + k_exchange_wait") + " per step")
        if st.accel == rtb200.RT_ACCEL_BVH:
            line["roofline"] = bvh_roofline(tr, wl, spp, traced_rank / (sum(step_ms) * 1e-3), 0.8 if wf else 0.98, peaks, peaks_src, st.pipeline)
        else:
            line["roofline"] = fp32_roofline(objs, st, segs_rank / args.steps, traced_rank / args.steps, kern_s, peaks, peaks_src, w, h)
        if world > 1:
            line["multi_gpu_check"] = multi_check if multi_check is not None else "not run (--reduce nccl)"
            line["exchange_ms"] = exchange_ms
            if strong_obj:
                line["strong"] = strong_obj
    tr.close()
    del accum, flush
    if rank == 0:
        if world == 1 and args.config == "c2" and not args.no_configs and args.scene == "Scene1":
            legs = []
            for c in ("c1", "c3", "c4", "c5"):
                try:
                    legs.append(run_leg(args, c, torch, stream))
                except Exception as e:                # a leg must not take the headline down with it
                    legs.append({"config": c, "error": "%s: %s" % (type(e).__name__, e)})
            line["configs"] = legs
            # the metric's "ms/frame at 1080p", measured (ms_per_1spp_frame above is the 1024-spp step divided by its samples): one
            # rt_render_frame(1) per frame at 1920x1080 into a page-locked host surface, static camera, as the c5 leg does at 720p
            try:
                wl_f = make_workload("c2", "Scene1", 1)
                tr_f = make_tracer(args, 0, stream.cuda_stream, wl_f)
                with torch.cuda.stream(stream):
                    fl = interactive_line(tr_f, wl_f, frames=200)
                tr_f.close()
                line["frame_1080p_1spp"] = {"p50_ms": fl["value"], "p99_ms": fl["p99_ms"], "render_kernel_ms_p50": fl["render_kernel_ms_p50"], "frames": fl["frames"],
                                            "what": "host clock around rt_render_frame(1) at 1920x1080: render + resolve + 8.3 MB to the host per frame"}
            except Exception as e:
                line["frame_1080p_1spp"] = {"error": "%s: %s" % (type(e).__name__, e)}
        # the CPU baseline comes LAST: measured on the same box, the BVH legs (about 40 small launches per step) ran 11-19 % slower
        # when they followed the reference's 16-thread CPU run (profiles/r2l_bench_n1.json vs the --no-cpu run of the same call)
        if world == 1 and not args.no_cpu and args.config in ("c1", "c2"):
            rate, info = cpu_reference_run(objs, args.cpu_frames, w, h)
            line["cpu_baseline"] = {"value": rate / 1e6, "unit": UNIT, "cores": info["cores"], "kind": info["kind"],
                                    "sample": info["sample"], "threads": info["threads"]}
            # config 3 on the CPU: the reference has no accelerator, its loop tests all 10 009 objects per segment - a small frame of the
            # same scene and camera is all it can do in seconds (a rate, resolution-independent up to the sky / object mix)
            for leg in line.get("configs", []):
                if leg.get("config") == "c4" and "error" not in leg:
                    leg["cpu_baseline"] = None
                    leg["cpu_baseline_note"] = ("the reference has no triangle path (SURVEY.md 8d): nothing of its own to time; the mesh extension is pinned by the oracle's brute force "
                                                "and a float64 Moller-Trumbore check on sampled rays (tests), which are correctness checks, not baselines")
                if leg.get("config") == "c3" and "error" not in leg:
                    try:
                        wl3 = make_workload("c3", "Scene1", 0)
                        r3, i3 = cpu_reference_run(wl3["objs"], 1, 256, 144, cam=wl3["cam"], fov=int(wl3["cam"].fov_deg), label="the config-3 scene and camera")
                        leg["cpu_baseline"] = {"value": r3 / 1e6, "unit": UNIT, "cores": i3["cores"], "kind": i3["kind"], "threads": i3["threads"], "sample": i3["sample"]}
                    except Exception as e:
                        leg["cpu_baseline"] = {"error": "%s: %s" % (type(e).__name__, e)}
            line["cpu_baseline"]["paths_per_s_M"] = args.cpu_frames * w * h / info["seconds"] / 1e6
            line["cpu_baseline"]["ms_per_1spp_frame"] = 1e3 * info["seconds"] / args.cpu_frames
            if "glibc_rand_variant" in info:
                line["cpu_baseline"]["glibc_rand_variant"] = info["glibc_rand_variant"]
        print(json.dumps(line), flush=True)
        if args.dump_outputs:
            write_outputs(args.dump_outputs, outputs)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c2", choices=["c1", "c2", "c3", "c4", "c5"],
                    help="BASELINE.json configs[0..4]; the headline (and default) is c2, whose line also carries short legs of the others")
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--spp", type=int, default=0, help="samples per pixel per step: per GPU (weak) or in total (strong); default: the config's (c2 1024, c1 64, c3 16, c4 64)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="N > 1: weak = every GPU renders --spp samples of its own; strong = --spp samples in total, sharded by rt_set_shard")
    ap.add_argument("--cpu-frames", type=int, default=24, help="1-spp frames of the CPU baseline sample")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the short legs of the other configs")
    ap.add_argument("--accel", default="auto", choices=["auto", "brute", "bvh", "flat"], help="closest-hit back end (results are identical)")
    ap.add_argument("--pipeline", default="auto", choices=["auto", "regen", "wavefront", "stream"],
                    help="regen: persistent-lane regeneration megakernel (default); wavefront: raygen/intersect/shade kernels over device queues (bit-identical)")
    ap.add_argument("--no-primary-reuse", action="store_true", help="re-trace the (identical) primary ray for every sample, like the reference")
    ap.add_argument("--reduce", default="fused", choices=["fused", "nccl"], help="N > 1 exchange: fused peer-memory reduce+resolve kernel with device-side ordering, or NCCL all-reduce")
    ap.add_argument("--bvh-sched", type=int, default=-1, help="RT_OPT_BVH_SCHED override")
    ap.add_argument("--wait-k", type=int, default=-1, help="RT_OPT_BVH_WAIT_K override")
    ap.add_argument("--bvh-wide", type=int, default=-1, help="RT_OPT_BVH_WIDE: 0 binary BVH nodes (default), 1 8-wide quantised nodes for 1024+ primitives, 2 always")
    ap.add_argument("--flat-coop", type=int, default=-1, help="RT_OPT_FLAT_COOP: 0 per-lane levels 2/3, 1 warp-cooperative, 2 measured per scene (default)")
    ap.add_argument("--wf-refill", type=int, default=-1, help="RT_OPT_WF_REFILL override")
    ap.add_argument("--wf-node-min", type=int, default=-1, help="RT_OPT_WF_NODE_MIN override")
    ap.add_argument("--wave-mpaths", type=int, default=-1, help="RT_OPT_WF_WAVE_MPATHS override")
    ap.add_argument("--scene", default="Scene1", help="bundled scene fixture (the headline config is Scene1)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
