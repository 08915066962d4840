"""GPU (B200): the pixel filter (rt_set_pixel_filter, csrc/rt_filter.cuh) through the C-ABI.

rt_read_sample_dirs against the float32 numpy statement bit for bit; every jittered render form against the oracle with the filter in
front (tests/oracle_filtered.c) with exact segment counts; pipeline requests that fall back to the megakernel; NONE restoring today's bits;
call splits, shards and a group; anti-aliasing itself (filter-weighted coverage of an emissive sphere's edge pixels); the present
paths on a filtered buffer; and the frames that ignore the filter."""
import math

import numpy as np
import pytest
from scipy import ndimage

import rtb200
import filter_reference as ref
from conftest import SEED
from oracle_filtered import filtered_oracle
from oracle_py import OrcCamera
from test_gpu_render_params import DEFAULT_OPTIONS, FORMS, SHORT, SPLIT, H, W, camera, close, load, scene_of, set_options
from test_render_params_cpu import make_params

pytestmark = pytest.mark.gpu

O = rtb200
FILTERS = [(O.RT_FILTER_BOX, 0.5), (O.RT_FILTER_TENT, 1.0)]
AA_FORMS = ["lane", "pixel_pool", "flat_pooled", "flat_lane", "brute", "bvh_float_nodes", "bvh_quant_nodes", "bvh_wide", "traversal_stats"]
SETS = ["defaults", "bounces_3"]


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


_ORACLE = {}


def expected_filtered(oracle, scenes, key, name, calls, ftype, radius):
    total, segs, s0 = np.zeros((H, W, 3), np.float32), 0, 0
    for n in calls:
        k = (key, name, s0, n, ftype, radius)
        if k not in _ORACLE:
            objs, _, _, _ = scene_of(scenes, key)
            p = make_params(oracle.default_params, name, W, H)
            _ORACLE[k] = filtered_oracle().render_filtered(objs, camera(OrcCamera, scenes, key, name), p, s0, n, ftype, radius)[::2]
        total = total + _ORACLE[k][0]
        segs += _ORACLE[k][1]
        s0 += n
    return total, segs


@pytest.mark.parametrize("ftype,radius", [(O.RT_FILTER_BOX, 0.5), (O.RT_FILTER_BOX, 4.0), (O.RT_FILTER_TENT, 1.0), (O.RT_FILTER_TENT, 0.5)])
def test_read_sample_dirs_is_the_numpy_statement(tracer, scenes, ftype, radius):
    load(tracer, scenes, "Scene1", "right_x1.3")
    cam = camera(rtb200.RtCamera, scenes, "Scene1", "right_x1.3")
    try:
        tracer.set_pixel_filter(ftype, radius)
        for sample in (0, 5, 1023, 0x80000005):
            assert np.array_equal(_bits(tracer.read_sample_dirs(sample)), _bits(ref.sample_dirs(cam, W, H, SEED, ftype, radius, sample)))
        tracer.set_pixel_filter(None)
        assert np.array_equal(_bits(tracer.read_sample_dirs(7)), _bits(tracer.read_ray_dirs()))
    finally:
        tracer.set_pixel_filter(None)


def test_filter_arguments_are_checked(tracer, scenes):
    load(tracer, scenes, "Scene1", "defaults")
    tracer.set_pixel_filter(O.RT_FILTER_TENT, 1.5)
    bad = [dict(type=3), dict(type=-1), dict(radius=0.0), dict(radius=-0.5), dict(radius=4.0001), dict(radius=float("nan")),
           dict(radius=float("inf"))]
    try:
        for kw in bad:
            with pytest.raises(rtb200.RtError):
                tracer.set_pixel_filter(rtb200.default_pixel_filter(**dict(dict(type=O.RT_FILTER_BOX), **kw)))
        f = rtb200.default_pixel_filter(type=O.RT_FILTER_BOX)
        f.reserved[1] = 1
        with pytest.raises(rtb200.RtError):
            tracer.set_pixel_filter(f)
        g = tracer.pixel_filter()
        assert (g.type, g.radius) == (O.RT_FILTER_TENT, 1.5)                       # unchanged by the refused calls
        tracer.set_pixel_filter(O.RT_FILTER_BOX, 4.0)
        assert tracer.pixel_filter().radius == 4.0
    finally:
        tracer.set_pixel_filter(None)
    g = tracer.pixel_filter()
    assert (g.type, g.radius) == (O.RT_FILTER_NONE, 0.5)


CASES = [(f, s, t, r) for f in AA_FORMS for s in SETS for t, r in FILTERS]


@pytest.mark.parametrize("form,name,ftype,radius", CASES)
def test_filtered_form_matches_oracle(tracer, oracle, scenes, form, name, ftype, radius):
    opts, key, calls, _ = FORMS[form]
    key = key or ("Scene_indirect" if name.startswith("bounces") else "Scene1")
    try:
        set_options(tracer, opts)
        load(tracer, scenes, key, name)
        tracer.set_pixel_filter(ftype, radius)
        for n in calls:
            tracer.render_spp(n)
        acc, n = tracer.read_accum()
        st = tracer.stats()
        trav = tracer.traversal_stats()
    finally:
        set_options(tracer, DEFAULT_OPTIONS)
        tracer.set_pixel_filter(None)
    want, segs = expected_filtered(oracle, scenes, key, name, calls, ftype, radius)
    assert n == sum(calls) and st.paths == W * H * sum(calls)
    assert st.segments == segs
    assert st.traced_segments == st.segments                      # every sample traced its own primary ray
    assert st.pipeline == O.RT_PIPELINE_REGEN
    assert close(acc[..., :3], want)
    if O.RT_OPT_ACCEL in opts:
        assert st.accel == opts[O.RT_OPT_ACCEL]
    if opts.get(O.RT_OPT_TRAVERSAL_STATS):
        assert trav.queries > 0 and trav.node_visits > 0


@pytest.mark.parametrize("ftype,radius", FILTERS)
def test_filtered_render_frame_matches_oracle(tracer, oracle, scenes, ftype, radius):
    """rt_render_frame's fused 1-spp frame (the pixel pool resolves the surface inside the render) and a 2-spp frame."""
    surf, owner = rtb200.host_surface(W, H)
    load(tracer, scenes, "Scene1", "defaults")
    try:
        tracer.set_pixel_filter(ftype, radius)
        for calls in ((1,), (1, 2)):
            surf[:] = 0
            tracer.render_frame(calls[-1], out=surf)
            acc, n = tracer.read_accum()
            want, segs = expected_filtered(oracle, scenes, "Scene1", "defaults", calls, ftype, radius)
            assert n == sum(calls) and tracer.stats().segments == segs
            assert close(acc[..., :3], want)
            assert np.array_equal(surf, oracle.resolve_argb8(acc, n)), calls
    finally:
        tracer.set_pixel_filter(None)
    del owner


def _render(t, scenes, key, name, calls, opts=None, f=None):
    try:
        set_options(t, opts or {})
        load(t, scenes, key, name)
        t.set_pixel_filter(f)
        for n in calls:
            t.render_spp(n)
        acc, n = t.read_accum()
        return acc, t.stats()
    finally:
        set_options(t, DEFAULT_OPTIONS)
        t.set_option(O.RT_OPT_BVH_SCHED, 0)
        t.set_pixel_filter(None)


@pytest.mark.parametrize("opts,key", [
    ({O.RT_OPT_PIPELINE: O.RT_PIPELINE_WAVEFRONT}, "Scene1"),
    ({O.RT_OPT_PIPELINE: O.RT_PIPELINE_STREAM, O.RT_OPT_ACCEL: O.RT_ACCEL_BVH}, "big"),
    ({O.RT_OPT_PIPELINE: O.RT_PIPELINE_AUTO, O.RT_OPT_ACCEL: O.RT_ACCEL_BVH, O.RT_OPT_BVH_SCHED: 1}, "big"),
])
def test_pipeline_requests_render_with_the_megakernel(tracer, scenes, opts, key):
    f = rtb200.default_pixel_filter(type=O.RT_FILTER_TENT, radius=1.0)
    calls = (9, 11)
    acc, st = _render(tracer, scenes, key, "defaults", calls, opts, f)
    mk, _ = _render(tracer, scenes, key, "defaults", calls, {k: v for k, v in opts.items() if k == O.RT_OPT_ACCEL}, f)
    assert st.pipeline == O.RT_PIPELINE_REGEN
    assert np.array_equal(_bits(acc), _bits(mk))
    assert st.traced_segments == st.segments


def test_none_restores_the_unfiltered_render_and_calls_split_freely(scenes):
    fresh, used = rtb200.PathTracer(0), rtb200.PathTracer(0)
    try:
        a, _ = _render(fresh, scenes, "Scene1", "defaults", SPLIT)
        load(used, scenes, "Scene1", "defaults")
        used.set_pixel_filter(O.RT_FILTER_BOX, 0.5)
        used.render_spp(3)
        used.set_pixel_filter(None)
        used.reset_accumulation()
        for n in SPLIT:
            used.render_spp(n)
        b, _ = used.read_accum()
        assert np.array_equal(_bits(a), _bits(b))
        # one call of n spp == n calls of 1 spp (pixel pool) with a filter
        f = rtb200.default_pixel_filter(type=O.RT_FILTER_TENT, radius=1.0)
        one, _ = _render(fresh, scenes, "Scene1", "defaults", (8,), None, f)
        many, _ = _render(fresh, scenes, "Scene1", "defaults", (1,) * 8, None, f)
        assert np.array_equal(_bits(one), _bits(many))
    finally:
        fresh.close(); used.close()


def test_shards_and_group_give_the_single_context_sum(tracer, scenes):
    import torch
    f = rtb200.default_pixel_filter(type=O.RT_FILTER_BOX, radius=0.5)
    single, _ = _render(tracer, scenes, "Scene1", "defaults", SPLIT, None, f)
    parts = []
    for rank in range(2):
        t = rtb200.PathTracer(0)
        try:
            load(t, scenes, "Scene1", "defaults")
            t.set_pixel_filter(f)
            t.set_shard(rank, 2)
            for n in SPLIT:
                t.render_spp(n)
            parts.append(t.read_accum())
        finally:
            t.close()
    assert parts[0][1] + parts[1][1] == sum(SPLIT)
    assert close(parts[0][0][..., :3] + parts[1][0][..., :3], single[..., :3])
    g = rtb200.TracerGroup(list(range(min(torch.cuda.device_count(), 2))))
    try:
        g.set_scene(scenes["Scene1"])
        g.set_camera(camera(rtb200.RtCamera, scenes, "Scene1", "defaults"))
        g.set_params(make_params(rtb200.default_params, "defaults", W, H))
        g.set_pixel_filter(f)
        assert all(m.pixel_filter().type == O.RT_FILTER_BOX for m in g.members)
        g.reset_accumulation()
        for n in SPLIT:
            g.render_spp(n)
        mean = g.read_denoised(rtb200.default_denoise_params(passes=0))
    finally:
        g.close()
    assert close(mean[..., :3], single[..., :3] / np.float32(sum(SPLIT)))


# ---- anti-aliasing itself -------------------------------------------------------------------------------------------
AW, AH, ASPP, GRID = 64, 48, 1024, 24


def _sphere_scene():
    o = np.zeros(1, rtb200.OBJECT_DTYPE)
    o[0]["type"] = O.RT_OBJ_SPHERE
    o[0]["pos"] = (0.13, -0.07, 0.9)
    o[0]["radius"] = 0.2
    o[0]["emissive"] = (1.0, 1.0, 1.0)
    return o


def _dark_params(factory):
    p = factory(width=AW, height=AH, mode=O.RT_MODE_PATH, max_bounces=0, seed_lo=SEED[0], seed_hi=SEED[1])
    for k in ("sky", "horizon", "ground", "sun"):
        for i in range(3):
            getattr(p, k)[i] = 0.0
    return p


def _coverage(oracle, objs, ftype, radius):
    """Filter-weighted coverage of every pixel's footprint from a GRID x GRID sub-pixel grid of oracle primary hits."""
    cam = OrcCamera(); cam.right[0] = 1; cam.up[1] = 1; cam.forward[2] = 1; cam.fov_deg = 55
    from temporal_reference import pose_of_camera
    _, u, v, f = pose_of_camera(cam, AW, AH)
    t = ((np.arange(GRID) + 0.5) / GRID * 2 - 1) * radius                         # midpoints on (-r, r)
    wt = np.ones(GRID) if ftype == O.RT_FILTER_BOX else (radius - np.abs(t))
    wt = wt / wt.sum()
    jx, jy = np.meshgrid(t.astype(np.float32), t.astype(np.float32))
    X = ((np.arange(AW, dtype=np.float32)[None, :, None, None] + jx) / np.float32(AW)) * np.float32(2) - np.float32(1)
    Y = ((np.arange(AH, dtype=np.float32)[:, None, None, None] + jy) / np.float32(AH)) * np.float32(2) - np.float32(1)
    c = [(u[k] * X + v[k] * Y) + f[k] for k in range(3)]
    ln = np.sqrt((c[0] * c[0] + c[1] * c[1]) + c[2] * c[2])
    d = np.stack([c[k] / ln for k in range(3)], -1).reshape(-1, 3).astype(np.float32)
    ids, _, _, _ = oracle.trace_rays(objs, np.zeros_like(d), d)
    hit = (ids >= 0).reshape(AH, AW, GRID, GRID)
    cov = np.clip(np.einsum("hwij,i,j->hw", hit.astype(np.float64), wt, wt), 0.0, 1.0)
    return cov, hit.all(axis=(2, 3)), ~hit.any(axis=(2, 3))


@pytest.mark.parametrize("ftype,radius", FILTERS)
def test_filter_anti_aliases_an_emissive_edge(tracer, oracle, ftype, radius):
    """Emission 1, black environment, max_bounces 0: every sample is exactly 1 on a hit and 0 on a miss, so a pixel's mean is the
    filter-weighted coverage of its footprint. Edge pixels lie within a binomial bound of the coverage; pixels whose footprint
    (and its neighbourhood) lies wholly on or off the sphere are exactly 1 or 0; without a filter every pixel is 0 or 1."""
    objs = _sphere_scene()
    tracer.set_scene(objs)
    tracer.set_camera(rtb200.default_camera())
    tracer.set_params(_dark_params(rtb200.default_params))
    try:
        tracer.reset_accumulation()
        tracer.render_spp(16)
        plain, n = tracer.read_accum()
        assert set(np.unique(plain[..., :3] / n).tolist()) == {0.0, 1.0}
        tracer.set_pixel_filter(ftype, radius)
        tracer.reset_accumulation()
        tracer.render_spp(ASPP)
        acc, n = tracer.read_accum()
    finally:
        tracer.set_pixel_filter(None)
    assert n == ASPP
    mean = acc[..., 0].astype(np.float64) / ASPP
    assert np.array_equal(acc[..., 0], acc[..., 1]) and np.array_equal(acc[..., 0], acc[..., 2])
    cov, full, empty = _coverage(oracle, objs, ftype, radius)
    reach = 2 * math.ceil(radius) + 3
    inside = ndimage.minimum_filter(full, size=reach, mode="nearest")
    outside = ndimage.minimum_filter(empty, size=reach, mode="nearest")
    assert inside.any() and outside.any()
    assert np.all(mean[inside] == 1.0) and np.all(mean[outside] == 0.0)
    edge = ~full & ~empty
    assert edge.sum() > 20
    bound = 5 * np.sqrt(np.maximum(cov * (1 - cov), 1e-3) / ASPP) + 3.0 / GRID
    assert np.all(np.abs(mean - cov)[edge] <= bound[edge]), np.abs(mean - cov)[edge].max()
    fractional = (mean > 0) & (mean < 1)
    assert fractional.sum() >= 0.5 * edge.sum()                    # the edge really is anti-aliased


# ---- the present paths and the frames that ignore the filter ----------------------------------------------------------
def test_denoise_and_temporal_on_a_filtered_buffer(tracer, scenes):
    tp = rtb200.default_temporal_params()
    load(tracer, scenes, "Scene1", "defaults")
    try:
        tracer.set_pixel_filter(O.RT_FILTER_TENT, 1.0)
        tracer.render_spp(4)
        out = tracer.denoise_rgba8(rtb200.default_denoise_params())
        assert out.any()
        tracer.read_temporal(tp)                                   # history of 4 samples
        tracer.reset_accumulation()
        tracer.render_spp(4)
        assert np.allclose(tracer.read_temporal(tp)[..., 3][tracer.read_aov()[0] >= 0], 8.0)   # the prior of the same pose counts
        tracer.reset_accumulation()
        tracer.set_pixel_filter(O.RT_FILTER_BOX, 0.5)              # a filter change drops the history
        tracer.render_spp(4)
        assert np.all(tracer.read_temporal(tp)[..., 3] == 4.0)
    finally:
        tracer.set_pixel_filter(None)
        tracer.reset_temporal()


@pytest.mark.parametrize("mode", ["preview", "blocks"])
def test_preview_and_block_filled_frames_ignore_the_filter(tracer, scenes, mode):
    def run(f):
        load(tracer, scenes, "Scene1", "defaults")
        if mode == "preview":
            tracer.set_params(make_params(rtb200.default_params, "defaults", W, H), mode=O.RT_MODE_PREVIEW)
        else:
            tracer.set_pixel_step(2, rtb200.reference_strip_columns(W))
            tracer.reset_accumulation()
        tracer.set_pixel_filter(f)
        for n in SHORT:
            tracer.render_spp(n)
        return tracer.read_accum()[0]
    try:
        a = run(None)
        b = run(rtb200.default_pixel_filter(type=O.RT_FILTER_BOX, radius=2.0))
    finally:
        tracer.set_pixel_filter(None)
        tracer.set_pixel_step(1, 0)
        tracer.set_params(make_params(rtb200.default_params, "defaults", W, H))
    assert np.array_equal(_bits(a), _bits(b))
