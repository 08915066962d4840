"""GPU (B200): the packed FP32x2 arithmetic (add / sub / mul / fma.rn.f32x2) of the flat accelerator's culls.

The packed ops must give the bits of the scalar .rn ops they replace, and the flat accelerator, whose cull records are staged as
packed pairs, must select exactly what brute force selects - also with an odd number of level-1 single spheres, where the last
pair has no partner."""
import numpy as np
import pytest

import rtb200

pytestmark = pytest.mark.gpu


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def test_packed_pair_ops_are_exact_on_device(tracer):
    """add / sub / mul / fma.rn.f32x2 == the scalar .rn ops on each half, bit for bit on 2^26 operand sets (subnormals, +-0,
    +-inf, values near overflow, mixed exponents, any bit pattern; two NaNs count as equal)."""
    assert tracer.selftest(2) == 0


def singles_scene(n_big, seed):
    """Small spheres in tight groups (the builder clusters them) plus n_big large ones and the ground sphere, which stay level-1
    singles: n_big + 1 of them, so n_big = 1..5 gives both odd and even counts."""
    rng = np.random.default_rng(seed)
    n_small = 40
    n = n_small + n_big + 1
    o = np.zeros(n, rtb200.OBJECT_DTYPE)
    o["type"] = 1
    centres = rng.uniform([-6, 0, 6], [6, 4, 18], (5, 3))
    o["pos"][:n_small] = (centres[np.arange(n_small) % 5] + rng.uniform(-0.6, 0.6, (n_small, 3))).astype(np.float32)
    o["radius"][:n_small] = rng.uniform(0.05, 0.3, n_small).astype(np.float32)
    o["pos"][n_small:n - 1] = rng.uniform([-8, 0, 8], [8, 6, 20], (n_big, 3)).astype(np.float32)
    o["radius"][n_small:n - 1] = rng.uniform(2.0, 4.0, n_big).astype(np.float32)
    o["base"] = rng.uniform(0.1, 0.9, (n, 3)).astype(np.float32); o["spec_color"] = 1
    o["spec_amount"][::3] = 1; o["smoothness"][::3] = 0.9
    o["emissive"][::9] = 15
    o["pos"][n - 1] = [0, -500, 20]; o["radius"][n - 1] = 500
    return o


@pytest.mark.parametrize("n_big", [1, 2, 3, 4, 5])
def test_flat_accel_with_odd_and_even_singles_is_bit_identical(tracer, n_big):
    o = singles_scene(n_big, 100 + n_big)
    cam = rtb200.default_camera(60); cam.pos[1] = 2.0; cam.pos[2] = -4.0
    res = {}
    try:
        for accel in (rtb200.RT_ACCEL_FLAT, rtb200.RT_ACCEL_BRUTE):
            tracer.set_option(rtb200.RT_OPT_ACCEL, accel)
            tracer.set_scene(o)
            tracer.set_camera(cam)
            tracer.set_params(rtb200.default_params(width=256, height=144, mode=rtb200.RT_MODE_PATH, max_bounces=6, seed_lo=7))
            tracer.reset_accumulation()
            aov = tracer.read_aov()
            tracer.render_spp(8)
            st = tracer.stats()
            assert st.accel == accel
            res[accel] = (aov, tracer.read_accum()[0], st.segments)
    finally:
        tracer.set_option(rtb200.RT_OPT_ACCEL, rtb200.RT_ACCEL_AUTO)
    a, b = res[rtb200.RT_ACCEL_FLAT], res[rtb200.RT_ACCEL_BRUTE]
    assert np.array_equal(a[0][0], b[0][0])
    for x, y in zip(a[0][1:], b[0][1:]):
        assert np.array_equal(bits(x), bits(y))
    assert np.array_equal(bits(a[1]), bits(b[1])) and a[2] == b[2]
