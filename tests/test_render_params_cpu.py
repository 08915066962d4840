"""CPU: the device functions (path_ends / scatter_segment / env_color, compiled for the host by tests/host_emu) against
the oracle at render parameters other than the reference's defaults: environment colours and sun direction, dissipation,
the surface offset eps, the path depth, the camera, and fields that must not change the image. The suite's other
radiance checks run at the defaults, where a hoisted constant or a misplaced field gives the same numbers.

PARAM_SETS is shared with tests/test_gpu_render_params.py, which runs the same sets through every render kernel form."""
import numpy as np
import pytest

import rtb200
from conftest import SEED
from oracle_py import OrcCamera
from test_device_logic_cpu import emu  # noqa: F401  (the session fixture)

RAD_RTOL, RAD_ATOL = 1e-5, 1e-6


def _unit(v):
    v = np.asarray(v, np.float64)
    return tuple(float(x) for x in (v / np.linalg.norm(v)).astype(np.float32))


# name -> (scene, rt_params fields, camera fields); each applies to the base below. sun_dir points from the sun into the
# scene (the disc is where dot(d, -sun_dir) > 0.99). Colours have three different channels, so a swapped channel shows.
PARAM_SETS = {
    "defaults": ("Scene1", {}, {}),
    "sun_near_horizon": ("Scene1", {"sun_dir": _unit([-0.12, -0.06, -1.0])}, {}),       # a disc in view, just above the horizon
    "sun_below_horizon": ("Scene1", {"sun_dir": _unit([0.3, 0.6, -0.7])}, {}),
    "sky": ("Scene1", {"sky": (0.9, 4.0, 11.0)}, {}),
    "horizon": ("Scene1", {"horizon": (6.0, 2.5, 0.7)}, {}),
    "ground": ("Scene1", {"ground": (0.5, 0.12, 0.03)}, {}),
    "sun": ("Scene1", {"sun": (900.0, 350.0, 60.0)}, {}),
    "dissipation_0.5": ("Scene1", {"dissipation": 0.5}, {}),
    "dissipation_1": ("Scene1", {"dissipation": 1.0}, {}),
    "eps_1e-3": ("Scene1", {"eps": 1e-3}, {}),                     # larger than the default: accelerator margins must grow
    "eps_1e-7": ("Scene1", {"eps": 1e-7}, {}),
    "bounces_-3": ("Scene_indirect", {"max_bounces": -3}, {}),      # MAXBOUNCES = max(MAXBOUNCES, 0)
    "bounces_1": ("Scene_indirect", {"max_bounces": 1}, {}),
    "bounces_3": ("Scene_indirect", {"max_bounces": 3}, {}),
    "bounces_60": ("Scene_indirect", {"max_bounces": 60}, {}),      # the deepest path the bounce-round pipelines take
    "bounces_61": ("Scene_indirect", {"max_bounces": 61}, {}),
    "fov_20": ("Scene1", {}, {"fov_deg": 20}),
    "fov_120": ("Scene1", {}, {"fov_deg": 120}),
    "right_x1.3": ("Scene1", {}, {"right": (1.3, 0.0, 0.0)}),      # the basis is used as given, never re-orthonormalised
    "selected_id": ("Scene1", {"selected_id": 5}, {}),              # preview-mode highlight only
    "seed_hi_max": ("Scene1", {"seed_lo": 0x9E3779B9, "seed_hi": 0xFFFFFFFF}, {}),
}
ENV_SETS = ["sun_near_horizon", "sun_below_horizon", "sky", "horizon", "ground", "sun"]


def make_params(factory, name, w, h):
    """factory: rtb200.default_params or Oracle.default_params. Path mode, 8 bounces and the suite's seed, then the set."""
    p = factory(width=w, height=h, mode=rtb200.RT_MODE_PATH, max_bounces=8, seed_lo=SEED[0], seed_hi=SEED[1])
    for k, v in PARAM_SETS[name][1].items():
        if isinstance(v, tuple):
            for i, x in enumerate(v):
                getattr(p, k)[i] = x
        else:
            setattr(p, k, v)
    return p


def make_cam(cls, name):
    c = cls()
    c.right[0] = 1; c.up[1] = 1; c.forward[2] = 1; c.fov_deg = 55
    for k, v in PARAM_SETS[name][2].items():
        if isinstance(v, tuple):
            for i, x in enumerate(v):
                getattr(c, k)[i] = x
        else:
            setattr(c, k, v)
    return c


@pytest.mark.parametrize("accel", [0, 1, 2])                       # brute force, binary BVH, flat two-level accelerator
@pytest.mark.parametrize("name", list(PARAM_SETS))
def test_device_functions_match_oracle_at_render_parameters(emu, oracle, scenes, name, accel):  # noqa: F811
    w, h, s0, n = 47, 29, 5, 3
    objs = scenes[PARAM_SETS[name][0]]
    par = make_params(rtb200.default_params, name, w, h)
    par.max_bounces = max(par.max_bounces, 0)                      # what rt_set_params stores; the frame constants take it from there
    got, segs, _ = emu(objs, make_cam(rtb200.RtCamera, name), par, accel, s0, n)
    assert segs >= 0, "accelerator not usable for this scene"
    want, _, want_segs = oracle.render(objs, make_cam(OrcCamera, name), make_params(oracle.default_params, name, w, h), s0, n)
    assert segs == want_segs
    assert np.allclose(got, want, rtol=RAD_RTOL, atol=RAD_ATOL)


def env_reference(p, dirs):
    """GetEnvironmentColor (Raytracer.cpp:77-89) in float64 from the float32 inputs; also returns the sun-disc decision and
    the float64 dot product it is made from."""
    d = np.asarray(dirs, np.float64)
    sky, hor, gnd, sun = (np.array(getattr(p, k)[:], np.float64) for k in ("sky", "horizon", "ground", "sun"))
    sdot = d @ -np.array(p.sun_dir[:], np.float64)
    disc = sdot > 0.99
    up = d[:, 1:2]
    lerp = lambda a, b, t: a * (1 - t) + b * t
    above = lerp(lerp(hor, sky, np.abs(up) ** 0.1), sky * 0.1, up)
    below = lerp(hor, gnd, np.abs(up) ** 0.05)
    c = np.where(up > 0, above, below) + np.where(disc[:, None], sun, 0.0)
    return c, disc, sdot


def env_directions(p):
    """Random unit directions, directions clustered around the sun disc's rim, and the axes and horizon."""
    rng = np.random.default_rng(17)
    r = rng.normal(size=(4000, 3))
    s = -np.array(p.sun_dir[:], np.float64)
    a = np.cross(s, [0.0, 0.0, 1.0] if abs(s[2]) < 0.9 else [1.0, 0.0, 0.0]); a /= np.linalg.norm(a)
    b = np.cross(s, a)
    ang = rng.uniform(0, 2 * np.pi, 4000)
    cos_t = rng.uniform(0.985, 0.995, 4000)                        # across the 0.99 rim
    sin_t = np.sqrt(1 - cos_t ** 2)
    rim = cos_t[:, None] * s + sin_t[:, None] * (np.cos(ang)[:, None] * a + np.sin(ang)[:, None] * b)
    axes = [[0, 1, 0], [0, -1, 0], [1, 0, 0], [0, 0, 1], [0.6, 0, 0.8], [0, 1e-4, 1], [0, -1e-4, 1]]
    d = np.concatenate([r, rim, np.array(axes, np.float64)])
    return (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)


def env_cameras(p):
    """Cameras whose pixel rays cover the sky, the ground, the horizon and the sun disc's rim (forward, fov)."""
    sun = -np.array(p.sun_dir[:], np.float64)
    return [((0.0, 0.0, 1.0), 120), ((0.0, 0.9, 0.3), 120), ((0.2, -0.9, 0.4), 120), ((0.9, 0.02, -0.4), 90), (tuple(sun), 30)]


def look_camera(cls, forward, fov):
    f = np.asarray(forward, np.float64); f /= np.linalg.norm(f)
    r = np.cross([0.0, 1.0, 0.0], f); r /= np.linalg.norm(r)       # the default basis: right = up x forward
    u = np.cross(f, r)
    c = cls()
    for k, v in (("right", r), ("up", u), ("forward", f)):
        for i in range(3):
            getattr(c, k)[i] = float(np.float32(v[i]))
    c.fov_deg = fov
    return c


@pytest.mark.parametrize("name", ENV_SETS)
def test_env_color_matches_float64_statement(emu, oracle, name):  # noqa: F811
    """A path whose primary ray misses is GetEnvironmentColor of the pixel's ray: one sample in an empty scene gives the device
    function on every ray of a camera, whose directions the oracle states exactly."""
    w, h = 64, 48
    p = make_params(rtb200.default_params, name, w, h)
    got, dirs = [], []
    for fwd, fov in env_cameras(p):
        out, segs, _ = emu(np.zeros(0, rtb200.OBJECT_DTYPE), look_camera(rtb200.RtCamera, fwd, fov), p, 0, 0, 1)
        assert segs == w * h
        got.append(out.reshape(-1, 3)); dirs.append(oracle.ray_dirs(look_camera(OrcCamera, fwd, fov), w, h).reshape(-1, 3))
    out, dirs = np.concatenate(got), np.concatenate(dirs)
    want, disc, sdot = env_reference(p, dirs)
    assert disc.sum() > 200 and (~disc).sum() > 200 and (dirs[:, 1] < 0).sum() > 2000    # sky, ground and both sides of the rim
    clear = np.abs(sdot - 0.99) > 1e-6                             # the float32 dot may land on either side of the rim
    assert clear.sum() > len(dirs) - 20
    assert np.allclose(out[clear], want[clear], rtol=2e-6, atol=1e-6)
    sun = np.array(p.sun[:], np.float32)
    got_disc = np.all(out >= sun * np.float32(0.999), axis=1)      # the disc adds the sun colour, far above the sky's
    assert np.array_equal(got_disc[clear], disc[clear])
