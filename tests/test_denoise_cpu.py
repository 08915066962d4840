"""CPU: the denoised resolve's filter (csrc/rt_denoise.cuh: tap weight and combine, shared with the CUDA kernels of rt_denoise.cu)
compiled for the host through tests/host_emu/cuda_shim.h, against the float32 numpy reference (tests/denoise_reference.py) on
emulated renders and guides; and the C-ABI additions (header declarations, struct layout, defaults)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import rtb200
from conftest import ROOT, SEED
import denoise_reference as ref

EMU_DIR = os.path.join(ROOT, "tests", "host_emu")
CSRC = os.path.join(ROOT, "software-raytracer_b200", "csrc")


@pytest.fixture(scope="session")
def dn_emu(tmp_path_factory):
    """g++ build of tests/host_emu/denoise_emu.cpp (the filter's passes as host loops over rt_denoise.cuh) into a temporary library."""
    so = str(tmp_path_factory.mktemp("denoise_emu") / "libdenoise_emu.so")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-o", so, os.path.join(EMU_DIR, "denoise_emu.cpp")])
    lib = C.CDLL(so)
    lib.emu_denoise.argtypes = [C.c_void_p, C.c_uint, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_void_p]

    def run(accum, samples, ids, nt, passes, normal_power, sigma_color, sigma_depth):
        h, w = ids.shape
        accum = np.ascontiguousarray(accum, np.float32); nt = np.ascontiguousarray(nt, np.float32); ids = np.ascontiguousarray(ids, np.int32)
        out = np.zeros((h, w, 4), np.float32)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        lib.emu_denoise(p(accum), samples, p(nt), p(ids), w, h, passes, normal_power.bit_length() - 1, sigma_color, sigma_depth, p(out))
        return out
    return run


@pytest.fixture(scope="session")
def renders(scenes):
    """Emulated noisy sums and primary-hit guides at 97 x 61 (odd sizes), depth 8: Scene1, Scene_indirect and a heightfield mesh."""
    from test_device_logic_cpu import build_emu
    from rtb200.scenes import heightfield_mesh, mesh_scene
    lib = C.CDLL(build_emu())
    lib.emu_render.restype = C.c_longlong
    lib.emu_render_mesh.restype = C.c_longlong
    w, h = 97, 61
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    out = {}
    cases = [("Scene1", scenes["Scene1"], None), ("Scene_indirect", scenes["Scene_indirect"], None)]
    v, tr = heightfield_mesh(24, 16, seed=3)
    cases.append(("mesh", mesh_scene(), (np.ascontiguousarray(v, np.float32).reshape(-1, 3), np.ascontiguousarray(tr, np.int32).reshape(-1, 3))))
    for name, objs, mesh in cases:
        objs = np.ascontiguousarray(objs, rtb200.OBJECT_DTYPE)
        cam = rtb200.default_camera(55)
        if mesh is not None:
            cam.pos[1] = 1.5; cam.pos[2] = -1.0
        par = rtb200.default_params(width=w, height=h, mode=0, max_bounces=8, seed_lo=SEED[0], seed_hi=SEED[1])
        for spp, s0 in ((1, 0), (4, 0), (64, 1000)):
            if spp == 64 and name != "Scene1":
                continue
            rad = np.zeros((h, w, 3), np.float32)
            ids = np.zeros((h, w), np.int32); t = np.zeros((h, w), np.float32)
            nrm = np.zeros((h, w, 3), np.float32); pt = np.zeros((h, w, 3), np.float32)
            if mesh is None:
                lib.emu_render(p(objs), len(objs), C.byref(cam), C.byref(par), 0, C.c_uint32(s0), spp, p(rad), p(ids), p(t), p(nrm), p(pt))
            else:
                mv, mt = mesh
                lib.emu_render_mesh(p(objs), len(objs), C.byref(cam), C.byref(par), 0, C.c_uint32(s0), spp, p(rad), p(ids), p(t), p(nrm), p(pt),
                                    p(mv), len(mv), p(mt), len(mt), 0)
            accum = np.concatenate([rad, np.zeros((h, w, 1), np.float32)], -1)
            nt = np.concatenate([nrm, t[..., None]], -1)
            out[(name, spp)] = (accum, ids, nt)
    return out


PARAMS = [(128, 1.0, 1.0), (32, 0.5, 2.0), (256, 2.0, 0.25), (1, 1.0, 1.0)]


@pytest.mark.parametrize("scene", ["Scene1", "Scene_indirect", "mesh"])
@pytest.mark.parametrize("passes", [1, 3, 5])
@pytest.mark.parametrize("spp", [1, 4])
def test_host_build_of_the_filter_matches_the_numpy_reference(dn_emu, renders, scene, passes, spp):
    accum, ids, nt = renders[(scene, spp)]
    hit = ids >= 0
    assert hit.mean() > 0.2
    for power, sc, sz in PARAMS:
        got = dn_emu(accum, spp, ids, nt, passes, power, sc, sz)
        want = ref.denoise(accum, spp, ids, nt, passes, power, sc, sz)
        np.testing.assert_allclose(got[..., :3], want, rtol=1e-5, atol=1e-6 * float(want.max()), err_msg=str((power, sc, sz)))
        # the stored luminance is the one the next pass reads
        np.testing.assert_allclose(got[..., 3], ref.luma(got[..., :3]), rtol=1e-6, atol=0)
        # sky pixels are the plain mean, bit for bit
        mean = ref.mean_of(accum, spp)
        assert np.array_equal(got[~hit][:, :3].view(np.uint32), mean[~hit].view(np.uint32))


def test_host_build_leaves_constant_objects_unchanged(dn_emu, renders):
    """One colour per object id: no colour crosses an id, so every pixel keeps its value (to rounding)."""
    _, ids, nt = renders[("Scene1", 4)]
    rng = np.random.default_rng(3)
    pal = rng.uniform(0.0, 50.0, (int(ids.max()) + 2, 3)).astype(np.float32)
    mean = pal[ids + 1]
    accum = np.concatenate([mean, np.zeros(ids.shape + (1,), np.float32)], -1)
    got = dn_emu(accum, 0, ids, nt, 5, 128, 1.0, 1.0)
    np.testing.assert_allclose(got[..., :3], mean, rtol=1e-6, atol=0)


def test_filter_reduces_noise_on_emulated_renders(renders):
    """The reference filter moves 1- and 4-spp Scene1 renders towards a 64-spp render of other samples (a check of the definition
    itself; the GPU suite measures the same against 4096 spp)."""
    a64, _, _ = renders[("Scene1", 64)]
    gt = ref.mean_of(a64, 64)
    for spp in (1, 4):
        a, ids, nt = renders[("Scene1", spp)]
        raw = ref.psnr(ref.mean_of(a, spp), gt)
        den = ref.psnr(ref.denoise(a, spp, ids, nt), gt)
        print("Scene1 97x61, %d spp: raw %.2f dB, denoised %.2f dB (against 64 spp of other samples)" % (spp, raw, den))
        assert den > raw + 1.0


def test_denoise_abi_declarations():
    from test_capi_cpu import header_functions
    names = header_functions()
    for n in ("rt_default_denoise_params", "rt_denoise_rgba8", "rt_read_denoised"):
        assert n in names and n in rtb200.EXPORTS
    assert C.sizeof(rtb200.RtDenoiseParams) == 16
    lib = rtb200.load_library()
    for n in ("rt_default_denoise_params", "rt_denoise_rgba8", "rt_read_denoised"):
        assert hasattr(lib, n)
    p = rtb200.default_denoise_params()
    assert (p.passes, p.normal_power) == (5, 128) and p.sigma_color > 0 and p.sigma_depth > 0
    q = rtb200.default_denoise_params(passes=2, sigma_color=0.5)
    assert (q.passes, q.normal_power, q.sigma_color) == (2, 128, 0.5)


def test_denoise_calls_refuse_without_a_device_or_context():
    """No context (NULL): RT_ERR_INVALID, never a CPU path."""
    lib = rtb200.load_library()
    out = np.zeros(16, np.uint32)
    assert lib.rt_denoise_rgba8(None, None, out.ctypes.data_as(C.c_void_p), 16, 1) == rtb200.RT_ERR_INVALID
    assert lib.rt_read_denoised(None, None, out.ctypes.data_as(C.c_void_p)) == rtb200.RT_ERR_INVALID
