"""rtb200 - thin ctypes binding of librt_b200.so (include/rt_b200.h).

Used by tests/, bench.py and __graft_entry__.py. It only marshals arguments: every compute
call goes through the C-ABI into the CUDA kernels, and a missing library or GPU raises
(there is no CPU path in the product).
"""
import ctypes as C
import os

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
PRODUCT_DIR = os.path.normpath(os.path.join(_PKG, "..", ".."))
REPO_ROOT = os.path.normpath(os.path.join(PRODUCT_DIR, ".."))
LIB_PATH = os.path.join(PRODUCT_DIR, "lib", "librt_b200.so")

RT_OK, RT_ERR_INVALID, RT_ERR_CUDA, RT_ERR_IO, RT_ERR_PARSE, RT_ERR_NOMEM = 0, -1, -2, -3, -4, -5
RT_OBJ_NONE, RT_OBJ_SPHERE, RT_OBJ_CUBE, RT_OBJ_MESH = 0, 1, 2, 3
RT_MODE_PATH, RT_MODE_PREVIEW = 0, 1
RT_OPT_PIPELINE, RT_OPT_ACCEL, RT_OPT_BVH_THRESHOLD, RT_OPT_BVH_SCHED, RT_OPT_BVH_WAIT_K, RT_OPT_BVH_LEAF, RT_OPT_PRIMARY_REUSE = 1, 2, 3, 4, 5, 6, 7
RT_OPT_WF_REFILL, RT_OPT_WF_NODE_MIN, RT_OPT_POOL_TILES, RT_OPT_FLAT_COOP, RT_OPT_BVH_WIDE, RT_OPT_WF_WAVE_MPATHS = 8, 9, 10, 11, 12, 13
RT_OPT_TRAVERSAL_STATS = 14
RT_OPT_BVH_QUANT = 15
RT_MAX_PEERS = 16
RT_PIPELINE_AUTO, RT_PIPELINE_REGEN, RT_PIPELINE_WAVEFRONT, RT_PIPELINE_STREAM = 0, 1, 2, 3
RT_ACCEL_AUTO, RT_ACCEL_BRUTE, RT_ACCEL_BVH, RT_ACCEL_FLAT = 0, 1, 2, 3


class RtObject(C.Structure):
    _fields_ = [("type", C.c_int32), ("pos", C.c_float * 3), ("radius", C.c_float), ("half", C.c_float * 3),
                ("base", C.c_float * 3), ("emissive", C.c_float * 3), ("spec_color", C.c_float * 3),
                ("smoothness", C.c_float), ("spec_amount", C.c_float)]


class RtCamera(C.Structure):
    _fields_ = [("pos", C.c_float * 3), ("right", C.c_float * 3), ("up", C.c_float * 3), ("forward", C.c_float * 3),
                ("fov_deg", C.c_int32)]


class RtParams(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("max_bounces", C.c_int32), ("mode", C.c_int32),
                ("selected_id", C.c_int32), ("sun_dir", C.c_float * 3), ("sky", C.c_float * 3),
                ("horizon", C.c_float * 3), ("ground", C.c_float * 3), ("sun", C.c_float * 3),
                ("dissipation", C.c_float), ("eps", C.c_float), ("seed_lo", C.c_uint32), ("seed_hi", C.c_uint32)]


class RtStats(C.Structure):
    _fields_ = [("paths", C.c_uint64), ("segments", C.c_uint64), ("samples", C.c_uint32), ("n_objects", C.c_uint32),
                ("last_render_ms", C.c_float), ("last_resolve_ms", C.c_float), ("pipeline", C.c_int32),
                ("accel", C.c_int32), ("sm_count", C.c_int32), ("reserved", C.c_int32),
                ("total_paths", C.c_uint64), ("total_segments", C.c_uint64),
                ("traced_segments", C.c_uint64), ("total_traced_segments", C.c_uint64)]


class RtDenoiseParams(C.Structure):
    _fields_ = [("passes", C.c_int32), ("normal_power", C.c_int32), ("sigma_color", C.c_float), ("sigma_depth", C.c_float)]


class RtTemporalParams(C.Structure):
    _fields_ = [("max_history", C.c_int32), ("tau_depth", C.c_float), ("tau_normal", C.c_float), ("reserved", C.c_int32)]


class RtTraversalStats(C.Structure):
    _fields_ = [("queries", C.c_uint64), ("node_visits", C.c_uint64), ("prim_tests", C.c_uint64),
                ("sphere_tests", C.c_uint64), ("cube_tests", C.c_uint64), ("tri_tests", C.c_uint64),
                ("node_bytes", C.c_uint32), ("reserved", C.c_uint32)]


OBJECT_DTYPE = np.dtype([("type", "<i4"), ("pos", "<f4", 3), ("radius", "<f4"), ("half", "<f4", 3),
                         ("base", "<f4", 3), ("emissive", "<f4", 3), ("spec_color", "<f4", 3),
                         ("smoothness", "<f4"), ("spec_amount", "<f4")])
assert OBJECT_DTYPE.itemsize == C.sizeof(RtObject) == 76

# every symbol include/rt_b200.h declares
EXPORTS = [
    "rt_create", "rt_destroy", "rt_render_frame", "rt_last_error", "rt_abi_version", "rt_load_scene", "rt_save_scene", "rt_set_scene",
    "rt_get_scene", "rt_default_params", "rt_default_camera", "rt_rotate_camera", "rt_set_camera", "rt_set_params",
    "rt_set_option", "rt_set_shard", "rt_shard_range", "rt_reset_accumulation", "rt_render_spp", "rt_resolve_rgba8", "rt_pick",
    "rt_read_accum", "rt_read_aov", "rt_read_ray_dirs", "rt_trace_rays", "rt_env_color", "rt_philox_block",
    "rt_scene_file_read", "rt_scene_file_read_names", "rt_scene_file_write", "rt_object_name", "rt_set_object_name", "rt_scene_name",
    "rt_write_accum", "rt_selftest", "rt_get_stats", "rt_accum_device_ptr", "rt_set_stream", "rt_sync", "rt_set_sample_count", "rt_resolve_device",
    "rt_host_alloc", "rt_host_free", "rt_set_mesh", "rt_load_mesh_obj", "rt_get_mesh_info", "rt_set_pixel_step", "rt_reference_pixel_step", "rt_reference_strip_columns",
    "rt_argb_device_ptr", "rt_ipc_export", "rt_ipc_open", "rt_ipc_close", "rt_resolve_fused", "rt_read_surface",
    "rt_get_traversal_stats", "rt_exchange_setup", "rt_exchange_resolve",
    "rt_create_multi", "rt_group_destroy", "rt_group_size", "rt_group_ctx", "rt_group_last_error", "rt_group_set_scene", "rt_group_load_scene",
    "rt_group_set_mesh", "rt_group_set_camera", "rt_group_set_params", "rt_group_set_option", "rt_group_reset_accumulation",
    "rt_group_render_spp", "rt_group_resolve_rgba8", "rt_group_get_stats",
    "rt_default_denoise_params", "rt_denoise_rgba8", "rt_read_denoised",
    "rt_default_temporal_params", "rt_temporal_rgba8", "rt_read_temporal", "rt_reset_temporal",
    "rt_group_denoise_rgba8", "rt_group_read_denoised", "rt_group_temporal_rgba8", "rt_group_read_temporal", "rt_group_reset_temporal",
]


class RtError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("rt_b200 error %d: %s" % (code, msg))
        self.code = code


_lib = None


def load_library(path=None):
    """dlopen the product library; raises if it was not built (no fallback)."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or os.environ.get("RTB200_LIB") or LIB_PATH     # RTB200_LIB: A/B builds of the same library (benchmarks)
    if not os.path.exists(p):
        raise FileNotFoundError("%s not built: run `make -C %s` (or __graft_entry__.build())" % (p, PRODUCT_DIR))
    lib = C.CDLL(p)
    lib.rt_last_error.restype = C.c_char_p
    lib.rt_last_error.argtypes = [C.c_void_p]
    lib.rt_accum_device_ptr.restype = C.c_void_p
    lib.rt_accum_device_ptr.argtypes = [C.c_void_p]
    lib.rt_argb_device_ptr.restype = C.c_void_p
    lib.rt_argb_device_ptr.argtypes = [C.c_void_p]
    lib.rt_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    for name in EXPORTS:
        fn = getattr(lib, name)
        if name in ("rt_host_alloc", "rt_host_free", "rt_last_error", "rt_accum_device_ptr", "rt_argb_device_ptr", "rt_create", "rt_default_params", "rt_default_camera",
                    "rt_default_denoise_params", "rt_default_temporal_params", "rt_rotate_camera", "rt_abi_version", "rt_object_name", "rt_scene_name", "rt_group_ctx", "rt_group_last_error"):
            continue
        fn.restype = C.c_int
    lib.rt_group_ctx.restype = C.c_void_p
    lib.rt_group_ctx.argtypes = [C.c_void_p, C.c_int]
    lib.rt_group_last_error.restype = C.c_char_p
    lib.rt_group_last_error.argtypes = [C.c_void_p]
    lib.rt_create_multi.argtypes = [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]
    for name in ("rt_group_destroy", "rt_group_size", "rt_group_reset_accumulation", "rt_group_reset_temporal"):
        getattr(lib, name).argtypes = [C.c_void_p]
    lib.rt_group_denoise_rgba8.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    lib.rt_group_read_denoised.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.rt_group_temporal_rgba8.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    lib.rt_group_read_temporal.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.rt_object_name.restype = C.c_char_p
    lib.rt_object_name.argtypes = [C.c_void_p, C.c_int]
    lib.rt_scene_name.restype = C.c_char_p
    lib.rt_scene_name.argtypes = [C.c_void_p]
    lib.rt_host_alloc.restype = C.c_void_p
    lib.rt_host_alloc.argtypes = [C.c_size_t]
    lib.rt_host_free.restype = None
    lib.rt_host_free.argtypes = [C.c_void_p]
    lib.rt_default_params.restype = None
    lib.rt_default_camera.restype = None
    lib.rt_default_denoise_params.restype = None
    lib.rt_default_temporal_params.restype = None
    lib.rt_rotate_camera.restype = None
    if path is None:
        _lib = lib
    return lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def default_params(**kw):
    p = RtParams()
    load_library().rt_default_params(C.byref(p))
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def default_denoise_params(**kw):
    """rt_default_denoise_params, with any field overridden by keyword (passes, normal_power, sigma_color, sigma_depth)."""
    p = RtDenoiseParams()
    load_library().rt_default_denoise_params(C.byref(p))
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def default_temporal_params(**kw):
    """rt_default_temporal_params, with any field overridden by keyword (max_history, tau_depth, tau_normal)."""
    p = RtTemporalParams()
    load_library().rt_default_temporal_params(C.byref(p))
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def default_camera(fov=55):
    c = RtCamera()
    load_library().rt_default_camera(C.byref(c))
    c.fov_deg = fov
    return c


def rotate_camera(cam, angle, axis):
    ax = (C.c_float * 3)(*[float(v) for v in axis])
    load_library().rt_rotate_camera(C.byref(cam), C.c_float(angle), ax)


def scene_file_read(path):
    """Host-only: parse a scene file -> (status, objects parsed, error message)."""
    lib = load_library()
    n = C.c_int(0)
    err = C.create_string_buffer(512)
    rc = lib.rt_scene_file_read(str(path).encode(), None, 0, C.byref(n), err, 512)
    out = np.zeros(n.value, OBJECT_DTYPE)
    if n.value:
        lib.rt_scene_file_read(str(path).encode(), _p(out), n.value, C.byref(n), err, 512)
    return rc, out, err.value.decode()


def scene_file_names(path):
    lib = load_library()
    need = lib.rt_scene_file_read_names(str(path).encode(), None, 0, None, 0)
    buf = C.create_string_buffer(max(need, 1)); sn = C.create_string_buffer(1024)
    lib.rt_scene_file_read_names(str(path).encode(), buf, need, sn, 1024)
    names = buf.raw[:need].split(b"\0")[:-1] if need else []
    return [n.decode() for n in names], sn.value.decode()


def scene_file_write(path, objs, names=None, scene_name=""):
    lib = load_library()
    objs = np.ascontiguousarray(objs, OBJECT_DTYPE)
    arr = None
    if names is not None:
        arr = (C.c_char_p * len(objs))(*[n.encode() for n in names])
    return lib.rt_scene_file_write(str(path).encode(), scene_name.encode(), _p(objs), arr, len(objs))


def host_surface(width, height):
    """A page-locked (height, width) uint32 array for resolve_rgba8 / read_surface; keep the returned owner alive."""
    lib = load_library()
    ptr = lib.rt_host_alloc(width * height * 4)
    if not ptr:
        raise MemoryError("rt_host_alloc failed")

    class _Owner:
        def __del__(self):
            lib.rt_host_free(ptr)
    arr = np.ctypeslib.as_array((C.c_uint32 * (width * height)).from_address(ptr)).reshape(height, width)
    return arr, _Owner()


def reference_pixel_step(screen_scale, progressive_scaler=1.0):
    lib = load_library()
    lib.rt_reference_pixel_step.argtypes = [C.c_float, C.c_float]
    return lib.rt_reference_pixel_step(screen_scale, progressive_scaler)


def reference_strip_columns(width):
    return load_library().rt_reference_strip_columns(width)


def shard_range(spp, rank, world, next_sample=0):
    first, count = C.c_uint32(0), C.c_int(0)
    rc = load_library().rt_shard_range(spp, rank, world, C.c_uint32(next_sample), C.byref(first), C.byref(count))
    if rc != RT_OK:
        raise RtError(rc, "rt_shard_range: bad arguments")
    return first.value, count.value


class PathTracer:
    """One rt_ctx. Mirrors the call sequence main() makes into the hot path (SURVEY.md 3.3)."""

    def __init__(self, device=0, _borrowed=None):
        self.lib = load_library()
        self.owned = _borrowed is None
        if _borrowed is not None:                  # a member of a TracerGroup: the group owns the handle
            self.h = C.c_void_p(_borrowed)
        else:
            h = C.c_void_p()
            rc = self.lib.rt_create(device, C.byref(h))
            if rc != RT_OK:
                raise RtError(rc, (self.lib.rt_last_error(None) or b"").decode())
            self.h = h
        self.params = default_params()
        self.camera = default_camera()

    def close(self):
        if getattr(self, "h", None):
            if self.owned:
                self.lib.rt_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc < 0:
            raise RtError(rc, (self.lib.rt_last_error(self.h) or b"").decode())
        return rc

    # scene
    def load_scene(self, path):
        return self._chk(self.lib.rt_load_scene(self.h, str(path).encode()))

    def save_scene(self, path):
        return self._chk(self.lib.rt_save_scene(self.h, str(path).encode()))

    def set_scene(self, objs):
        objs = np.ascontiguousarray(objs, OBJECT_DTYPE)
        return self._chk(self.lib.rt_set_scene(self.h, _p(objs), len(objs)))

    def set_mesh(self, object_index, vertices, triangles):
        """mesh extension: attach triangles (object-space float32 xyz, int32 index triples) to an RT_OBJ_MESH object."""
        v = np.ascontiguousarray(vertices, np.float32).reshape(-1, 3)
        t = np.ascontiguousarray(triangles, np.int32).reshape(-1, 3)
        return self._chk(self.lib.rt_set_mesh(self.h, object_index, _p(v), len(v), _p(t), len(t)))

    def load_mesh_obj(self, object_index, path):
        return self._chk(self.lib.rt_load_mesh_obj(self.h, object_index, str(path).encode()))

    def mesh_info(self, object_index):
        nv, nt = C.c_int(0), C.c_int(0)
        self._chk(self.lib.rt_get_mesh_info(self.h, object_index, C.byref(nv), C.byref(nt)))
        return nv.value, nt.value

    def get_scene(self):
        n = self._chk(self.lib.rt_get_scene(self.h, None, 0))
        out = np.zeros(n, OBJECT_DTYPE)
        self._chk(self.lib.rt_get_scene(self.h, _p(out), n))
        return out

    # state
    def set_camera(self, cam):
        self.camera = cam
        return self._chk(self.lib.rt_set_camera(self.h, C.byref(cam)))

    def set_params(self, params=None, **kw):
        if params is not None:
            self.params = params
        for k, v in kw.items():
            setattr(self.params, k, v)
        return self._chk(self.lib.rt_set_params(self.h, C.byref(self.params)))

    def set_option(self, opt, value):
        return self._chk(self.lib.rt_set_option(self.h, opt, value))

    def set_pixel_step(self, steps, strip_columns=0):
        return self._chk(self.lib.rt_set_pixel_step(self.h, steps, strip_columns))

    def set_shard(self, rank, world):
        return self._chk(self.lib.rt_set_shard(self.h, rank, world))

    # hot path
    def reset_accumulation(self):
        return self._chk(self.lib.rt_reset_accumulation(self.h))

    def render_spp(self, spp):
        return self._chk(self.lib.rt_render_spp(self.h, spp))

    def resolve_rgba8(self, flip_y=True, out=None):
        w, h = self.params.width, self.params.height
        if out is None:
            out = np.zeros((h, w), np.uint32)
        self._chk(self.lib.rt_resolve_rgba8(self.h, _p(out), out.strides[0], int(flip_y)))
        return out

    def render_frame(self, spp=1, flip_y=True, out=None):
        """rt_render_frame: spp more samples per pixel and the resolved frame in `out` (a host_surface() makes it one fused pass)."""
        w, h = self.params.width, self.params.height
        if out is None:
            out = np.zeros((h, w), np.uint32)
        self._chk(self.lib.rt_render_frame(self.h, int(spp), _p(out), out.strides[0], int(flip_y)))
        return out

    def denoise_rgba8(self, params=None, flip_y=True, out=None):
        """rt_denoise_rgba8: the resolved frame with the a-trous filter in front (params None: the library's defaults)."""
        w, h = self.params.width, self.params.height
        if out is None:
            out = np.zeros((h, w), np.uint32)
        self._chk(self.lib.rt_denoise_rgba8(self.h, C.byref(params) if params is not None else None, _p(out), out.strides[0], int(flip_y)))
        return out

    def read_denoised(self, params=None):
        """rt_read_denoised: the filtered mean radiance, (height, width, 4) float32 (r, g, b, 0), y-up."""
        w, h = self.params.width, self.params.height
        out = np.zeros((h, w, 4), np.float32)
        self._chk(self.lib.rt_read_denoised(self.h, C.byref(params) if params is not None else None, _p(out)))
        return out

    def temporal_rgba8(self, tparams=None, dn=None, flip_y=True, out=None):
        """rt_temporal_rgba8: the frame with the reprojected history blended in (tparams None: the library's defaults; dn None: no filter)."""
        w, h = self.params.width, self.params.height
        if out is None:
            out = np.zeros((h, w), np.uint32)
        self._chk(self.lib.rt_temporal_rgba8(self.h, C.byref(tparams) if tparams is not None else None, C.byref(dn) if dn is not None else None,
                                             _p(out), out.strides[0], int(flip_y)))
        return out

    def read_temporal(self, tparams=None, dn=None):
        """rt_read_temporal: (height, width, 4) float32 (r, g, b, N_eff), y-up."""
        w, h = self.params.width, self.params.height
        out = np.zeros((h, w, 4), np.float32)
        self._chk(self.lib.rt_read_temporal(self.h, C.byref(tparams) if tparams is not None else None, C.byref(dn) if dn is not None else None, _p(out)))
        return out

    def reset_temporal(self):
        self._chk(self.lib.rt_reset_temporal(self.h))

    def pick(self, x, y_window):
        i = C.c_int(-2)
        self._chk(self.lib.rt_pick(self.h, x, y_window, C.byref(i)))
        return i.value

    # hooks
    def read_accum(self):
        w, h = self.params.width, self.params.height
        out = np.zeros((h, w, 4), np.float32)
        n = C.c_uint32(0)
        self._chk(self.lib.rt_read_accum(self.h, _p(out), C.byref(n)))
        return out, n.value

    def write_accum(self, rgba, samples):
        rgba = np.ascontiguousarray(rgba, np.float32)
        return self._chk(self.lib.rt_write_accum(self.h, _p(rgba), samples))

    def object_name(self, i):
        v = self.lib.rt_object_name(self.h, i)
        return v.decode() if v is not None else None

    def scene_name(self):
        v = self.lib.rt_scene_name(self.h)
        return v.decode() if v is not None else None

    def read_aov(self):
        w, h = self.params.width, self.params.height
        ids = np.zeros((h, w), np.int32); t = np.zeros((h, w), np.float32)
        nrm = np.zeros((h, w, 3), np.float32); pt = np.zeros((h, w, 3), np.float32)
        self._chk(self.lib.rt_read_aov(self.h, _p(ids), _p(t), _p(nrm), _p(pt)))
        return ids, t, nrm, pt

    def read_ray_dirs(self):
        w, h = self.params.width, self.params.height
        out = np.zeros((h, w, 3), np.float32)
        self._chk(self.lib.rt_read_ray_dirs(self.h, _p(out)))
        return out

    def trace_rays(self, origin, direction):
        origin = np.ascontiguousarray(origin, np.float32)
        direction = np.ascontiguousarray(direction, np.float32)
        n = origin.shape[0]
        ids = np.zeros(n, np.int32); t = np.zeros(n, np.float32)
        nrm = np.zeros((n, 3), np.float32); pt = np.zeros((n, 3), np.float32)
        self._chk(self.lib.rt_trace_rays(self.h, _p(origin), _p(direction), n, _p(ids), _p(t), _p(nrm), _p(pt)))
        return ids, t, nrm, pt

    def env_color(self, dirs):
        dirs = np.ascontiguousarray(dirs, np.float32)
        out = np.zeros_like(dirs)
        self._chk(self.lib.rt_env_color(self.h, _p(dirs), dirs.shape[0], _p(out)))
        return out

    def philox(self, ctr, key):
        ctr = np.asarray(ctr, np.uint32); key = np.asarray(key, np.uint32); out = np.zeros(4, np.uint32)
        self._chk(self.lib.rt_philox_block(self.h, _p(ctr), _p(key), _p(out)))
        return out

    def selftest(self, which=0):
        n = C.c_int(-1)
        self._chk(self.lib.rt_selftest(self.h, which, C.byref(n)))
        return n.value

    def stats(self):
        s = RtStats()
        self._chk(self.lib.rt_get_stats(self.h, C.byref(s)))
        return s

    def traversal_stats(self):
        s = RtTraversalStats()
        self._chk(self.lib.rt_get_traversal_stats(self.h, C.byref(s)))
        return s

    def exchange_setup(self, rank, world, accum_ptrs, flag_ptrs, dst_argb_ptr):
        """accum_ptrs / flag_ptrs: device pointers in rank order (None for this rank's own)."""
        a = (C.c_void_p * world)(*accum_ptrs)
        f = (C.c_void_p * world)(*flag_ptrs)
        return self._chk(self.lib.rt_exchange_setup(self.h, rank, world, a, f, C.c_void_p(dst_argb_ptr) if dst_argb_ptr else None))

    def exchange_resolve(self, total_samples, flip_y=True):
        return self._chk(self.lib.rt_exchange_resolve(self.h, total_samples, int(flip_y)))

    # interop
    def accum_device_ptr(self):
        return self.lib.rt_accum_device_ptr(self.h)

    def argb_device_ptr(self):
        return self.lib.rt_argb_device_ptr(self.h)

    def ipc_export(self, which):
        buf = (C.c_ubyte * 64)()
        self._chk(self.lib.rt_ipc_export(self.h, which, buf))
        return bytes(buf)

    def ipc_open(self, handle):
        p = C.c_void_p()
        self._chk(self.lib.rt_ipc_open(self.h, (C.c_ubyte * 64).from_buffer_copy(handle), C.byref(p)))
        return p.value

    def ipc_close(self, ptr):
        return self._chk(self.lib.rt_ipc_close(self.h, C.c_void_p(ptr)))

    def resolve_fused(self, accum_ptrs, total_samples, first_pixel, n_pixels, dst_argb_ptr, flip_y=True):
        arr = (C.c_void_p * len(accum_ptrs))(*accum_ptrs)
        return self._chk(self.lib.rt_resolve_fused(self.h, arr, len(accum_ptrs), total_samples, first_pixel, n_pixels,
                                                   C.c_void_p(dst_argb_ptr), int(flip_y)))

    def read_surface(self):
        w, h = self.params.width, self.params.height
        out = np.zeros((h, w), np.uint32)
        self._chk(self.lib.rt_read_surface(self.h, _p(out), w * 4))
        return out

    def set_stream(self, stream_handle):
        return self._chk(self.lib.rt_set_stream(self.h, C.c_void_p(stream_handle)))

    def sync(self):
        return self._chk(self.lib.rt_sync(self.h))

    def set_sample_count(self, n):
        return self._chk(self.lib.rt_set_sample_count(self.h, n))

    def resolve_device(self, dev_accum_ptr, samples, first_pixel, n_pixels, dev_out_ptr, flip_y=True):
        return self._chk(self.lib.rt_resolve_device(self.h, C.c_void_p(dev_accum_ptr), samples, first_pixel, n_pixels,
                                                    C.c_void_p(dev_out_ptr), int(flip_y)))


class TracerGroup:
    """rt_group: library-owned multi-GPU in one process (rt_create_multi). members[i] is a PathTracer view of member i."""

    def __init__(self, devices):
        self.lib = load_library()
        devices = list(devices)
        arr = (C.c_int * len(devices))(*devices)
        g = C.c_void_p()
        rc = self.lib.rt_create_multi(len(devices), arr, C.byref(g))
        if rc != RT_OK:
            raise RtError(rc, (self.lib.rt_group_last_error(None) or b"").decode())
        self.g = g
        self.params = default_params()
        self.members = [PathTracer(_borrowed=self.lib.rt_group_ctx(self.g, i)) for i in range(len(devices))]

    def close(self):
        if getattr(self, "g", None):
            for m in self.members:
                m.close()
            self.lib.rt_group_destroy(self.g)
            self.g = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc < 0:
            raise RtError(rc, (self.lib.rt_group_last_error(self.g) or b"").decode())
        return rc

    def size(self):
        return self.lib.rt_group_size(self.g)

    def set_scene(self, objs):
        objs = np.ascontiguousarray(objs, OBJECT_DTYPE)
        return self._chk(self.lib.rt_group_set_scene(self.g, _p(objs), len(objs)))

    def load_scene(self, path):
        return self._chk(self.lib.rt_group_load_scene(self.g, str(path).encode()))

    def set_mesh(self, object_index, vertices, triangles):
        v = np.ascontiguousarray(vertices, np.float32).reshape(-1, 3)
        t = np.ascontiguousarray(triangles, np.int32).reshape(-1, 3)
        return self._chk(self.lib.rt_group_set_mesh(self.g, object_index, _p(v), len(v), _p(t), len(t)))

    def set_camera(self, cam):
        return self._chk(self.lib.rt_group_set_camera(self.g, C.byref(cam)))

    def set_params(self, params=None, **kw):
        if params is not None:
            self.params = params
        for k, v in kw.items():
            setattr(self.params, k, v)
        for m in self.members:
            m.params = self.params
        return self._chk(self.lib.rt_group_set_params(self.g, C.byref(self.params)))

    def set_option(self, opt, value):
        return self._chk(self.lib.rt_group_set_option(self.g, opt, value))

    def reset_accumulation(self):
        return self._chk(self.lib.rt_group_reset_accumulation(self.g))

    def render_spp(self, spp):
        return self._chk(self.lib.rt_group_render_spp(self.g, spp))

    def resolve_rgba8(self, flip_y=True, out=None):
        w, h = self.params.width, self.params.height
        if out is None:
            out = np.zeros((h, w), np.uint32)
        self._chk(self.lib.rt_group_resolve_rgba8(self.g, _p(out), out.strides[0], int(flip_y)))
        return out

    def denoise_rgba8(self, params=None, flip_y=True, out=None):
        """rt_group_denoise_rgba8: the group's frame with the a-trous filter in front (params None: the library's defaults)."""
        w, h = self.params.width, self.params.height
        if out is None:
            out = np.zeros((h, w), np.uint32)
        self._chk(self.lib.rt_group_denoise_rgba8(self.g, C.byref(params) if params is not None else None, _p(out), out.strides[0], int(flip_y)))
        return out

    def read_denoised(self, params=None):
        """rt_group_read_denoised: the filtered mean radiance of the group's samples, (height, width, 4) float32 (r, g, b, 0), y-up."""
        w, h = self.params.width, self.params.height
        out = np.zeros((h, w, 4), np.float32)
        self._chk(self.lib.rt_group_read_denoised(self.g, C.byref(params) if params is not None else None, _p(out)))
        return out

    def temporal_rgba8(self, tparams=None, dn=None, flip_y=True, out=None):
        """rt_group_temporal_rgba8: the group's frame with the reprojected history blended in (dn None: no filter)."""
        w, h = self.params.width, self.params.height
        if out is None:
            out = np.zeros((h, w), np.uint32)
        self._chk(self.lib.rt_group_temporal_rgba8(self.g, C.byref(tparams) if tparams is not None else None, C.byref(dn) if dn is not None else None,
                                                   _p(out), out.strides[0], int(flip_y)))
        return out

    def read_temporal(self, tparams=None, dn=None):
        """rt_group_read_temporal: (height, width, 4) float32 (r, g, b, N_eff), y-up."""
        w, h = self.params.width, self.params.height
        out = np.zeros((h, w, 4), np.float32)
        self._chk(self.lib.rt_group_read_temporal(self.g, C.byref(tparams) if tparams is not None else None, C.byref(dn) if dn is not None else None, _p(out)))
        return out

    def reset_temporal(self):
        self._chk(self.lib.rt_group_reset_temporal(self.g))

    def stats(self):
        s = RtStats()
        self._chk(self.lib.rt_group_get_stats(self.g, C.byref(s)))
        return s
