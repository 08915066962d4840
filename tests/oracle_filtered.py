"""The oracle with the product's pixel filter in front (tests/oracle_filtered.c, which includes oracle/pt_oracle.c unchanged): an
Oracle whose library also has orc_render_filtered and orc_sample_dirs. Built with the oracle's flags into a temporary directory."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from oracle_py import Oracle, _p

HERE = os.path.dirname(os.path.abspath(__file__))
_INSTANCE = None


class FilteredOracle(Oracle):
    def __init__(self):
        super().__init__()
        so = os.path.join(tempfile.mkdtemp(prefix="oracle_filtered"), "liboracle_filtered.so")
        subprocess.check_call(["gcc", "-std=c11", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-pthread",
                               "-o", so, os.path.join(HERE, "oracle_filtered.c"), "-lm"])
        base, self.lib = self.lib, C.CDLL(so)
        for name in ("orc_render", "orc_time_render", "orc_resolve_pixel"):
            getattr(self.lib, name).restype = getattr(base, name).restype
        self.lib.orc_resolve_pixel.argtypes = base.orc_resolve_pixel.argtypes
        self.lib.orc_render_filtered.restype = C.c_longlong

    def render_filtered(self, objs, cam, params, s0, nspp, filter_type, radius, threads=None, per_sample=False):
        """render() (Philox streams) with the PRODUCT'S pixel filter: every sample's primary ray is sample_dirs()'s.
        Returns (sum, samples|None, segments)."""
        w, h = params.width, params.height
        out = np.zeros((h, w, 3), np.float32)
        samples = np.zeros((nspp, h, w, 3), np.float32) if per_sample else None
        threads = threads or (os.cpu_count() or 1)
        segs = self.lib.orc_render_filtered(_p(objs), len(objs), C.byref(cam), C.byref(params), s0, nspp, int(filter_type),
                                            C.c_float(radius), threads, _p(out), _p(samples))
        return out, samples, segs

    def sample_dirs(self, cam, w, h, seed_lo, seed_hi, filter_type, radius, sample):
        """(H, W, 3) primary direction of global sample `sample` of every pixel under the product's pixel filter."""
        out = np.zeros((h, w, 3), np.float32)
        self.lib.orc_sample_dirs(C.byref(cam), w, h, C.c_uint32(seed_lo), C.c_uint32(seed_hi), int(filter_type), C.c_float(radius),
                                 C.c_uint32(sample), _p(out))
        return out


def filtered_oracle():
    """One FilteredOracle per process."""
    global _INSTANCE
    if _INSTANCE is None:
        _INSTANCE = FilteredOracle()
    return _INSTANCE
