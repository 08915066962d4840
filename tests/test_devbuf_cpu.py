"""CPU: the ownership rules of DeviceArray (csrc/rt_devbuf.h), the owner of every device buffer of a context and of the wavefront
pipeline, compiled with g++ against a fake CUDA allocator (tests/host_emu/fake_cuda/cuda_runtime.h) that counts allocations and
frees, fails the n-th cudaMalloc on request and models the runtime's last error. The checks are in tests/host_emu/devbuf_emu.cpp."""
import ctypes as C
import os
import subprocess

import pytest

from conftest import ROOT

EMU_DIR = os.path.join(ROOT, "tests", "host_emu")
CHECKS = ["devbuf_reserve_within_capacity", "devbuf_growth_frees_old_once", "devbuf_failed_reserve_leaves_empty",
          "devbuf_move_leaves_source_empty", "devbuf_group_all_or_nothing", "devbuf_everything_freed_once"]


@pytest.fixture(scope="session")
def devbuf_emu(tmp_path_factory):
    """g++ build of tests/host_emu/devbuf_emu.cpp with the fake cuda_runtime.h first on the include path."""
    so = str(tmp_path_factory.mktemp("devbuf_emu") / "libdevbuf_emu.so")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-Wextra", "-Werror", "-fPIC", "-shared", "-I", os.path.join(EMU_DIR, "fake_cuda"),
                           "-o", so, os.path.join(EMU_DIR, "devbuf_emu.cpp")])
    return C.CDLL(so)


@pytest.mark.parametrize("check", CHECKS)
def test_devbuf_cpu(devbuf_emu, check):
    fn = getattr(devbuf_emu, check)
    fn.restype = C.c_int
    line = fn()
    assert line == 0, f"{check}: condition at tests/host_emu/devbuf_emu.cpp:{line} does not hold"
