"""Loader of the lane engine's CPU emulator, libptv_emu_lane.so (built by tests/emu/Makefile, which __graft_entry__.build() runs).

load(required): the ctypes handle with its signatures.  A missing or stale library is (re)built with the Makefile's command when the
CUDA headers are present.  Without them: required=False skips the calling test (a CPU machine without CUDA), required=True fails it
(the GPU tests use the emulator as their reference and must not pass without one)."""
import ctypes as C
import os
import subprocess

import pytest

EMU_DIR = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(EMU_DIR, "libptv_emu_lane.so")
SOURCES = (os.path.join(EMU_DIR, "emu_lane.cu"), os.path.join(EMU_DIR, "..", "..", "proxtv_b200", "csrc", "lane_core.cuh"))
CUDA_INC = "/usr/local/cuda/include"
dp = C.POINTER(C.c_double)
fp = C.POINTER(C.c_float)


def load(required=False):
    if not os.path.exists(SO) or any(os.path.getmtime(f) > os.path.getmtime(SO) for f in SOURCES):
        if not os.path.isdir(CUDA_INC):
            msg = "lane emulator %s is missing and the CUDA headers to build it are not available" % SO
            if required:
                pytest.fail(msg)
            pytest.skip(msg)
        subprocess.check_call(["make", "-s", "-C", EMU_DIR, "CUDA_INC=" + CUDA_INC, "libptv_emu_lane.so"])
    lib = C.CDLL(SO)
    lib.emu_lane_f64.argtypes = [C.c_int, dp, dp, dp, dp, dp, C.c_longlong, C.c_int, C.c_longlong, C.c_double, C.c_int, C.c_int, C.c_int, C.c_int,
                                 C.POINTER(C.c_longlong)]
    lib.emu_lane_f32.argtypes = [C.c_int, fp, fp, fp, fp, fp, C.c_longlong, C.c_int, C.c_longlong, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int,
                                 C.POINTER(C.c_longlong)]
    lib.emu_slope_seq_f64.argtypes = [dp, C.c_int, C.c_double, dp, C.POINTER(C.c_longlong)]
    lib.emu_slope_seq_rows_f64.argtypes = [dp, C.c_longlong, C.c_int, C.c_double, dp]
    lib.emu_plan.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.emu_taskplan.argtypes = [C.c_int, C.c_longlong, C.c_longlong]; lib.emu_taskplan.restype = C.c_longlong
    return lib
