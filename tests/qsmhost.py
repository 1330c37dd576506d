"""TEST INFRASTRUCTURE: the host build of tinygp_b200/csrc/qsm.cu (-DQSM_HOSTCHECK: the SAME source as the CUDA
kernels, warp bodies run with one lane, loops instead of launches) behind the context interface that
tinygp_b200.solvers.quasisep.core expects, so `-m "not gpu"` tests drive the real Python classes."""

import ctypes
import os
import shutil
import subprocess
from ctypes import byref, c_void_p

import pytest

from tinygp_b200 import _cabi

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "..", "tinygp_b200", "csrc")
SRC = os.path.join(CSRC, "qsm.cu")
OUT = os.path.join(HERE, "csrc", "_build", "libqsm_hostcheck.so")
DEPS = [SRC, os.path.join(CSRC, "qsm_core.cuh")]


class HostBackend:
    def __init__(self):
        gxx = shutil.which("g++")
        if gxx is None:
            pytest.skip("g++ not available")
        if not os.path.exists(OUT) or any(os.path.getmtime(d) > os.path.getmtime(OUT) for d in DEPS):
            os.makedirs(os.path.dirname(OUT), exist_ok=True)
            tmp = f"{OUT}.{os.getpid()}"     # parallel workers each build their own copy and swap it in whole
            subprocess.run([gxx, "-O2", "-std=c++17", "-DQSM_HOSTCHECK", "-fPIC", "-shared", "-x", "c++", SRC, "-o", tmp],
                           check=True)
            os.replace(tmp, OUT)
        lib = ctypes.CDLL(OUT)
        for name, (res, args) in _cabi.SIGNATURES.items():
            if hasattr(lib, name):
                fn = getattr(lib, name)
                fn.restype, fn.argtypes = res, args
        self.lib = lib
        self.handle = c_void_p()
        assert lib.b200gp_create(0, None, byref(self.handle)) == 0

    def check(self, rc):
        if rc != 0:
            raise _cabi.B200Error((self.lib.b200gp_last_error(self.handle) or b"unknown error").decode())

    def set_option(self, key, value):
        self.check(self.lib.b200gp_set_option(self.handle, key.encode(), int(value)))
