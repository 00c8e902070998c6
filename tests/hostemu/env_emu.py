"""ctypes front-end of tests/hostemu/libkzemu_env.so: the host emulation (emu_py) plus the environment table, sampling and density of
kz_env.h (env_emu.cpp; dev/test harness only)."""
import ctypes as C
import os
import subprocess

import numpy as np

import emu_py

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "libkzemu_env.so")
ENV_ZERO, ENV_CONSTANT, ENV_IMAGE = 0, 1, 2


def build():
    srcs = [os.path.join(HERE, "env_emu.cpp"), os.path.join(HERE, "emu.cpp")] + [
        os.path.join(emu_py.ROOT, "nano-kazen_b200", "csrc", f) for f in os.listdir(os.path.join(emu_py.ROOT, "nano-kazen_b200", "csrc")) if f.endswith(".h")]
    if os.path.exists(LIB) and all(os.path.getmtime(LIB) >= os.path.getmtime(s) for s in srcs):
        return
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-mfma", "-pthread", "-shared", "-o", LIB, os.path.join(HERE, "env_emu.cpp")])


class EnvEmu:
    def __init__(self, desc):
        build()
        self.lib = C.CDLL(LIB)
        self.h = C.c_void_p()
        rc = self.lib.kzenv_create(C.byref(desc), C.byref(self.h))
        if rc != 0:
            raise RuntimeError(f"kzenv_create failed ({rc})")
        self._desc = desc
        kind, w, h, counted, total = C.c_int(), C.c_int(), C.c_int(), C.c_int(), C.c_double()
        self.lib.kzenv_info(self.h, C.byref(kind), C.byref(w), C.byref(h), C.byref(counted), C.byref(total))
        self.kind, self.w, self.h_, self.counted, self.total = kind.value, w.value, h.value, bool(counted.value), total.value

    def close(self):
        if self.h:
            self.lib.kzenv_destroy(self.h); self.h = C.c_void_p()

    def table(self):
        """(row CDFs (h, w + 1), marginal (h + 1,), cell probabilities (h, w)) float32"""
        cdf = np.zeros((self.h_, self.w + 1), np.float32); marg = np.zeros(self.h_ + 1, np.float32); prob = np.zeros((self.h_, self.w), np.float32)
        self.lib.kzenv_table(self.h, cdf.ctypes.data_as(C.c_void_p), marg.ctypes.data_as(C.c_void_p), prob.ctypes.data_as(C.c_void_p))
        return cdf, marg, prob

    def eval(self, dirs):
        """(kz_background (n, 3), kz_env_pdf (n,)) per direction"""
        dirs = np.ascontiguousarray(dirs, np.float32).reshape(-1, 3)
        rgb = np.zeros((dirs.shape[0], 3), np.float32); pdf = np.zeros(dirs.shape[0], np.float32)
        self.lib.kzenv_eval(self.h, dirs.ctypes.data_as(C.c_void_p), C.c_size_t(dirs.shape[0]), rgb.ctypes.data_as(C.c_void_p), pdf.ctypes.data_as(C.c_void_p))
        return rgb, pdf

    def sample(self, u2):
        """(n, 8) float32 in kzgpu_env_sample_dump's layout"""
        u2 = np.ascontiguousarray(u2, np.float32).reshape(-1, 2)
        out = np.zeros((u2.shape[0], 8), np.float32)
        rc = self.lib.kzenv_sample(self.h, u2.ctypes.data_as(C.c_void_p), C.c_size_t(u2.shape[0]), out.ctypes.data_as(C.c_void_p))
        if rc != 0:
            raise RuntimeError(f"kzenv_sample failed ({rc})")
        return out
