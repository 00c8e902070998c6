"""ctypes front-end of tests/hostemu/libkzemu_refit.so: the host emulation (emu_py) plus the accel refit of kz_refit.h (refit_emu.cpp;
dev/test harness only)."""
import ctypes as C
import os
import subprocess

import numpy as np

import emu_py

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "libkzemu_refit.so")


def build():
    srcs = [os.path.join(HERE, "refit_emu.cpp"), os.path.join(HERE, "emu.cpp")] + [
        os.path.join(emu_py.ROOT, "nano-kazen_b200", "csrc", f) for f in os.listdir(os.path.join(emu_py.ROOT, "nano-kazen_b200", "csrc")) if f.endswith(".h")]
    if os.path.exists(LIB) and all(os.path.getmtime(LIB) >= os.path.getmtime(s) for s in srcs):
        return
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-mfma", "-pthread", "-shared", "-o", LIB, os.path.join(HERE, "refit_emu.cpp")])


class RefitEmu(emu_py.Emu):
    def __init__(self, desc):
        build()
        self.lib = C.CDLL(LIB)
        self.h = C.c_void_p()
        rc = self.lib.kzemu_create(C.byref(desc), C.byref(self.h))
        if rc != 0:
            raise RuntimeError(f"kzemu_create failed ({rc})")
        self._desc = desc

    def refit(self, desc):
        """the scene becomes `desc` (same topology, new positions); the accel built for the old positions is refitted"""
        self._call("refit", self.h, C.byref(desc))
        self._desc = desc

    def accel_dump(self):
        """(nodes as raw (n_nodes, 80) uint8, triangle records as (n_tris, 3, 4) float32)"""
        n, t, _ = self.bvh_info()
        nodes = np.zeros((n, 80), np.uint8); tris = np.zeros((t, 3, 4), np.float32)
        self._call("accel_dump", self.h, nodes.ctypes.data_as(C.c_void_p), tris.ctypes.data_as(C.c_void_p))
        return nodes, tris

    def scene_max_abs(self):
        v = C.c_float()
        self._call("scene_max_abs", self.h, C.byref(v))
        return v.value
