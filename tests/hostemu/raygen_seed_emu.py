"""ctypes front-end of tests/hostemu/libkzemu_raygen_seed.so: the host emulation (emu_py) plus the primary-hit seed split the way the
device runs it -- the seed test in k_raygen, the install in k_extend<true> (raygen_seed_emu.cpp; dev/test harness only)."""
import ctypes as C
import os
import subprocess

import numpy as np

import emu_py
from emu_py import pk

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "libkzemu_raygen_seed.so")


def build():
    srcs = [os.path.join(HERE, "raygen_seed_emu.cpp"), os.path.join(HERE, "emu.cpp")] + [
        os.path.join(emu_py.ROOT, "nano-kazen_b200", "csrc", f) for f in os.listdir(os.path.join(emu_py.ROOT, "nano-kazen_b200", "csrc")) if f.endswith(".h")]
    if os.path.exists(LIB) and all(os.path.getmtime(LIB) >= os.path.getmtime(s) for s in srcs):
        return
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-mfma", "-pthread", "-shared", "-o", LIB, os.path.join(HERE, "raygen_seed_emu.cpp")])


class RaygenSeedEmu(emu_py.Emu):
    def __init__(self, desc):
        build()
        self.lib = C.CDLL(LIB)
        self.h = C.c_void_p()
        rc = self.lib.kzemu_create(C.byref(desc), C.byref(self.h))
        if rc != 0:
            raise RuntimeError(f"kzemu_create failed ({rc})")
        self._desc = desc

    def seed_split(self, rays, seeds):
        """per ray and hint: (kz_seed_hit's hit, kz_trav_seed's best hit, taken bits: 1 seed test hit, 2 kz_trav_seed seeded, 4 preset installed)"""
        rays = np.ascontiguousarray(rays, pk.RAY_DTYPE)
        seeds = np.ascontiguousarray(seeds, np.uint32).reshape(rays.shape[0], 2)
        pure = np.zeros(rays.shape[0], pk.HIT_DTYPE)
        trav = np.zeros(rays.shape[0], pk.HIT_DTYPE)
        taken = np.zeros(rays.shape[0], np.uint8)
        self._call("seed_split", self.h, rays.ctypes.data_as(C.c_void_p), seeds.ctypes.data_as(C.c_void_p), C.c_size_t(rays.shape[0]),
                   pure.ctypes.data_as(C.c_void_p), trav.ctypes.data_as(C.c_void_p), taken.ctypes.data_as(C.c_void_p))
        return pure, trav, taken

    def trace_preset(self, rays, presets):
        """closest hits of traversals started from preset hits (pk.HIT_DTYPE, geom_id 0xFFFFFFFF: none) as k_extend<true> installs them"""
        rays = np.ascontiguousarray(rays, pk.RAY_DTYPE)
        presets = np.ascontiguousarray(presets, pk.HIT_DTYPE)
        hits = np.zeros(rays.shape[0], pk.HIT_DTYPE)
        self._call("trace_preset", self.h, rays.ctypes.data_as(C.c_void_p), presets.ctypes.data_as(C.c_void_p), C.c_size_t(rays.shape[0]),
                   hits.ctypes.data_as(C.c_void_p))
        return hits
