"""ctypes front-end of tests/hostemu/libkzemu_seed.so: the host emulation (emu_py) plus the traversal seeded with a closest-hit
hint (seed_emu.cpp; dev/test harness only)."""
import ctypes as C
import os
import subprocess

import numpy as np

import emu_py
from emu_py import pk

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "libkzemu_seed.so")


def build():
    srcs = [os.path.join(HERE, "seed_emu.cpp"), os.path.join(HERE, "emu.cpp")] + [
        os.path.join(emu_py.ROOT, "nano-kazen_b200", "csrc", f) for f in os.listdir(os.path.join(emu_py.ROOT, "nano-kazen_b200", "csrc")) if f.endswith(".h")]
    if os.path.exists(LIB) and all(os.path.getmtime(LIB) >= os.path.getmtime(s) for s in srcs):
        return
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-mfma", "-pthread", "-shared", "-o", LIB, os.path.join(HERE, "seed_emu.cpp")])


class SeedEmu(emu_py.Emu):
    def __init__(self, desc):
        build()
        self.lib = C.CDLL(LIB)
        self.h = C.c_void_p()
        rc = self.lib.kzemu_create(C.byref(desc), C.byref(self.h))
        if rc != 0:
            raise RuntimeError(f"kzemu_create failed ({rc})")
        self._desc = desc

    def trace_seeded(self, rays, seeds):
        """kz_trace with a closest-hit hint per ray: seeds = n x (geomID, primID) as uint32 (KZ_INVALID_ID: none); returns (hits, hints hit)"""
        rays = np.ascontiguousarray(rays, pk.RAY_DTYPE)
        seeds = np.ascontiguousarray(seeds, np.uint32).reshape(rays.shape[0], 2)
        hits = np.zeros(rays.shape[0], pk.HIT_DTYPE)
        k = C.c_uint64(0)
        self._call("trace_seeded", self.h, rays.ctypes.data_as(C.c_void_p), seeds.ctypes.data_as(C.c_void_p), C.c_size_t(rays.shape[0]),
                   hits.ctypes.data_as(C.c_void_p), C.byref(k))
        return hits, int(k.value)

    def trace_stats(self, rays, seeds):
        """node steps and triangle tests per ray of the plain per-ray loop, each ray seeded as in trace_seeded"""
        rays = np.ascontiguousarray(rays, pk.RAY_DTYPE)
        seeds = np.ascontiguousarray(seeds, np.uint32).reshape(rays.shape[0], 2)
        out = (C.c_uint64 * 2)()
        self._call("trace_stats_seeded", self.h, rays.ctypes.data_as(C.c_void_p), seeds.ctypes.data_as(C.c_void_p), C.c_size_t(rays.shape[0]), out)
        n = max(1, rays.shape[0])
        return {"nodes": out[0] / n, "tris": out[1] / n}
