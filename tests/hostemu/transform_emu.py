"""ctypes front-end of tests/hostemu/libkzemu_transform.so: the per-vertex body of kzgpu_mesh_transform (kz_transform.h) compiled for
the host (transform_emu.cpp; dev/test harness only)."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
LIB = os.path.join(HERE, "libkzemu_transform.so")
SRCS = [os.path.join(HERE, "transform_emu.cpp")] + [os.path.join(ROOT, "nano-kazen_b200", "csrc", f) for f in ("kz_transform.h", "kz_common.h")]


def build():
    if os.path.exists(LIB) and all(os.path.getmtime(LIB) >= os.path.getmtime(s) for s in SRCS):
        return
    # the flags of the other emulation libraries: -mfma lets g++ contract whatever the kz_* helpers do not pin down
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-mfma", "-shared", "-o", LIB, SRCS[0]])


def transform(matrix, inverse, positions, normals=None):
    """(positions, normals) placed as k_transform_vertices places them: float32 (n, 3) arrays (normals None if not given)"""
    build()
    lib = C.CDLL(LIB)
    f = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))
    M = np.ascontiguousarray(matrix, np.float32).reshape(16)
    I = np.ascontiguousarray(np.zeros(16) if inverse is None else inverse, np.float32).reshape(16)
    P = np.ascontiguousarray(positions, np.float32).reshape(-1, 3)
    N = None if normals is None else np.ascontiguousarray(normals, np.float32).reshape(-1, 3)
    op = np.zeros_like(P); on = None if N is None else np.zeros_like(N)
    lib.kzemu_transform(f(M), f(I), f(P), None if N is None else f(N), C.c_size_t(P.shape[0]), f(op), None if N is None else f(on))
    return op, on
