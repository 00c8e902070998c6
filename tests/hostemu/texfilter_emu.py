"""ctypes front-end of tests/hostemu/libkzemu_texfilter.so: the host emulation (emu_py) plus the texture-filtering bodies of kz_texlod.h
and kz_shade.h (texfilter_emu.cpp; dev/test harness only)."""
import ctypes as C
import os
import subprocess

import numpy as np

import emu_py

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "libkzemu_texfilter.so")
LOD_FLOATS = 19          # camera_from_world[12], ddx[3], ddy[3], spp_scale
CASE_FLOATS = 56         # lod[19], camera_to_world[16], p, n, p0, p1, p2, uv0, uv1, uv2


def build():
    srcs = [os.path.join(HERE, "texfilter_emu.cpp"), os.path.join(HERE, "emu.cpp")] + [
        os.path.join(emu_py.ROOT, "nano-kazen_b200", "csrc", f) for f in os.listdir(os.path.join(emu_py.ROOT, "nano-kazen_b200", "csrc")) if f.endswith(".h")]
    if os.path.exists(LIB) and all(os.path.getmtime(LIB) >= os.path.getmtime(s) for s in srcs):
        return
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-mfma", "-pthread", "-shared", "-o", LIB, os.path.join(HERE, "texfilter_emu.cpp")])


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(LIB)
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def lod(camera, sample_count):
    """kz_tex_lod of a pykazen CameraDesc: 19 float32"""
    out = np.zeros(LOD_FLOATS, np.float32)
    lib().kztf_lod(C.byref(camera), C.c_uint32(sample_count), _p(out))
    return out


def footprint(cases):
    """kz_uv_footprint per (n, 56) case row -> (n, 4) du/dx, dv/dx, du/dy, dv/dy"""
    cases = np.ascontiguousarray(cases, np.float32).reshape(-1, CASE_FLOATS)
    out = np.zeros((cases.shape[0], 4), np.float32)
    lib().kztf_footprint(_p(cases), C.c_size_t(cases.shape[0]), _p(out))
    return out


def lam(w, h, dst4):
    dst4 = np.ascontiguousarray(dst4, np.float32).reshape(-1, 4)
    out = np.zeros(dst4.shape[0], np.float32)
    lib().kztf_lambda(C.c_int(w), C.c_int(h), _p(dst4), C.c_size_t(dst4.shape[0]), _p(out))
    return out


def _pyr(levels):
    """list of (h, w, 3) float32 levels -> (w, h, n_levels, flat float4 texels)"""
    flat = np.concatenate([np.concatenate([l.astype(np.float32), np.ones(l.shape[:2] + (1,), np.float32)], -1).reshape(-1, 4) for l in levels])
    return levels[0].shape[1], levels[0].shape[0], len(levels) - 1, np.ascontiguousarray(flat)


def filtered(levels, st, lambdas):
    w, h, nl, tex = _pyr(levels)
    st = np.ascontiguousarray(st, np.float32).reshape(-1, 2); lambdas = np.ascontiguousarray(lambdas, np.float32).reshape(-1)
    out = np.zeros((st.shape[0], 3), np.float32)
    lib().kztf_filtered(C.c_int(w), C.c_int(h), C.c_int(nl), _p(tex), _p(st), _p(lambdas), C.c_size_t(st.shape[0]), _p(out))
    return out


def bicubic(levels, st, level):
    w, h, nl, tex = _pyr(levels)
    st = np.ascontiguousarray(st, np.float32).reshape(-1, 2)
    out = np.zeros((st.shape[0], 3), np.float32)
    lib().kztf_bicubic(C.c_int(w), C.c_int(h), C.c_int(nl), _p(tex), _p(st), C.c_int(level), C.c_size_t(st.shape[0]), _p(out))
    return out


def lookup_filtered(levels, st, dst4):
    w, h, nl, tex = _pyr(levels)
    st = np.ascontiguousarray(st, np.float32).reshape(-1, 2); dst4 = np.ascontiguousarray(dst4, np.float32).reshape(-1, 4)
    out = np.zeros((st.shape[0], 3), np.float32)
    lib().kztf_lookup_filtered(C.c_int(w), C.c_int(h), C.c_int(nl), _p(tex), _p(st), _p(dst4), C.c_size_t(st.shape[0]), _p(out))
    return out


def layout(desc):
    """(counts, total texels, per-image n_levels) of the upload's texture-filtering decision; raises with the upload's message"""
    counts, total = C.c_int(), C.c_uint64()
    levels = np.zeros(max(1, desc.n_images), np.int32)
    err = C.create_string_buffer(512)
    rc = lib().kztf_layout(C.byref(desc), C.byref(counts), C.byref(total), _p(levels), err, C.c_size_t(len(err)))
    if rc != 0:
        raise RuntimeError(err.value.decode())
    return bool(counts.value), total.value, levels[:desc.n_images]


class FootprintEmu:
    """the emulated scene (this library's own kzemu) with kzgpu_texture_footprint_dump's probe"""

    def __init__(self, desc):
        self.lib = lib()
        self.h = C.c_void_p()
        rc = self.lib.kzemu_create(C.byref(desc), C.byref(self.h))
        if rc != 0:
            raise RuntimeError(f"kzemu_create failed ({rc})")
        self._desc = desc

    def close(self):
        if self.h:
            self.lib.kzemu_destroy(self.h); self.h = C.c_void_p()

    def texture_footprint_dump(self, rays):
        rays = np.ascontiguousarray(rays, emu_py.pk.RAY_DTYPE)
        out = np.zeros((rays.shape[0], 8), np.float32)
        rc = self.lib.kztf_footprint_dump(self.h, _p(rays), C.c_size_t(rays.shape[0]), _p(out))
        if rc != 0:
            raise RuntimeError(f"kztf_footprint_dump failed ({rc})")
        return out
