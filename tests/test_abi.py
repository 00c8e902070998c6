"""The C-ABI shared library loads on a box without a GPU, exports every symbol include/kzgpu.h
declares, and refuses to run (no CPU fallback) when no CUDA device is present."""
import ctypes as C
import os
import re

import pykazen as pk

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared(header):
    src = open(os.path.join(ROOT, "include", header)).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(kzgpu_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(gpu_lib):
    lib = C.CDLL(gpu_lib)
    names = _declared("kzgpu.h")
    assert len(names) >= 15
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/kzgpu.h but not exported"


def test_struct_sizes_match_header():
    """ctypes mirrors of the POD tables (pykazen) vs. the sizes the C compiler sees"""
    import subprocess, tempfile
    prog = '#include "kzgpu.h"\n#include <stdio.h>\nint main(){printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\\n",' \
           'sizeof(kz_ray),sizeof(kz_hit),sizeof(kz_mesh_desc),sizeof(kz_texture_desc),sizeof(kz_image_desc),sizeof(kz_bsdf_desc),' \
           'sizeof(kz_light_desc),sizeof(kz_camera_desc),sizeof(kz_sampler_desc),sizeof(kz_integrator_desc),sizeof(kz_filter_desc),' \
           'sizeof(kz_scene_desc),sizeof(kz_stats));return 0;}\n'
    with tempfile.TemporaryDirectory() as td:
        open(os.path.join(td, "s.c"), "w").write(prog)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", os.path.join(td, "s"), os.path.join(td, "s.c")])
        out = subprocess.check_output([os.path.join(td, "s")]).split()
    got = [int(v) for v in out]
    exp = [pk.RAY_DTYPE.itemsize, pk.HIT_DTYPE.itemsize] + [C.sizeof(t) for t in (
        pk.MeshDesc, pk.TextureDesc, pk.ImageDesc, pk.BsdfDesc, pk.LightDesc, pk.CameraDesc, pk.SamplerDesc, pk.IntegratorDesc,
        pk.FilterDesc, pk.SceneDesc, pk.Stats)]
    assert got == exp


NO_DEVICE_CHECK = r"""
import ctypes as C, sys
sys.path[:0] = sys.argv[2:]
import pykazen as pk, scenes
lib = C.CDLL(sys.argv[1])
lib.kzgpu_last_error.restype = C.c_char_p
h = C.c_void_p()
rc = lib.kzgpu_create(None, 0, C.byref(h))
assert rc == pk.KZ_ERR_NO_DEVICE and not h.value, rc
assert b"no CUDA device" in lib.kzgpu_last_error(None), lib.kzgpu_last_error(None)
try:
    pk.Gpu(scenes.soup_scene(10).desc(), lib_path=sys.argv[1])
    raise SystemExit("pykazen.Gpu did not raise")
except RuntimeError as e:
    assert "kzgpu_create failed" in str(e), e
print("no-device ok")
"""


def test_no_cpu_fallback(gpu_lib):
    """without a CUDA device kzgpu_create must fail loudly with KZ_ERR_NO_DEVICE (checked in a process that sees no device, so that
    it runs on GPU machines as well)"""
    import subprocess, sys
    r = subprocess.run([sys.executable, "-c", NO_DEVICE_CHECK, gpu_lib, os.path.join(ROOT, "nano-kazen_b200"), os.path.join(ROOT, "tests")],
                       capture_output=True, text=True, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), timeout=300)
    assert r.returncode == 0 and "no-device ok" in r.stdout, r.stderr[-2000:]


def test_product_never_touches_the_oracle():
    """nothing under nano-kazen_b200/ or include/ may reference oracle/ or the host emulation"""
    bad = []
    for base in ("nano-kazen_b200", "include"):
        for dp, _, fs in os.walk(os.path.join(ROOT, base)):
            for f in fs:
                if f.endswith((".so", ".o", ".pyc")):
                    continue
                txt = open(os.path.join(dp, f), errors="ignore").read()
                if f.endswith((".h", ".cuh", ".cu", ".cpp", ".c")):       # comments may cite the oracle, code may not
                    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
                    txt = re.sub(r"//[^\n]*", "", txt)
                for needle in ("kzo_", "libkzoracle", "kzemu_", "libkzemu", "oracle/", "kzo_py", "emu_py"):
                    if needle in txt:
                        bad.append((f, needle))
    assert not bad, bad
