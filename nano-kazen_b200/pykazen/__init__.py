"""pykazen -- ctypes view of the kzgpu C ABI (include/kzgpu.h) plus helpers to assemble the POD
scene tables from numpy arrays.  This is plumbing for tests / bench.py; the product boundary is
the C ABI itself and the C++ host (nano-kazen_b200/host)."""
import ctypes as C
import math
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
PKG = os.path.join(ROOT, "nano-kazen_b200")
LIB_GPU = os.environ.get("KZGPU_LIB") or os.path.join(PKG, "csrc", "libkzgpu.so")      # KZGPU_LIB: another build of the same ABI (tuning experiments)
LIB_HOST = os.path.join(PKG, "host", "libkazen_host.so")

KZ_INVALID_ID = 0xFFFFFFFF
KZ_OK = 0
KZ_ERR_NO_DEVICE = -2

TEX_CONSTANT, TEX_IMAGE, TEX_BACKGROUND, TEX_COLORRAMP, TEX_BLEND = range(5)
BSDF_DIFFUSE, BSDF_KISS, BSDF_NORMALMAP, BSDF_DIELECTRIC, BSDF_MIRROR, BSDF_LAMBERTIAN, BSDF_GGX, BSDF_ROUGHCONDUCTOR, BSDF_ROUGHPLASTIC, BSDF_ROUGHDIELECTRIC = range(10)
CONDUCTORS = {"Au": ((0.1431189557, 0.3749570432, 1.4424785571), (3.9831604247, 2.3857207478, 1.6032152899)),
              "Cu": ((0.2004376970, 0.9240334304, 1.1022119527), (3.9129485033, 2.4528477015, 2.1421879552)),
              "Cr": ((4.3696828663, 2.9167024892, 1.6547005413), (5.2064337956, 4.2313645277, 3.7549467933))}
CAM_PERSPECTIVE, CAM_THINLENS = range(2)
SAMPLER_INDEPENDENT, SAMPLER_STRATIFIED, SAMPLER_CORRELATED, SAMPLER_PMJ02BN = range(4)
BUILD_HOST_SAH, BUILD_LBVH, BUILD_LBVH_MESHES = 0, 1, 2

RAY_DTYPE = np.dtype([("o", "<f4", 3), ("tmin", "<f4"), ("d", "<f4", 3), ("tmax", "<f4")])
HIT_DTYPE = np.dtype([("t", "<f4"), ("u", "<f4"), ("v", "<f4"), ("prim_id", "<u4"), ("geom_id", "<u4")])
assert RAY_DTYPE.itemsize == 32 and HIT_DTYPE.itemsize == 20

c_float_p = C.POINTER(C.c_float)
c_u32_p = C.POINTER(C.c_uint32)


class MeshDesc(C.Structure):
    _fields_ = [("positions", c_float_p), ("normals", c_float_p), ("uvs", c_float_p), ("indices", c_u32_p),
                ("n_vertices", C.c_uint32), ("n_triangles", C.c_uint32), ("bsdf", C.c_int32), ("light", C.c_int32)]


class TextureDesc(C.Structure):
    _fields_ = [("type", C.c_int32), ("color", C.c_float * 3), ("image", C.c_int32), ("scale", C.c_float),
                ("srgb", C.c_int32), ("a", C.c_float), ("b", C.c_float), ("mode", C.c_int32), ("child", C.c_int32 * 3)]


class ImageDesc(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("rgb", c_float_p)]


class BsdfDesc(C.Structure):
    _fields_ = [("type", C.c_int32), ("albedo", C.c_float * 3), ("base_color", C.c_int32), ("roughness", C.c_int32),
                ("metallic", C.c_int32), ("anisotropy", C.c_float), ("specular", C.c_float), ("specular_tint", C.c_float),
                ("clearcoat", C.c_float), ("clearcoat_roughness", C.c_float), ("sheen", C.c_float), ("sheen_tint", C.c_float),
                ("normal_map", C.c_int32), ("nested", C.c_int32), ("int_ior", C.c_float), ("ext_ior", C.c_float), ("alpha", C.c_float),
                ("eta", C.c_float * 3), ("k", C.c_float * 3)]


class LightDesc(C.Structure):
    _fields_ = [("radiance", C.c_float * 3), ("primary_visibility", C.c_int32)]


class CameraDesc(C.Structure):
    _fields_ = [("type", C.c_int32), ("width", C.c_int32), ("height", C.c_int32), ("sample_to_camera", C.c_float * 16),
                ("camera_to_world", C.c_float * 16), ("near_clip", C.c_float), ("far_clip", C.c_float),
                ("aperture_radius", C.c_float), ("focus_distance", C.c_float)]


class SamplerDesc(C.Structure):
    _fields_ = [("type", C.c_int32), ("sample_count", C.c_uint32), ("seed", C.c_uint64), ("res_x", C.c_int32),
                ("res_y", C.c_int32), ("blue_noise", C.POINTER(C.c_uint16)), ("pmj02bn", c_u32_p)]


class IntegratorDesc(C.Structure):
    _fields_ = [("max_depth", C.c_int32), ("trace_bias", C.c_float), ("regularization", C.c_int32),
                ("accumulated_roughness", C.c_float), ("type", C.c_int32), ("env_sampling", C.c_int32), ("texture_filtering", C.c_int32)]


class FilterDesc(C.Structure):
    _fields_ = [("radius", C.c_float), ("table", C.c_float * 33)]


class SceneDesc(C.Structure):
    _fields_ = [("meshes", C.POINTER(MeshDesc)), ("n_meshes", C.c_uint32),
                ("bsdfs", C.POINTER(BsdfDesc)), ("n_bsdfs", C.c_uint32),
                ("textures", C.POINTER(TextureDesc)), ("n_textures", C.c_uint32),
                ("images", C.POINTER(ImageDesc)), ("n_images", C.c_uint32),
                ("lights", C.POINTER(LightDesc)), ("n_lights", C.c_uint32),
                ("background", C.c_int32), ("camera", CameraDesc), ("sampler", SamplerDesc),
                ("integrator", IntegratorDesc), ("filter", FilterDesc)]


class RenderReq(C.Structure):
    _fields_ = [("x0", C.c_int32), ("y0", C.c_int32), ("x1", C.c_int32), ("y1", C.c_int32),
                ("spp_begin", C.c_int32), ("spp_end", C.c_int32), ("clear_frame", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [("paths", C.c_uint64), ("rays_extension", C.c_uint64), ("rays_shadow", C.c_uint64), ("vertices", C.c_uint64),
                ("kernel_launches", C.c_uint64), ("ms_trace", C.c_double), ("ms_shade", C.c_double), ("ms_total", C.c_double),
                ("bvh_nodes", C.c_uint64), ("bvh_bytes", C.c_uint64), ("ms_build", C.c_double),
                ("ms_upload", C.c_double), ("ms_merge", C.c_double), ("rays_seeded", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


# --------------------------------------------------------------------------- filter / camera setup
def filter_table(kind="gaussian", radius=2.0, stddev=0.5, B=1.0 / 3.0, Cc=1.0 / 3.0):
    """ImageBlock's 33-entry table (block.cpp:13-21) for the rfilter plugins (rfilter.cpp:10-102)."""
    f32 = np.float32
    if kind == "tent":
        radius = 1.0
    if kind == "box":
        radius = 0.5
    radius = f32(radius)

    def ev(x):
        x = f32(x)
        if kind == "gaussian":
            alpha = f32(-1.0) / (f32(2.0) * f32(stddev) * f32(stddev))
            # std::exp(float) of the reference is glibc's expf; numpy's float32 exp is a SIMD kernel that differs in the last bit for a
            # third of the entries (found against tests/golden/math_kat.json), the double exp rounded to float does not
            return max(f32(0), f32(math.exp(float(f32(alpha * x * x)))) - f32(math.exp(float(f32(alpha * radius * radius)))))
        if kind == "mitchell":
            Bf, Cf = f32(B), f32(Cc)
            x = abs(f32(2.0) * x / radius)
            x2 = x * x
            x3 = x2 * x
            if x < 1:
                return f32(1.0) / f32(6.0) * ((12 - 9 * Bf - 6 * Cf) * x3 + (-18 + 12 * Bf + 6 * Cf) * x2 + (6 - 2 * Bf))
            if x < 2:
                return f32(1.0) / f32(6.0) * ((-Bf - 6 * Cf) * x3 + (6 * Bf + 30 * Cf) * x2 + (-12 * Bf - 48 * Cf) * x + (8 * Bf + 24 * Cf))
            return f32(0)
        if kind == "tent":
            return max(f32(0), f32(1) - abs(x))
        return f32(1)

    tab = np.zeros(33, np.float32)
    for i in range(32):
        tab[i] = ev(f32(radius * f32(i)) / f32(32))
    return float(radius), tab


def perspective_sample_to_camera(width, height, fov, near, far):
    """Camera::activate, camera.cpp:35-62 (row-major 4x4, float32)."""
    aspect = width / float(height)
    recip = 1.0 / (far - near)
    cot = 1.0 / math.tan(math.radians(fov / 2.0))
    P = np.array([[cot, 0, 0, 0], [0, cot, 0, 0], [0, 0, far * recip, -near * far * recip], [0, 0, 1, 0]], np.float64)
    T = np.eye(4); T[0, 3] = -1.0; T[1, 3] = -1.0 / aspect
    S = np.diag([-0.5, -0.5 * aspect, 1.0, 1.0])
    return np.linalg.inv(S @ T @ P).astype(np.float32)


def lookat(origin, target, up):
    """parser.cpp:273-287 (lookat transform op), row-major."""
    o, t, u = (np.asarray(v, np.float64) for v in (origin, target, up))
    d = (t - o); d /= np.linalg.norm(d)
    left = np.cross(u / np.linalg.norm(u), d); left /= np.linalg.norm(left)
    nu = np.cross(d, left); nu /= np.linalg.norm(nu)
    M = np.eye(4)
    M[:3, 0], M[:3, 1], M[:3, 2], M[:3, 3] = left, nu, d, o
    return M.astype(np.float32)


def fill_camera(c, width, height, fov, to_world, near=1e-4, far=1e4, thinlens=None):
    """CameraDesc `c` of a perspective (thinlens = (aperture_radius, focus_distance): thin-lens) camera after Camera::activate"""
    c.type = CAM_THINLENS if thinlens else CAM_PERSPECTIVE
    c.width, c.height, c.near_clip, c.far_clip = width, height, near, far
    c.sample_to_camera[:] = perspective_sample_to_camera(width, height, fov, near, far).reshape(-1).tolist()
    c.camera_to_world[:] = np.asarray(to_world, np.float32).reshape(-1).tolist()
    c.aperture_radius, c.focus_distance = thinlens if thinlens else (1.0, 0.0)
    return c


class SceneBuilder:
    """Assembles a kz_scene_desc; keeps every numpy buffer alive for the lifetime of the object."""

    def __init__(self):
        self._keep = []
        self.meshes, self.bsdfs, self.textures, self.images, self.lights = [], [], [], [], []
        self.background = -1
        self.camera = CameraDesc()
        self.sampler = SamplerDesc()
        self.integrator = IntegratorDesc(5, 1e-3, 0, 0.5, 0)
        self.filter = FilterDesc()
        self.set_filter("gaussian")
        self.set_sampler("independent", 1)
        self.set_camera(64, 64, 30.0, np.eye(4, dtype=np.float32))

    def _arr(self, a, dtype):
        a = np.ascontiguousarray(a, dtype=dtype)
        self._keep.append(a)
        return a

    # textures -----------------------------------------------------------------------------------
    def tex_constant(self, rgb):
        t = TextureDesc(); t.type = TEX_CONSTANT
        t.color[:] = [float(c) for c in rgb]; t.child[:] = [-1, -1, -1]
        self.textures.append(t); return len(self.textures) - 1

    def tex_image(self, rgb_hw3, scale=1.0, srgb=True):
        img = self._arr(rgb_hw3, np.float32)
        d = ImageDesc(img.shape[1], img.shape[0], img.ctypes.data_as(c_float_p))
        self.images.append(d)
        t = TextureDesc(); t.type = TEX_IMAGE; t.image = len(self.images) - 1; t.scale = scale; t.srgb = int(srgb)
        t.child[:] = [-1, -1, -1]
        self.textures.append(t); return len(self.textures) - 1

    def tex_background(self, intensity, child):
        t = TextureDesc(); t.type = TEX_BACKGROUND; t.a = intensity; t.child[:] = [child, -1, -1]
        self.textures.append(t); return len(self.textures) - 1

    def tex_colorramp(self, lo, hi, child):
        t = TextureDesc(); t.type = TEX_COLORRAMP; t.a = lo; t.b = hi; t.child[:] = [child, -1, -1]
        self.textures.append(t); return len(self.textures) - 1

    def tex_blend(self, mode, mask=-1, input1=-1, input2=-1):
        t = TextureDesc(); t.type = TEX_BLEND; t.mode = {"mix": 0, "multiply": 1}.get(mode, 2)
        t.child[:] = [mask, input1, input2]
        self.textures.append(t); return len(self.textures) - 1

    # bsdfs --------------------------------------------------------------------------------------
    def bsdf_diffuse(self, albedo=(0.5, 0.5, 0.5)):
        b = BsdfDesc(); b.type = BSDF_DIFFUSE; b.albedo[:] = [float(c) for c in albedo]
        b.base_color = b.roughness = b.metallic = b.normal_map = b.nested = -1
        self.bsdfs.append(b); return len(self.bsdfs) - 1

    def bsdf_kiss(self, base_color, roughness, metallic, anisotropy=0.0, specular=0.5, specular_tint=0.5, clearcoat=0.0,
                  clearcoat_roughness=0.5, sheen=0.0, sheen_tint=0.5):
        b = BsdfDesc(); b.type = BSDF_KISS
        b.base_color, b.roughness, b.metallic = base_color, roughness, metallic
        b.anisotropy, b.specular, b.specular_tint = anisotropy, specular, specular_tint
        b.clearcoat, b.clearcoat_roughness, b.sheen, b.sheen_tint = clearcoat, clearcoat_roughness, sheen, sheen_tint
        b.normal_map = b.nested = -1
        self.bsdfs.append(b); return len(self.bsdfs) - 1

    def bsdf_normalmap(self, normal_tex, nested):
        b = BsdfDesc(); b.type = BSDF_NORMALMAP; b.normal_map = normal_tex; b.nested = nested
        b.base_color = b.roughness = b.metallic = -1
        self.bsdfs.append(b); return len(self.bsdfs) - 1

    def _blank(self, t):
        b = BsdfDesc(); b.type = t
        b.base_color = b.roughness = b.metallic = b.normal_map = b.nested = -1
        b.int_ior, b.ext_ior = 1.5046, 1.000277
        return b

    def bsdf_dielectric(self, int_ior=1.5046, ext_ior=1.000277):
        b = self._blank(BSDF_DIELECTRIC); b.int_ior, b.ext_ior = int_ior, ext_ior
        self.bsdfs.append(b); return len(self.bsdfs) - 1

    def bsdf_mirror(self):
        self.bsdfs.append(self._blank(BSDF_MIRROR)); return len(self.bsdfs) - 1

    def bsdf_lambertian(self, albedo_tex):
        b = self._blank(BSDF_LAMBERTIAN); b.base_color = albedo_tex
        self.bsdfs.append(b); return len(self.bsdfs) - 1

    def bsdf_ggx(self, albedo_tex, roughness=0.5, anisotropy=0.0):
        b = self._blank(BSDF_GGX); b.base_color = albedo_tex; b.alpha = roughness; b.anisotropy = anisotropy
        self.bsdfs.append(b); return len(self.bsdfs) - 1

    @staticmethod
    def _alpha(roughness):
        return float(max(np.float32(0.001), np.float32(roughness) * np.float32(roughness)))

    def bsdf_roughconductor(self, alpha=0.1, material="Au"):
        b = self._blank(BSDF_ROUGHCONDUCTOR); b.alpha = self._alpha(alpha)
        b.eta[:] = CONDUCTORS[material][0]; b.k[:] = CONDUCTORS[material][1]
        self.bsdfs.append(b); return len(self.bsdfs) - 1

    def bsdf_roughplastic(self, alpha=0.1, int_ior=1.5046, ext_ior=1.000277, kd=(0.5, 0.5, 0.5)):
        b = self._blank(BSDF_ROUGHPLASTIC); b.alpha = self._alpha(alpha); b.int_ior, b.ext_ior = int_ior, ext_ior
        b.albedo[:] = [float(c) for c in kd]
        self.bsdfs.append(b); return len(self.bsdfs) - 1

    def bsdf_roughdielectric(self, roughness=0.1, int_ior=1.5046, ext_ior=1.000277):
        b = self._blank(BSDF_ROUGHDIELECTRIC); b.alpha = self._alpha(roughness); b.int_ior, b.ext_ior = int_ior, ext_ior
        self.bsdfs.append(b); return len(self.bsdfs) - 1

    def light(self, radiance, primary_visibility=False):
        l = LightDesc(); l.radiance[:] = [float(c) for c in radiance]; l.primary_visibility = int(primary_visibility)
        self.lights.append(l); return len(self.lights) - 1

    def mesh(self, positions, indices, bsdf, normals=None, uvs=None, light=-1):
        P = self._arr(positions, np.float32).reshape(-1, 3)
        F = self._arr(indices, np.uint32).reshape(-1, 3)
        m = MeshDesc()
        m.positions = P.ctypes.data_as(c_float_p); m.indices = F.ctypes.data_as(c_u32_p)
        m.n_vertices, m.n_triangles, m.bsdf, m.light = P.shape[0], F.shape[0], bsdf, light
        self._keep += [P, F]
        if normals is not None:
            N = self._arr(normals, np.float32).reshape(-1, 3); m.normals = N.ctypes.data_as(c_float_p); self._keep.append(N)
        if uvs is not None:
            U = self._arr(uvs, np.float32).reshape(-1, 2); m.uvs = U.ctypes.data_as(c_float_p); self._keep.append(U)
        self.meshes.append(m); return len(self.meshes) - 1

    # setup --------------------------------------------------------------------------------------
    def set_camera(self, width, height, fov, to_world, near=1e-4, far=1e4, thinlens=None):
        fill_camera(self.camera, width, height, fov, to_world, near, far, thinlens)

    def set_sampler(self, kind, sample_count, seed=1, resolution=4, tables=None):
        """Applies the constructors' rounding rules (sampler.cpp:83-93,178-189,275-289)."""
        s = self.sampler
        s.type = {"independent": 0, "stratified": 1, "correlated": 2, "pmj02bn": 3}[kind]
        s.seed = seed
        if kind == "stratified":
            res = resolution
            while res * res < sample_count:
                res += 1
            s.res_x = s.res_y = res; s.sample_count = res * res
        elif kind == "correlated":
            ry = int(np.float32(math.sqrt(sample_count)))     # int m_resolution[1] = sqrt(uint32) -> double sqrt, truncated
            ry = int(math.sqrt(sample_count))
            rx = (sample_count + ry - 1) // ry
            s.res_x, s.res_y, s.sample_count = rx, ry, rx * ry
        else:
            s.res_x = s.res_y = 0; s.sample_count = min(sample_count, 65536) if kind == "pmj02bn" else sample_count
        if tables is not None:
            bn = self._arr(tables[0], np.uint16); pm = self._arr(tables[1], np.uint32)
            s.blue_noise = bn.ctypes.data_as(C.POINTER(C.c_uint16)); s.pmj02bn = pm.ctypes.data_as(c_u32_p)

    def set_filter(self, kind="gaussian", **kw):
        r, tab = filter_table(kind, **kw)
        self.filter.radius = r
        self.filter.table[:] = tab.tolist()

    def set_integrator(self, max_depth=5, trace_bias=1e-3, regularization=False, accumulated_roughness=0.5, kind="path_mis", env_sampling=False,
                       texture_filtering=False):
        """env_sampling: path_mis also samples the background as a light (kz_integrator_desc::env_sampling in include/kzgpu.h);
        texture_filtering: path_mis filters image textures by their screen footprint (kz_integrator_desc::texture_filtering)"""
        t = {"path_mis": 0, "normals": 1, "ao": 2, "whitted": 3, "path_mats": 4}[kind]
        self.integrator = IntegratorDesc(min(512, max_depth), trace_bias, int(regularization), accumulated_roughness, t, int(env_sampling),
                                         int(texture_filtering))

    def desc(self):
        d = SceneDesc()

        def arr(lst, T):
            a = (T * max(1, len(lst)))(*lst)
            self._keep.append(a)
            return a
        d.meshes, d.n_meshes = arr(self.meshes, MeshDesc), len(self.meshes)
        d.bsdfs, d.n_bsdfs = arr(self.bsdfs, BsdfDesc), len(self.bsdfs)
        d.textures, d.n_textures = arr(self.textures, TextureDesc), len(self.textures)
        d.images, d.n_images = arr(self.images, ImageDesc), len(self.images)
        d.lights, d.n_lights = arr(self.lights, LightDesc), len(self.lights)
        d.background = self.background
        d.camera, d.sampler, d.integrator, d.filter = self.camera, self.sampler, self.integrator, self.filter
        self._keep.append(d)
        return d


# --------------------------------------------------------------------------- library front-ends
class _Backend:
    """Common front-end over a library exporting the kzgpu-shaped API with some prefix."""

    def frame_shape(self):
        w, h, b = C.c_int32(), C.c_int32(), C.c_int32()
        self._call("frame_dims", self.h, C.byref(w), C.byref(h), C.byref(b))
        return h.value + 2 * b.value, w.value + 2 * b.value, b.value

    def resolve(self, frame):
        H, W, b = self.frame_shape()
        rgb = np.zeros((H - 2 * b, W - 2 * b, 3), np.float32)
        srgb = np.zeros((H - 2 * b, W - 2 * b, 3), np.uint8)
        self._call("resolve", self.h, frame.ctypes.data_as(c_float_p), rgb.ctypes.data_as(c_float_p),
                   srgb.ctypes.data_as(C.POINTER(C.c_uint8)))
        return rgb, srgb


    def intersection_dump(self, rays):
        """closest hit + post-intersection record per ray: (n, 24) float32, layout in include/kzgpu.h"""
        rays = np.ascontiguousarray(rays, RAY_DTYPE)
        out = np.zeros((rays.shape[0], 24), np.float32)
        self._call("intersection_dump", self.h, rays.ctypes.data_as(C.c_void_p), C.c_size_t(rays.shape[0]), out.ctypes.data_as(c_float_p))
        return out

    def light_sample_dump(self, ref, u5):
        """emitter sample per (reference point, 5 random numbers): (n, 16) float32, layout in include/kzgpu.h"""
        ref = np.ascontiguousarray(ref, np.float32).reshape(-1, 3)
        u5 = np.ascontiguousarray(u5, np.float32).reshape(-1, 5)
        out = np.zeros((ref.shape[0], 16), np.float32)
        self._call("light_sample_dump", self.h, ref.ctypes.data_as(c_float_p), u5.ctypes.data_as(c_float_p), C.c_size_t(ref.shape[0]), out.ctypes.data_as(c_float_p))
        return out


class HostScene:
    """A kazen XML scene loaded through the C++ host (nano-kazen_b200/host: XML parser + plugin registry).
    `.desc` is the flattened kz_scene_desc the host would upload; it stays valid until close()."""

    def __init__(self, xml_path, overrides=None, lib_path=LIB_HOST):
        if not os.path.exists(lib_path):
            raise RuntimeError(f"{lib_path} missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
        self.lib = C.CDLL(lib_path)
        self.lib.kazen_host_last_error.restype = C.c_char_p
        self.lib.kazen_host_load.restype = C.c_void_p
        self.lib.kazen_host_scene_desc.restype = C.POINTER(SceneDesc)
        self.lib.kazen_host_scene_desc.argtypes = [C.c_void_p]
        self.lib.kazen_host_free.argtypes = [C.c_void_p]
        self.lib.kazen_host_describe.argtypes = [C.c_void_p, C.c_char_p, C.c_size_t]
        self.lib.kazen_host_accel_builder.argtypes = [C.c_void_p]
        self.lib.kazen_host_render.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int]
        ov = ";".join(f"{k}={v}" for k, v in (overrides or {}).items()).encode() if overrides else None
        self.h = self.lib.kazen_host_load(os.fsencode(xml_path), ov)
        if not self.h:
            raise RuntimeError(self.lib.kazen_host_last_error().decode())
        p = self.lib.kazen_host_scene_desc(self.h)
        if not p:
            raise RuntimeError(self.lib.kazen_host_last_error().decode())
        self.desc = p.contents

    def describe(self):
        buf = C.create_string_buffer(1 << 16)
        self.lib.kazen_host_describe(self.h, buf, len(buf))
        return buf.value.decode()

    def accel_builder(self):
        return self.lib.kazen_host_accel_builder(self.h)

    def render(self, output_stem, gpus=1, raw=True):
        if self.lib.kazen_host_render(self.h, os.fsencode(output_stem), gpus, int(raw)) != 0:
            raise RuntimeError(self.lib.kazen_host_last_error().decode())

    def close(self):
        if self.h:
            self.lib.kazen_host_free(self.h); self.h = None


def host_registered_plugins(lib_path=LIB_HOST):
    lib = C.CDLL(lib_path)
    buf = C.create_string_buffer(1 << 14)
    lib.kazen_host_registered(buf, len(buf))
    return buf.value.decode().split()


def host_read_image(path, lib_path=LIB_HOST):
    """Decode an image file with the C++ host's imagetexture readers (PNG / PFM / HDR / EXR) -> (H, W, 3) float32."""
    lib = C.CDLL(lib_path)
    lib.kazen_host_last_error.restype = C.c_char_p
    w, h = C.c_int(), C.c_int()
    if lib.kazen_host_read_image(os.fsencode(path), C.byref(w), C.byref(h), None) != 0:
        raise RuntimeError(lib.kazen_host_last_error().decode())
    out = np.zeros((h.value, w.value, 3), np.float32)
    lib.kazen_host_read_image(os.fsencode(path), C.byref(w), C.byref(h), out.ctypes.data_as(c_float_p))
    return out


def host_write_exr(path, rgb, lib_path=LIB_HOST):
    """Write (H, W, 3) float32 linear RGB with the C++ host's EXR writer (the file `kazen` saves next to the PNG)."""
    rgb = np.ascontiguousarray(rgb, np.float32)
    lib = C.CDLL(lib_path)
    lib.kazen_host_last_error.restype = C.c_char_p
    if lib.kazen_host_write_exr(os.fsencode(path), C.c_int(rgb.shape[1]), C.c_int(rgb.shape[0]), rgb.ctypes.data_as(c_float_p)) != 0:
        raise RuntimeError(lib.kazen_host_last_error().decode())


def host_fallback_tables(lib_path=LIB_HOST):
    lib = C.CDLL(lib_path)
    bn = np.zeros((48, 128, 128), np.uint16); pm = np.zeros((5, 65536, 2), np.uint32)
    lib.kazen_host_fallback_tables(bn.ctypes.data_as(C.c_void_p), pm.ctypes.data_as(C.c_void_p))
    return bn, pm


def shard_range(begin, end, rank, world):
    """Contiguous slice of sample indices [begin, end) owned by `rank` of `world` (SURVEY 8e)."""
    n = end - begin
    return begin + n * rank // world, begin + n * (rank + 1) // world


def _pattern_floats(pattern):
    return sum(1 if ch == "1" else 2 for ch in pattern)


class Gpu(_Backend):
    """libkzgpu.so: the product.  Raises if the library or a CUDA device is missing (no fallback)."""

    def __init__(self, desc, devices=(0,), builder=BUILD_HOST_SAH, lib_path=LIB_GPU):
        if not os.path.exists(lib_path):
            raise RuntimeError(f"{lib_path} missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
        self.lib = C.CDLL(lib_path)
        self.lib.kzgpu_last_error.restype = C.c_char_p
        self.h = C.c_void_p()
        ids = (C.c_int * len(devices))(*devices)
        rc = self.lib.kzgpu_create(ids, len(devices), C.byref(self.h))
        if rc != KZ_OK:
            raise RuntimeError(f"kzgpu_create failed ({rc}): {self.lib.kzgpu_last_error(None).decode()}")
        self._call("scene_upload", self.h, C.byref(desc))
        self._call("accel_build", self.h, C.c_int(builder))
        self._desc = desc

    def _call(self, name, *args):
        rc = getattr(self.lib, "kzgpu_" + name)(*args)
        if rc != KZ_OK:
            raise RuntimeError(f"kzgpu_{name} failed ({rc}): {self.lib.kzgpu_last_error(self.h).decode()}")

    def close(self):
        if self.h:
            self.lib.kzgpu_destroy(self.h); self.h = C.c_void_p()

    def trace(self, rays, shadow=False, device=0):
        rays = np.ascontiguousarray(rays, RAY_DTYPE)
        hits = np.zeros(rays.shape[0], HIT_DTYPE)
        self._call("trace", self.h, C.c_int(device), rays.ctypes.data_as(C.c_void_p), C.c_size_t(rays.shape[0]),
                   C.c_int(int(shadow)), hits.ctypes.data_as(C.c_void_p))
        return hits

    def trace_device(self, d_rays_ptr, n, d_hits_ptr, shadow=False, device=0, stream=None):
        self._call("trace_device", self.h, C.c_int(device), C.c_void_p(d_rays_ptr), C.c_size_t(n), C.c_int(int(shadow)),
                   C.c_void_p(d_hits_ptr), C.c_void_p(stream or 0))

    def trace_host_ptr(self, rays_ptr, n, hits_ptr, shadow=False, device=0):
        self._call("trace", self.h, C.c_int(device), C.c_void_p(rays_ptr), C.c_size_t(n), C.c_int(int(shadow)), C.c_void_p(hits_ptr))

    def occluded(self, rays, trace_bias, device=0):
        rays = np.ascontiguousarray(rays, RAY_DTYPE)
        occ = np.zeros(rays.shape[0], np.uint8); seg = np.zeros(rays.shape[0], np.uint8)
        self._call("occluded", self.h, C.c_int(device), rays.ctypes.data_as(C.c_void_p), C.c_size_t(rays.shape[0]),
                   C.c_float(trace_bias), occ.ctypes.data_as(C.c_void_p), seg.ctypes.data_as(C.c_void_p))
        return occ, seg

    def sample_dump(self, triples, pattern):
        t = np.ascontiguousarray(triples, np.int32).reshape(-1, 3)
        out = np.zeros((t.shape[0], _pattern_floats(pattern)), np.float32)
        self._call("sample_dump", self.h, t.ctypes.data_as(C.c_void_p), C.c_size_t(t.shape[0]), pattern.encode(), out.ctypes.data_as(c_float_p))
        return out

    def camera_rays(self, samples4):
        s = np.ascontiguousarray(samples4, np.float32).reshape(-1, 4)
        out = np.zeros(s.shape[0], RAY_DTYPE)
        self._call("camera_rays", self.h, s.ctypes.data_as(c_float_p), C.c_size_t(s.shape[0]), out.ctypes.data_as(C.c_void_p))
        return out

    def render(self, spp_begin=0, spp_end=None, rect=None, frame=None):
        H, W, b = self.frame_shape()
        if frame is None:
            frame = np.zeros((H, W, 4), np.float32)
        x0, y0, x1, y1 = rect if rect else (0, 0, W - 2 * b, H - 2 * b)
        req = RenderReq(x0, y0, x1, y1, spp_begin, self._desc.sampler.sample_count if spp_end is None else spp_end, 0)
        self._call("render", self.h, C.byref(req), frame.ctypes.data_as(c_float_p))
        return frame

    def render_device(self, spp_begin, spp_end, device=0, clear=True, stream=None, frame_ptr=None, rect=None):
        """Enqueues a render on `stream`; the (H+2b, W+2b, 4) float32 frame stays in HBM (frame_ptr:
        caller-owned device buffer, else the context's own).  Returns the frame's device pointer."""
        H, W, b = self.frame_shape()
        x0, y0, x1, y1 = rect if rect else (0, 0, W - 2 * b, H - 2 * b)
        req = RenderReq(x0, y0, x1, y1, spp_begin, spp_end, int(clear))
        ptr = C.c_void_p(frame_ptr or 0)
        self._call("render_device", self.h, C.c_int(device), C.byref(req), C.byref(ptr), C.c_void_p(stream or 0))
        return ptr.value

    def bsdf_query(self, bsdf, mode, wi, wo=(0, 0, 1), uv=(0.5, 0.5), acc_rough=0.0, s1=0.5, s2=(0.5, 0.5)):
        out = (C.c_float * 8)()
        f3 = lambda v: (C.c_float * 3)(*[float(x) for x in v])
        f2 = lambda v: (C.c_float * 2)(*[float(x) for x in v])
        self._call("bsdf_query", self.h, C.c_int(bsdf), C.c_int(mode), f3(wi), f3(wo), f2(uv), C.c_float(acc_rough), C.c_float(s1), f2(s2), out)
        return np.array(list(out), np.float32)

    def image_lookup(self, image, st, level=0):
        st = np.ascontiguousarray(st, np.float32).reshape(-1, 2)
        out = np.zeros((st.shape[0], 3), np.float32)
        self._call("image_lookup", self.h, C.c_int(image), C.c_int(level), st.ctypes.data_as(c_float_p), C.c_size_t(st.shape[0]), out.ctypes.data_as(c_float_p))
        return out

    def env_sample_dump(self, u2, device=0):
        """environment light samples of device `device` for (row draw, column draw) pairs: (n, 8) float32 = direction[3], density,
        radiance[3], 0 (include/kzgpu.h); raises unless the scene counts the environment as a light"""
        u2 = np.ascontiguousarray(u2, np.float32).reshape(-1, 2)
        out = np.zeros((u2.shape[0], 8), np.float32)
        self._call("env_sample_dump", self.h, C.c_int(device), u2.ctypes.data_as(c_float_p), C.c_size_t(u2.shape[0]), out.ctypes.data_as(c_float_p))
        return out

    def image_lookup_filtered(self, image, st, dst):
        """the shade kernels' filtered lookup of image `image` at (s, t) pairs with st derivatives dst = (ds/dx, dt/dx, ds/dy, dt/dy)
        per pair: (n, 3) float32; raises unless the scene filters its textures"""
        st = np.ascontiguousarray(st, np.float32).reshape(-1, 2)
        dst = np.ascontiguousarray(dst, np.float32).reshape(-1, 4)
        assert dst.shape[0] == st.shape[0]
        out = np.zeros((st.shape[0], 3), np.float32)
        self._call("image_lookup_filtered", self.h, C.c_int(image), st.ctypes.data_as(c_float_p), dst.ctypes.data_as(c_float_p), C.c_size_t(st.shape[0]),
                   out.ctypes.data_as(c_float_p))
        return out

    def texture_footprint_dump(self, rays, device=0):
        """the texture footprint at each ray's closest hit on device `device`: (n, 8) float32 = mesh (-1: miss), u, v, du/dx, dv/dx,
        du/dy, dv/dy, 0 (include/kzgpu.h)"""
        rays = np.ascontiguousarray(rays, RAY_DTYPE)
        out = np.zeros((rays.shape[0], 8), np.float32)
        self._call("texture_footprint_dump", self.h, C.c_int(device), rays.ctypes.data_as(C.c_void_p), C.c_size_t(rays.shape[0]), out.ctypes.data_as(c_float_p))
        return out

    def configure(self, key, value):
        self._call("configure", self.h, key.encode(), C.c_int(int(value)))

    # animation: update -> refit -> render ---------------------------------------------------------
    def mesh_update(self, mesh, positions, normals=None):
        """new vertex positions (and normals) of mesh `mesh`: numpy arrays of 3 * n_vertices floats, or device pointers (ints, e.g. a
        torch CUDA tensor's data_ptr()).  Trace and render need refit() (or a rebuild) afterwards."""
        def ptr(a):
            if a is None:
                return None
            if isinstance(a, (int, np.integer)):
                return C.c_void_p(int(a))
            a = np.ascontiguousarray(a, np.float32)
            keep.append(a)
            return a.ctypes.data_as(C.c_void_p)
        keep = []
        self._call("mesh_update", self.h, C.c_int(mesh), ptr(positions), ptr(normals))

    def mesh_transform(self, mesh, matrix, inverse=None):
        """places mesh `mesh`'s rest pose (its uploaded or last mesh_update arrays) by the 4x4 `matrix` (row-major array-like, as the
        C++ host's toWorld); normals go through `inverse`'s transpose.  inverse=None on a mesh with normals: np.linalg.inv of the matrix
        in float64, rounded to float32 (kazen's Transform inverts in double and rounds once too).  Trace and render need refit() (or a
        rebuild) afterwards."""
        M = np.ascontiguousarray(matrix, np.float32).reshape(4, 4)
        if inverse is None and 0 <= mesh < self._desc.n_meshes and self._desc.meshes[mesh].normals:
            inverse = np.linalg.inv(M.astype(np.float64))
        inv = None if inverse is None else np.ascontiguousarray(inverse, np.float32).reshape(4, 4)
        self._call("mesh_transform", self.h, C.c_int(mesh), M.ctypes.data_as(c_float_p), None if inv is None else inv.ctypes.data_as(c_float_p))

    def refit(self):
        """refits the accel to the current vertex positions on every device (same tree, new boxes)"""
        self._call("accel_refit", self.h)

    def camera_update(self, width, height, fov, to_world, near=1e-4, far=1e4, thinlens=None):
        """replaces the camera (arguments as SceneBuilder.set_camera; width / height must be the uploaded ones)"""
        c = fill_camera(CameraDesc(), width, height, fov, to_world, near, far, thinlens)
        self._call("camera_update", self.h, C.byref(c))

    def accel_dump(self, device=0):
        """device `device`'s accel: (nodes as raw (n_nodes, 80) uint8, triangle records as (n_tris, 3, 4) float32)"""
        s = Stats()
        self._call("stats", self.h, C.byref(s))
        n_tris = (s.bvh_bytes - 80 * s.bvh_nodes) // 48
        nodes = np.zeros((s.bvh_nodes, 80), np.uint8); tris = np.zeros((n_tris, 3, 4), np.float32)
        self._call("accel_dump", self.h, C.c_int(device), nodes.ctypes.data_as(C.c_void_p), tris.ctypes.data_as(C.c_void_p))
        return nodes, tris

    def render_host_ptr(self, spp_begin, spp_end, frame_ptr, clear=True, rect=None):
        """kzgpu_render into a caller-owned (pinned) host frame given by address"""
        H, W, b = self.frame_shape()
        x0, y0, x1, y1 = rect if rect else (0, 0, W - 2 * b, H - 2 * b)
        req = RenderReq(x0, y0, x1, y1, spp_begin, spp_end, int(clear))
        self._call("render", self.h, C.byref(req), C.c_void_p(frame_ptr))

    def stats(self, reset=False):
        s = Stats()
        self._call("stats", self.h, C.byref(s))
        if reset:
            self._call("stats_reset", self.h)
        return s.as_dict()
